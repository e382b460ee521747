"""Host-side checks of the batched hmmlearn training surface that need no GPU: argument validation of
hmmlearn_hmm.fit_vocabulary and train_hmm(..., batched=True) happens before any device work."""
import numpy as np
import pytest


def _model(S, D, seed):
    from sapr_b200.hmmlearn_hmm import GaussianHMM
    rng = np.random.default_rng(seed)
    h = GaussianHMM(n_components=S, covariance_type="diag", init_params="")
    h.means_ = rng.normal(size=(S, D))
    h.covars_ = rng.uniform(0.5, 1.5, (S, D))
    h.transmat_ = np.full((S, S), 1.0 / S)
    h.startprob_ = np.full(S, 1.0 / S)
    return h


def test_fit_vocabulary_refuses_mixed_shapes():
    from sapr_b200.hmmlearn_hmm import fit_vocabulary
    feats = [np.zeros((13, 20), dtype=np.float32)]
    with pytest.raises(ValueError):
        fit_vocabulary([_model(10, 13, 0), _model(8, 13, 1)], [feats, feats])
    with pytest.raises(ValueError):
        fit_vocabulary([_model(10, 13, 0), _model(10, 39, 1)], [feats, feats])


def test_fit_vocabulary_refuses_bad_arguments():
    from sapr_b200.hmmlearn_hmm import fit_vocabulary
    feats = [np.zeros((13, 20), dtype=np.float32)]
    with pytest.raises(ValueError):
        fit_vocabulary([_model(10, 13, 0), _model(10, 13, 1)], [feats, []])           # a word without utterances
    with pytest.raises(ValueError):
        fit_vocabulary([_model(10, 13, 0)], [feats, feats])                           # one feature list per model
    with pytest.raises(ValueError):
        fit_vocabulary([_model(10, 13, 0)], [feats], precision="fp16")


def test_train_hmm_batched_custom_refused():
    from sapr_b200.train import train_hmm
    with pytest.raises(ValueError):
        train_hmm("custom", batched=True)
