"""Stacking hmmlearn-style models into one DENSE word-model set (decoder.stack_hmmlearn_models): public attributes only,
the diagonal of the expanded covariance getter, and a ValueError for models of different shapes -- before any GPU work."""
import pickle

import numpy as np
import pytest


class _PublicOnly:
    """Stands in for hmmlearn's own GaussianHMM: only the public attributes, covars_ expanded to (S, D, D)."""

    def __init__(self, S, D, seed):
        rng = np.random.default_rng(seed)
        self.means_ = rng.standard_normal((S, D))
        self.covars_ = np.array([np.diag(v) for v in rng.uniform(0.5, 2.0, (S, D))])
        self.transmat_ = rng.dirichlet(np.ones(S), size=S)
        self.startprob_ = rng.dirichlet(np.ones(S))


def test_stack_reads_public_attributes():
    from sapr_b200.decoder import stack_hmmlearn_models
    ms = [_PublicOnly(5, 3, s) for s in range(4)]
    means, var, tm, sp = stack_hmmlearn_models(ms)
    assert means.shape == (4, 5, 3) and var.shape == (4, 5, 3) and tm.shape == (4, 5, 5) and sp.shape == (4, 5)
    for i, m in enumerate(ms):
        assert np.array_equal(var[i], np.diagonal(m.covars_, axis1=1, axis2=2))
        assert np.array_equal(means[i], m.means_) and np.array_equal(tm[i], m.transmat_) and np.array_equal(sp[i], m.startprob_)


def test_stack_refuses_mixed_shapes():
    from sapr_b200.decoder import stack_hmmlearn_models
    with pytest.raises(ValueError):
        stack_hmmlearn_models([_PublicOnly(5, 3, 0), _PublicOnly(6, 3, 1)])
    with pytest.raises(ValueError):
        stack_hmmlearn_models([_PublicOnly(5, 3, 0), _PublicOnly(5, 4, 1)])


def test_decode_batch_refuses_mixed_states(tmp_path):
    from sapr_b200.decoder import Decoder
    from sapr_b200.hmmlearn_hmm import GaussianHMM
    d = tmp_path / "hmmlearn"; d.mkdir()
    for w, S in (("heed", 5), ("hid", 6)):
        src = _PublicOnly(S, 13, S)
        h = GaussianHMM(n_components=S, covariance_type="diag", init_params="")
        h.means_, h.covars_, h.transmat_, h.startprob_ = src.means_, src.covars_, src.transmat_, src.startprob_
        with open(d / f"{w}_hmmlearn_15.pkl", "wb") as f:
            pickle.dump(h, f)
    dec = Decoder(models_dir=str(tmp_path), implementation="hmmlearn", n_iter=15)
    with pytest.raises(ValueError):
        dec.decode_batch([np.zeros((13, 7), dtype=np.float32)])
