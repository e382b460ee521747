"""Host side of the device hmmlearn M-step and the sharded vocabulary fit, no GPU needed: the priors block sapr_hl_mstep reads
(hmmlearn_hmm.expand_priors) and its refusals, the params flag bits, and the shard assignment of fit_vocabulary(dist=...)."""
import numpy as np
import pytest


def _model(S, D, seed, **kw):
    from sapr_b200.hmmlearn_hmm import GaussianHMM
    rng = np.random.default_rng(seed)
    h = GaussianHMM(n_components=S, covariance_type="diag", init_params="", **kw)
    h.means_ = rng.normal(size=(S, D))
    h.covars_ = rng.uniform(0.5, 1.5, (S, D))
    h.transmat_ = np.full((S, S), 1.0 / S)
    h.startprob_ = np.full(S, 1.0 / S)
    return h


def test_expand_priors_layout():
    from sapr_b200.hmmlearn_hmm import expand_priors
    S, D = 4, 3
    rng = np.random.default_rng(0)
    arr = dict(startprob_prior=rng.uniform(1, 2, S), transmat_prior=rng.uniform(1, 2, (S, S)), means_prior=rng.normal(size=(S, D)),
               means_weight=rng.uniform(0, 1, (S, D)), covars_prior=rng.uniform(0, 1, (S, D)), covars_weight=2.5)
    a, b = _model(S, D, 0), _model(S, D, 1, **arr)
    P = expand_priors([a, b])
    assert P.shape == (2, S + S * S + 3 * S * D + 1) and P.dtype == np.float64
    o = np.cumsum([0, S, S * S, S * D, S * D, S * D, 1])
    defaults = (1.0, 1.0, 0.0, 0.0, 1e-2, 1.0)                                        # GaussianHMM's defaults
    for k, (name, dflt) in enumerate(zip(("startprob_prior", "transmat_prior", "means_prior", "means_weight", "covars_prior",
                                          "covars_weight"), defaults)):
        assert np.all(P[0, o[k]:o[k + 1]] == dflt), name
        assert np.array_equal(P[1, o[k]:o[k + 1]], np.ravel(arr[name])), name


@pytest.mark.parametrize("name,value", [("startprob_prior", np.ones(5)), ("transmat_prior", np.ones((4, 5))),
                                        ("transmat_prior", np.ones(4)), ("means_prior", np.zeros((4, 4))),
                                        ("means_weight", np.zeros(3)), ("covars_prior", np.zeros((3, 4))),
                                        ("covars_weight", np.ones(4)), ("covars_weight", np.ones((4, 3)))])
def test_expand_priors_refuses_other_shapes(name, value):
    from sapr_b200.hmmlearn_hmm import expand_priors, fit_vocabulary
    h = _model(4, 3, 0, **{name: value})
    with pytest.raises(ValueError, match=name):
        expand_priors([_model(4, 3, 1), h])
    with pytest.raises(ValueError, match=name):                                        # before any device work
        fit_vocabulary([_model(4, 3, 1), h], [[np.zeros((3, 5), np.float32)]] * 2)


def test_param_flags():
    from sapr_b200.hmmlearn_hmm import param_flags
    ms = [_model(3, 2, 0, params=p) for p in ("stmc", "st", "mc", "s", "c", "", "ct")]
    assert param_flags(ms).tolist() == [15, 3, 12, 1, 8, 0, 10]
    assert param_flags(ms).dtype == np.int32


@pytest.mark.parametrize("world", [1, 2, 3, 5, 8])
def test_vocabulary_shards(world):
    from sapr_b200.hmmlearn_hmm import vocabulary_shards
    rng = np.random.default_rng(world)
    counts = rng.integers(1, 30, 11)
    lens = rng.integers(20, 200, counts.sum())
    sh = vocabulary_shards(lens, world)
    assert len(sh) == world and sh[0][0] == 0 and sh[-1][1] == len(lens)
    assert all(a <= b for a, b in sh) and all(sh[r][1] == sh[r + 1][0] for r in range(world - 1))   # contiguous, each once
    frames = np.array([lens[a:b].sum() for a, b in sh])
    assert frames.sum() == lens.sum()
    assert frames.max() - frames.min() <= 2 * lens.max()                              # balanced to within an utterance or two
    labels = np.repeat(np.arange(11), counts)                                         # the model-grouped order fit_vocabulary packs
    for a, b in sh:
        assert np.all(np.diff(labels[a:b]) >= 0)


def test_vocabulary_shards_small_corpus_leaves_a_rank_empty():
    from sapr_b200.hmmlearn_hmm import vocabulary_shards
    sh = vocabulary_shards([50, 50], 3)
    assert sum(b - a for a, b in sh) == 2 and any(a == b for a, b in sh)


def test_train_hmm_dist_needs_batched():
    from sapr_b200.train import train_hmm
    with pytest.raises(ValueError):
        train_hmm("hmmlearn", dist=object())
