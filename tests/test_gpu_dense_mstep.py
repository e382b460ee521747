"""The device hmmlearn M-step (sapr_hl_mstep, csrc/hmmlearn.cu) and the device-resident, shardable fit_vocabulary built on it:
the kernel against GaussianHMM._do_mstep bit for bit, fit_vocabulary's trajectories against the host loop it replaced
(WordModels.estep + _do_mstep per model), and fit_vocabulary / train_hmm(batched=True) sharded over two and three ranks."""
import copy
import os
import pickle
import socket
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WORDS = ["heed", "hid", "head", "had", "hard", "hud", "hod", "hoard", "hood", "whod", "heard"]


@pytest.fixture(scope="module")
def eng():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from sapr_b200 import engine
    return engine


def _lr(S, aii):
    A = np.zeros((S, S))
    for i in range(S - 1):
        A[i, i] = aii; A[i, i + 1] = 1 - aii
    A[S - 1, S - 1] = 1.0
    return A


def _synth(M, S, D, B, T_lo, T_hi, seed, lr=()):
    """M random models (those in ``lr`` left-to-right: zeros in startprob_ and transmat_) and B utterances drawn from them,
    model-interleaved, every model with utterances."""
    rng = np.random.default_rng(seed)
    means = rng.normal(0.0, 3.0, (M, S, D))
    var = rng.uniform(0.5, 1.5, (M, S, D)) ** 2
    tm = rng.dirichlet(np.ones(S), size=(M, S))
    sp = rng.dirichlet(np.ones(S), size=M)
    for m in lr:
        tm[m] = _lr(S, rng.uniform(0.6, 0.95))
        sp[m] = 0.0; sp[m, 0] = 1.0
    labels = rng.integers(0, M, B)
    labels[:M] = np.arange(M)
    feats = []
    for w in labels:
        T = int(rng.integers(T_lo, T_hi + 1))
        st = np.sort(rng.integers(0, S, T)) if w in lr else rng.integers(0, S, T)
        feats.append((means[w, st] + np.sqrt(var[w, st]) * rng.standard_normal((T, D))).T.astype(np.float32))
    return feats, labels, (means, var, tm, sp)


PARAMS = ["stmc", "st", "mc", "s", "c", ""]


def _priors(kind, S, D, rng):
    if kind == "default":
        return {}
    if kind == "scalar":
        return dict(startprob_prior=2.0, transmat_prior=1.5, means_prior=0.25, means_weight=0.5, covars_prior=0.5, covars_weight=3)
    return dict(startprob_prior=rng.uniform(1.0, 3.0, S), transmat_prior=rng.uniform(1.0, 2.0, (S, S)),
                means_prior=rng.normal(size=(S, D)), means_weight=rng.uniform(0.0, 2.0, (S, D)),
                covars_prior=rng.uniform(0.0, 1.0, (S, D)), covars_weight=3.0)


def _same(a, b):
    """bit for bit, NaN where numpy gives NaN"""
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and np.array_equal(a, b, equal_nan=True)


@pytest.mark.parametrize("S,D", [(3, 13), (10, 13), (32, 13), (3, 39), (10, 39), (32, 39), (40, 13), (130, 39), (801, 13),
                                 (1024, 39)])
def test_hl_mstep_bit_identical_to_do_mstep(eng, S, D):
    """Every (params, priors) pair of a set at once; statistics from a real float64 E-step, with a transmat row without counts
    and a state without posterior mass written in; the models whose flag is 0 stay unchanged bit for bit."""
    import torch
    from sapr_b200._lib import ptr
    from sapr_b200.hmmlearn_hmm import GaussianHMM, expand_priors, param_flags
    kinds = [(p, k) for p in PARAMS for k in ("default", "scalar", "array")]
    M = len(kinds)
    feats, labels, (means, var, tm, sp) = _synth(M, S, D, 3 * M, 20, 60, seed=S * 100 + D, lr=range(0, M, 2))
    rng = np.random.default_rng(S + D)
    hs = []
    for mi, (params, kind) in enumerate(kinds):
        h = GaussianHMM(n_components=S, covariance_type="diag", init_params="", params=params, **_priors(kind, S, D, rng))
        h.means_, h.covars_, h.transmat_, h.startprob_ = means[mi].copy(), var[mi].copy(), tm[mi].copy(), sp[mi].copy()
        hs.append(h)
    dev = eng.WordModels(M, S, D, eng.EMIT_DIAG, eng.TOPO_DENSE)
    dev.set(means, var, tm, sp)
    batch = eng.PackedBatch.from_features(feats)
    lab = torch.as_tensor(labels.astype(np.int32), device=batch.X.device)
    stats, _, _ = dev.estep(batch, lab, None, eng.FP64)
    st = stats.cpu().numpy()
    u = dev.unpack_stats(st)                                                          # views into st
    for mi in range(M):
        r = mi % S
        u["trans"][mi, r, :] = 0.0                                                    # a transmat row with zero counts
        j = (mi + 1) % S
        u["post"][mi, j] = 0.0; u["obs"][mi, j] = 0.0; u["obs2"][mi, j] = 0.0       # a state with zero posterior
    flags = param_flags(hs)
    flags[0] = 0                                                                      # an inactive 'stmc' model
    before = dev.get()
    d_st = torch.as_tensor(st, device=batch.X.device)
    d_pr = torch.as_tensor(expand_priors(hs), device=batch.X.device)
    dev.ctx.check(dev.lib.sapr_hl_mstep(dev.ctx.h, dev.h, ptr(d_st), ptr(d_pr), ptr(flags)))
    got = dev.get()
    for mi, h in enumerate(hs):
        if flags[mi] == 0:
            for a, b in zip(got, before):
                assert a[mi].tobytes() == b[mi].tobytes(), mi
            continue
        h._do_mstep({k: v[mi] for k, v in u.items()})
        for name, a, b in zip(("means_", "covars", "transmat_", "startprob_"), got,
                              (h.means_, h._covars, h.transmat_, h.startprob_)):
            assert _same(a[mi], b), (kinds[mi], name)
    nan_means = [mi for mi, (p, k) in enumerate(kinds) if "m" in p and k == "default" and flags[mi]]
    assert all(np.isnan(got[0][mi][(mi + 1) % S]).all() for mi in nan_means)          # 0 / 0 as numpy gives it


def test_hl_mstep_refusals(eng):
    import torch
    from sapr_b200._lib import SaprError, ptr
    st = torch.zeros(64, dtype=torch.float64, device="cuda")
    flags = np.ones(2, dtype=np.int32)
    ee = eng.WordModels(2, 3, 4)                                                      # ENTRY_EXIT
    with pytest.raises(SaprError):
        ee.ctx.check(ee.lib.sapr_hl_mstep(ee.ctx.h, ee.h, ptr(st), ptr(st), ptr(flags)))
    dn = eng.WordModels(2, 3, 4, eng.EMIT_DIAG, eng.TOPO_DENSE)
    for args in ((None, st, flags), (st, None, flags), (st, st, None)):
        assert dn.lib.sapr_hl_mstep(dn.ctx.h, dn.h, *(ptr(a) for a in args)) == -1


def _init_models(prm, n_iter, seed):
    means, var, tm, sp = prm
    rng = np.random.default_rng(seed)
    from sapr_b200.hmmlearn_hmm import GaussianHMM
    hs = []
    for mi in range(means.shape[0]):
        h = GaussianHMM(n_components=means.shape[1], covariance_type="diag", init_params="", n_iter=n_iter, tol=1e-2,
                        params="mc" if mi == 3 else "stmc")
        if mi == 5:
            h.tol = 1e12                                                              # converges after 2 iterations
        if mi == 7:
            h.n_iter = 0                                                              # never leaves its initial parameters
        h.means_ = means[mi] + 0.3 * np.sqrt(var[mi]) * rng.standard_normal(means[mi].shape)
        h.covars_ = var[mi] * 1.5
        h.transmat_, h.startprob_ = tm[mi].copy(), sp[mi].copy()
        hs.append(h)
    return hs


def _host_loop(eng, models, features, precision):
    """fit_vocabulary as it ran before the device M-step: parameters uploaded every iteration, statistics downloaded, and each
    active model's own numpy _do_mstep."""
    from sapr_b200.decoder import stack_hmmlearn_models
    from sapr_b200.hmmlearn_hmm import ConvergenceMonitor
    means, _, _, _ = stack_hmmlearn_models(models)
    M, S, D = means.shape
    feats = [np.asarray(x, dtype=np.float32) for f in features for x in f]
    counts = np.array([len(f) for f in features])
    bounds = np.concatenate([[0], np.cumsum(counts)])
    batch = eng.PackedBatch.from_features(feats, labels=np.repeat(np.arange(M), counts))
    dev = eng.WordModels(M, S, D, eng.EMIT_DIAG, eng.TOPO_DENSE)
    prec = eng.FP64 if precision == "fp64" else eng.FP32
    for mdl in models:
        mdl.monitor_ = ConvergenceMonitor(mdl.tol, mdl.n_iter, mdl.verbose)
    active = [i for i, mdl in enumerate(models) if mdl.n_iter > 0]
    while active:
        dev.set(*stack_hmmlearn_models(models))
        stats, loglik, _ = dev.estep(batch, batch.labels, None, prec)
        st = dev.unpack_stats(stats)
        ll = loglik.cpu().numpy()
        still = []
        for i in active:
            models[i]._do_mstep({k: v[i] for k, v in st.items()})
            models[i].monitor_.report(float(ll[bounds[i]:bounds[i + 1]].sum()))
            if not models[i].monitor_.converged:
                still.append(i)
        active = still
    return models


def _assert_same_fit(a_models, b_models):
    for mi, (a, b) in enumerate(zip(a_models, b_models)):
        assert list(a.monitor_.history) == list(b.monitor_.history), mi
        assert a.monitor_.iter == b.monitor_.iter, mi
        for k in ("means_", "_covars", "transmat_", "startprob_"):
            assert _same(getattr(a, k), getattr(b, k)), (mi, k)


@pytest.mark.parametrize("precision", ["fp32", "fp64"])
def test_fit_vocabulary_trajectory_equals_host_loop(eng, precision):
    from sapr_b200.hmmlearn_hmm import fit_vocabulary
    feats, labels, prm = _synth(11, 6, 13, 330, 20, 60, seed=21, lr=range(11))
    base = _init_models(prm, 5, 1)
    words = [[feats[u] for u in np.nonzero(labels == mi)[0]] for mi in range(11)]
    host = _host_loop(eng, copy.deepcopy(base), words, precision)
    dev = fit_vocabulary(copy.deepcopy(base), words, precision=precision)
    assert host[5].monitor_.iter == 2 and host[7].monitor_.iter == 0 and any(h.monitor_.iter == 5 for h in host)
    _assert_same_fit(dev, host)
    assert dev[7].means_ is not None and _same(dev[7].means_, base[7].means_)


# ---- sharded: worker processes on the one GPU, gloo (NCCL refuses two ranks on one device) ----
_WORKER = r'''
import os, pickle, sys
sys.path.insert(0, os.environ["SAPR_ROOT"])
import torch
from sapr_b200.dist import Dist


class HostDist(Dist):
    """sums through host tensors: the test does not depend on gloo's support for CUDA tensors"""
    def allreduce_(self, t, ctx=None):
        h = t.cpu()
        self.td.all_reduce(h, op=self.td.ReduceOp.SUM)
        t.copy_(h)
        return t


d = HostDist(backend="gloo")
torch.cuda.set_device(0)
job = pickle.load(open(os.environ["JOB"], "rb"))
out = os.path.join(os.environ["OUT"], f"rank{d.rank}.pkl")
if job["kind"] == "fit":
    from sapr_b200.hmmlearn_hmm import fit_vocabulary
    res = fit_vocabulary(job["models"], job["words"], precision=job["precision"], dist=d)
else:
    from sapr_b200.train import train_hmm
    train_hmm("hmmlearn", 8, 13, n_iter=3, feature_set_path=job["fs"], models_dir=os.path.join(os.environ["OUT"], f"models{d.rank}"),
              batched=True, dist=d)
    res = dict(train_hmm.histories)
pickle.dump(res, open(out, "wb"))
d.barrier(); d.shutdown()
print("RANK_OK", d.rank)
'''


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _run_ranks(tmp_path, world, job, timeout=600):
    script, jobf = tmp_path / "worker.py", tmp_path / "job.pkl"
    script.write_text(_WORKER)
    with open(jobf, "wb") as f:
        pickle.dump(job, f)
    env = dict(os.environ, SAPR_ROOT=ROOT, MASTER_ADDR="127.0.0.1", MASTER_PORT=str(_free_port()), WORLD_SIZE=str(world),
               SAPR_NATIVE_COMM="0", JOB=str(jobf), OUT=str(tmp_path), CUDA_VISIBLE_DEVICES=os.environ.get("CUDA_VISIBLE_DEVICES", "0"))
    procs = []
    try:
        for r in range(world):
            procs.append(subprocess.Popen([sys.executable, str(script)], env=dict(env, RANK=str(r), LOCAL_RANK="0"),
                                          stdout=subprocess.PIPE, stderr=subprocess.STDOUT))
        outs = [p.communicate(timeout=timeout)[0].decode() for p in procs]
    finally:
        for p in procs:                                                               # no worker outlives the test
            if p.poll() is None:
                p.kill()
                p.wait()
    for p, o in zip(procs, outs):
        assert p.returncode == 0 and "RANK_OK" in o, o[-4000:]
    res = []
    for r in range(world):
        with open(tmp_path / f"rank{r}.pkl", "rb") as f:
            res.append(pickle.load(f))
    return res


def _rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    assert np.array_equal(np.isnan(a), np.isnan(b))
    ok = ~np.isnan(b)
    return float(np.max(np.abs(a[ok] - b[ok]) / np.maximum(np.abs(b[ok]), 1e-300), initial=0.0))


def _check_sharded(ranks, single):
    for r in ranks[1:]:                                                               # every rank holds the same bytes
        for a, b in zip(r, ranks[0]):
            assert list(a.monitor_.history) == list(b.monitor_.history)
            for k in ("means_", "_covars", "transmat_", "startprob_"):
                assert np.asarray(getattr(a, k)).tobytes() == np.asarray(getattr(b, k)).tobytes(), k
    for mi, (a, b) in enumerate(zip(ranks[0], single)):
        assert a.monitor_.iter == b.monitor_.iter, mi
        assert _rel(list(a.monitor_.history), list(b.monitor_.history)) <= 1e-12, mi
        for k in ("means_", "_covars", "transmat_", "startprob_"):
            assert _rel(getattr(a, k), getattr(b, k)) <= 1e-10, (mi, k)


def test_fit_vocabulary_two_ranks_fp64(eng, tmp_path):
    from sapr_b200.hmmlearn_hmm import fit_vocabulary, vocabulary_shards
    feats, labels, prm = _synth(11, 6, 13, 330, 20, 60, seed=21, lr=range(11))
    base = _init_models(prm, 5, 1)
    words = [[feats[u] for u in np.nonzero(labels == mi)[0]] for mi in range(11)]
    sh = vocabulary_shards([x.shape[1] for w in words for x in w], 2)
    grouped = np.repeat(np.arange(11), [len(w) for w in words])
    assert all(len(set(grouped[a:b])) < 11 for a, b in sh)                           # each shard lacks some model
    ranks = _run_ranks(tmp_path, 2, dict(kind="fit", models=base, words=words, precision="fp64"))
    single = fit_vocabulary(copy.deepcopy(base), words, precision="fp64")
    _check_sharded(ranks, single)


def test_fit_vocabulary_three_ranks_one_empty_shard(eng, tmp_path):
    from sapr_b200.hmmlearn_hmm import fit_vocabulary, vocabulary_shards
    feats, labels, prm = _synth(2, 6, 13, 2, 80, 80, seed=5)
    words = [[feats[0]], [feats[1]]]
    assert any(a == b for a, b in vocabulary_shards([80, 80], 3))
    base = _init_models(prm, 4, 2)
    ranks = _run_ranks(tmp_path, 3, dict(kind="fit", models=base, words=words, precision="fp64"))
    single = fit_vocabulary(copy.deepcopy(base), words, precision="fp64")
    _check_sharded(ranks, single)


def test_train_hmm_two_ranks_pickles_on_rank0(eng, tmp_path, monkeypatch):
    from sapr_b200 import synth
    from sapr_b200.train import train_hmm
    fs = tmp_path / "feature_set"; fs.mkdir()
    feats, labels, _, _ = synth.make_corpus(11 * 8, 11, 8, 13, 40, 60, seed=4243)
    for u, (x, w) in enumerate(zip(feats, labels)):
        np.save(fs / f"sp{u // 11:02d}a_w{u:03d}_{WORDS[w]}.npy", x)
    h0, h1 = _run_ranks(tmp_path, 2, dict(kind="train", fs=str(fs)))
    assert h0 == h1
    assert sorted(p.name for p in (tmp_path / "models0" / "hmmlearn").iterdir()) == sorted(f"{w}_hmmlearn_3.pkl" for w in WORDS)
    assert not (tmp_path / "models1").exists() or not any((tmp_path / "models1").rglob("*.pkl"))
    monkeypatch.chdir(tmp_path)
    train_hmm("hmmlearn", 8, 13, n_iter=3, feature_set_path=str(fs), models_dir=str(tmp_path / "single"), batched=True)
    for w in WORDS:
        a, b = np.array(h0[w]), np.array(train_hmm.histories[w])
        assert len(a) == len(b) and np.max(np.abs(a - b) / np.abs(b)) <= 1e-5, w
