"""Batched scoring with hmmlearn-style word models (DENSE topology): sapr_score_words against sapr_hl_score per model
(GaussianHMM.score) + the strict-'>' arg-max, the fp32 fused forward (csrc/score_dense.cu) against the float64 verification
mode and the oracle, the edges of the fp32 range, the float64 re-scoring of word near-ties, the refusals, a large batch, and
train -> Decoder.score_batch."""
import ctypes as C

import numpy as np
import pytest

from conftest import assert_close, split_features
from oracle import oracle as orc

pytestmark = pytest.mark.gpu

WORDS = ["heed", "hid", "head", "had", "hard", "hud", "hod", "hoard", "hood", "whod", "heard"]


@pytest.fixture(scope="module")
def eng():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from sapr_b200 import engine
    return engine


def _dense(eng, means, var, tm, sp):
    M, S, D = means.shape
    m = eng.WordModels(M, S, D, eng.EMIT_DIAG, eng.TOPO_DENSE)
    m.set(means, var, tm, sp)
    return m


def _lr_transmat(S, aii=0.9):
    """The reference's initial left-to-right pattern: 2S - 2 finite arcs."""
    A = np.zeros((S, S))
    if S == 1:
        A[0, 0] = 1.0
        return A
    A[0, 1] = 1.0
    for i in range(1, S - 1):
        A[i, i] = aii; A[i, i + 1] = 1 - aii
    A[S - 1, S - 1] = 1.0
    return A


def _synth(M, S, D, B, T_lo, T_hi, dense, seed):
    """M random diagonal-Gaussian models and B utterances drawn from them (lengths U{T_lo..T_hi})."""
    rng = np.random.default_rng(seed)
    scale = 10.0 if D == 13 else 1.0
    means = rng.normal(0.0, 2.0, (M, S, D)) * scale
    var = (rng.uniform(0.5, 1.5, (M, S, D)) * scale) ** 2
    if dense:
        tm = rng.dirichlet(np.ones(S), size=(M, S))
        sp = rng.dirichlet(np.ones(S), size=M)
    else:
        tm = np.stack([_lr_transmat(S, rng.uniform(0.6, 0.95)) for _ in range(M)])
        sp = np.zeros((M, S)); sp[:, 0] = 1.0
    lens = rng.integers(T_lo, T_hi + 1, B)
    labels = rng.integers(0, M, B)
    feats = []
    for w, T in zip(labels, lens):
        st = np.sort(rng.integers(0, S, T)) if not dense else rng.integers(0, S, T)
        feats.append((means[w, st] + np.sqrt(var[w, st]) * rng.standard_normal((T, D))).T.astype(np.float32))
    return feats, labels, (means, var, tm, sp)


def _hl_score(m, batch):
    """sapr_hl_score (GaussianHMM.score's kernel) for every model: [B, M]."""
    import torch
    sc = np.empty((batch.B, m.M))
    for mi in range(m.M):
        lp = torch.zeros(batch.B, dtype=torch.float64, device=batch.X.device)
        m.ctx.check(m.lib.sapr_hl_score(m.ctx.h, m.h, mi, C.c_void_p(batch.X.data_ptr()), batch.ldx,
                                        C.c_void_p(batch.offsets.data_ptr()), batch.B, batch.total_frames, C.c_void_p(lp.data_ptr())))
        sc[:, mi] = lp.cpu().numpy()
    return sc


def _argmax_first(sc):
    bw = np.full(sc.shape[0], -1, dtype=np.int32); bs = np.full(sc.shape[0], -np.inf)
    for mi in range(sc.shape[1]):
        take = sc[:, mi] > bs
        bw[take] = mi; bs[take] = sc[take, mi]
    return bw, bs


def _oracle_scores(x_DT, means, var, tm, sp):
    return np.array([orc.hl_forward(orc.emission_diag(np.asarray(x_DT, dtype=np.float64), means[mi], var[mi], all_emit=True),
                                    sp[mi], tm[mi])[0] for mi in range(means.shape[0])])


def _np(out):
    return {k: (None if v is None else v.cpu().numpy()) for k, v in out.items()}


def _rung1_models(g):
    """11 DENSE models from the Rung-1 goldens (as test_gpu_dense_words builds them)."""
    S = 10
    rng = np.random.default_rng(3)
    ms, vs, tms, sps = [], [], [], []
    for w in range(11):
        means = g["means"][w].copy()
        means[0] = means[1] + 0.1 * rng.standard_normal(means.shape[1])
        means[-1] = means[-2] + 0.1 * rng.standard_normal(means.shape[1])
        var = g["var"][w].copy()
        var[0] = var[1]; var[-1] = var[-2]
        sp = np.zeros(S); sp[0] = 1.0
        if w == 4:
            sp[0] = 0.6; sp[1] = 0.4
        ms.append(means); vs.append(var); tms.append(g["A"][w].copy()); sps.append(sp)
    return np.stack(ms), np.stack(vs), np.stack(tms), np.stack(sps)


def _check_fp64(m, batch):
    from sapr_b200._lib import FP64
    out = _np(m.score_words(batch, FP64, want_scores=True))
    sc = _hl_score(m, batch)
    bw, bs = _argmax_first(sc)
    assert np.array_equal(out["scores"], sc)                                     # bit for bit
    assert np.array_equal(out["best_word"], bw)
    assert np.array_equal(out["best_score"], bs)
    return out, sc


def test_fp64_equals_hl_score_rung1(eng, rung1_d13):
    g = rung1_d13
    means, var, tm, sp = _rung1_models(g)
    feats = [f.astype(np.float32) for f in split_features(g)]
    feats += [feats[0][:, :1], feats[1][:, :2], feats[2][:, :0]]                # T = 1, 2 and an empty utterance
    m = _dense(eng, means, var, tm, sp)
    batch = eng.PackedBatch.from_features(feats)
    out, sc = _check_fp64(m, batch)
    assert np.all(sc[-1] == 0.0) and out["best_word"][-1] == 0
    from sapr_b200.hmmlearn_hmm import GaussianHMM
    for u in list(range(0, batch.B - 1, 23)) + [batch.B - 3, batch.B - 2]:
        for mi in range(11):
            h = GaussianHMM(n_components=10, covariance_type="diag", init_params="")
            h.means_, h.covars_, h.transmat_, h.startprob_ = means[mi], var[mi], tm[mi], sp[mi]
            assert h.score(feats[u].T) == sc[u, mi]


@pytest.mark.parametrize("S", [1, 2, 10, 33, 64])
def test_fp64_equals_hl_score_random(eng, S):
    feats, _, prm = _synth(5, S, 13, 150, 1, 40, True, seed=700 + S)
    m = _dense(eng, *prm)
    _check_fp64(m, eng.PackedBatch.from_features(feats))


@pytest.mark.parametrize("S", [1, 2, 4, 8, 9, 10, 16, 17, 32])
@pytest.mark.parametrize("D", [13, 39])
@pytest.mark.parametrize("dense", [False, True])
@pytest.mark.parametrize("ragged", [False, True])
@pytest.mark.parametrize("M", [1, 11, 17])
def test_fp32_against_fp64(eng, S, D, dense, ragged, M):
    B = 300
    feats, labels, (means, var, tm, sp) = _synth(M, S, D, B, 30 if ragged else 60, 90 if ragged else 60, dense,
                                                 seed=S * 1000 + D * 10 + M + 7 * dense)
    if ragged:
        feats[3] = feats[3][:, :1]                                               # one-frame and empty utterances
        feats[7] = feats[7][:, :0]
    m = _dense(eng, means, var, tm, sp)
    batch = eng.PackedBatch.from_features(feats)
    ref = _np(m.score_words(batch, eng.FP64))
    out = _np(m.score_words(batch, eng.FP32))
    assert np.array_equal(out["best_word"], ref["best_word"])
    assert_close(out["scores"], ref["scores"], 1e-6, what="scores")
    assert_close(out["best_score"], ref["best_score"], 1e-6, what="best scores")
    if ragged:
        assert np.all(out["scores"][7] == 0.0) and out["best_word"][7] == 0
        assert_close(out["scores"][3], _hl_score(m, batch)[3], 1e-6, what="one-frame utterance")
    for u in range(0, B, 97):                                                    # the oracle restatement of hmmlearn's forward
        assert_close(out["scores"][u], _oracle_scores(feats[u], means, var, tm, sp), 1e-6, what="oracle")


def test_zero_start_and_transition_probabilities(eng):
    M, S, D = 11, 10, 13
    feats, _, (means, var, tm, sp) = _synth(M, S, D, 600, 20, 80, True, seed=41)
    rng = np.random.default_rng(2)
    for mi in range(M):
        tm[mi][rng.random((S, S)) < 0.4] = 0.0
        tm[mi][np.arange(S), (np.arange(S) + 1) % S] += 0.05                    # every row keeps mass
        tm[mi] /= tm[mi].sum(axis=1, keepdims=True)
        sp[mi][rng.random(S) < 0.5] = 0.0
        sp[mi, mi % S] += 0.1
        sp[mi] /= sp[mi].sum()
    m = _dense(eng, means, var, tm, sp)
    batch = eng.PackedBatch.from_features(feats)
    ref, out = _np(m.score_words(batch, eng.FP64)), _np(m.score_words(batch, eng.FP32))
    assert np.array_equal(out["best_word"], ref["best_word"])
    assert_close(out["scores"], ref["scores"], 1e-6, what="scores")


def test_no_model_scores_gives_minus_one(eng):
    S, D = 6, 13
    feats, _, (means, var, tm, sp) = _synth(2, S, D, 70, 2, 9, False, seed=5)
    tm[:, S - 1] = 0.0
    sp[:] = 0.0; sp[:, S - 1] = 1.0
    m = _dense(eng, means, var, tm, sp)
    batch = eng.PackedBatch.from_features(feats)
    for p in (eng.FP64, eng.FP32):
        o = _np(m.score_words(batch, p))
        assert np.all(o["best_word"] == -1)
        assert np.all(o["best_score"] == -np.inf)
        assert np.all(o["scores"] == -np.inf)


def test_far_from_every_model(eng):
    M, S, D = 11, 10, 39
    feats, _, (means, var, tm, sp) = _synth(M, S, D, 400, 40, 100, False, seed=8)
    sd = np.sqrt(var).mean(axis=(0, 1))
    far = [f + (50.0 * sd * np.sign(np.random.default_rng(u).standard_normal(D)))[:, None].astype(np.float32)
           for u, f in enumerate(feats)]
    m = _dense(eng, means, var, tm, sp)
    batch = eng.PackedBatch.from_features(far)
    ref, out = _np(m.score_words(batch, eng.FP64)), _np(m.score_words(batch, eng.FP32))
    assert np.all(np.isfinite(out["scores"]))
    assert np.array_equal(out["best_word"], ref["best_word"])
    assert_close(out["scores"], ref["scores"], 1e-6, what="scores")


@pytest.mark.parametrize("tiny", [1e-50, 1e-45])
def test_transitions_below_the_fp32_range(eng, tiny):
    """The only arc into state k + 1 has probability 1e-50 (below fp32) or 1e-45 (its smallest denormal)."""
    M, S, D, k = 11, 10, 13, 4
    feats, _, (means, var, tm, sp) = _synth(M, S, D, 500, 30, 90, False, seed=13)
    for mi in range(M):
        tm[mi, k] = 0.0; tm[mi, k, k] = 1.0 - tiny; tm[mi, k, k + 1] = tiny
        tm[mi, k + 1] = 0.0; tm[mi, k + 1, k + 2] = 1.0
    m = _dense(eng, means, var, tm, sp)
    batch = eng.PackedBatch.from_features(feats)
    ref, out = _np(m.score_words(batch, eng.FP64)), _np(m.score_words(batch, eng.FP32))
    assert np.all(np.isfinite(ref["scores"]))
    assert np.all(np.isfinite(out["scores"]))
    assert np.array_equal(out["best_word"], ref["best_word"])
    assert_close(out["scores"], ref["scores"], 1e-6, what="scores")


def test_fp32_near_ties_are_rescored_in_float64(eng, monkeypatch):
    M, S, D, B = 11, 10, 13, 900
    feats, labels, (means, var, tm, sp) = _synth(M, S, D, B, 40, 64, False, seed=77)
    rng = np.random.default_rng(5)
    means[5] = means[3] + 1e-7 * np.sqrt(var[3]) * rng.standard_normal(means[3].shape)
    var[5] = var[3]; tm[5] = tm[3]; sp[5] = sp[3]
    m = _dense(eng, means, var, tm, sp)
    batch = eng.PackedBatch.from_features(feats)
    ref = _np(m.score_words(batch, eng.FP64))
    assert m.ctx.viterbi_flagged() == 0
    out = _np(m.score_words(batch, eng.FP32))
    flagged = m.ctx.viterbi_flagged()
    rw = ref["best_word"]
    near = np.isin(rw, (3, 5))
    assert near.sum() > 30 and flagged >= near.sum()
    assert np.array_equal(out["best_word"], rw)
    assert np.array_equal(out["best_score"][near], ref["best_score"][near])
    assert np.array_equal(out["scores"][near], ref["scores"][near])
    monkeypatch.setenv("SAPR_EXACT_WORDS", "0")
    raw = _np(m.score_words(batch, eng.FP32, want_scores=False))["best_word"]
    assert m.ctx.viterbi_flagged() == 0
    assert np.mean(raw[near] != rw[near]) > 0.05


def test_refusals(eng):
    import torch
    from sapr_b200._lib import SaprError
    feats, _, prm = _synth(3, 10, 13, 40, 20, 30, True, seed=1)
    m = _dense(eng, *prm)
    batch = eng.PackedBatch.from_features(feats)

    def call(mm, ldx=batch.ldx, precision=eng.FP32, outs=True):
        bw = torch.empty(batch.B, dtype=torch.int32, device=batch.X.device)
        mm.ctx.check(mm.lib.sapr_score_words(mm.ctx.h, mm.h, C.c_void_p(batch.X.data_ptr()), ldx,
                                             C.c_void_p(batch.offsets.data_ptr()), batch.B, batch.total_frames, precision,
                                             C.c_void_p(bw.data_ptr() if outs else 0), None, None))

    call(m)
    for kw in (dict(ldx=13), dict(precision=7), dict(precision=eng.FP32_SIMT), dict(outs=False)):
        with pytest.raises(SaprError) as e:
            call(m, **kw)
        assert e.value.code == -1, kw
    ee = eng.WordModels(3, 8, 13)                                                # ENTRY_EXIT (the custom models)
    ee.set(np.zeros((3, 10, 13)), np.ones((3, 10, 13)), np.stack([_lr_transmat(10)] * 3))
    with pytest.raises(SaprError) as e:
        call(ee)
    assert e.value.code == -1
    big = _dense(eng, *_synth(2, 33, 13, 4, 5, 6, True, seed=2)[2])
    with pytest.raises(SaprError) as e:
        call(big)
    assert e.value.code == -4 and "SAPR_FP64" in str(e.value)
    call(big, precision=eng.FP64)


def test_large_batch_deterministic_and_oracle(eng):
    import torch
    M, S, D, B, T = 11, 10, 39, 100_000, 200
    rng = np.random.default_rng(31)
    means = rng.normal(0.0, 2.0, (M, S, D)); var = rng.uniform(0.5, 1.5, (M, S, D)) ** 2
    tm = np.stack([_lr_transmat(S, rng.uniform(0.8, 0.95)) for _ in range(M)])
    sp = np.zeros((M, S)); sp[:, 0] = 1.0
    m = _dense(eng, means, var, tm, sp)
    dev = torch.device("cuda", torch.cuda.current_device())
    g = torch.Generator(device=dev); g.manual_seed(5)
    X = torch.zeros(B * T, 40, dtype=torch.float32, device=dev)
    mt = torch.tensor(means.reshape(M * S, D), dtype=torch.float32, device=dev)
    sd = torch.tensor(np.sqrt(var).reshape(M * S, D), dtype=torch.float32, device=dev)
    w = torch.randint(0, M, (B,), device=dev, generator=g).repeat_interleave(T)
    for r0 in range(0, B * T, 1 << 22):
        r1 = min(B * T, r0 + (1 << 22))
        st = w[r0:r1] * S + torch.randint(0, S, (r1 - r0,), device=dev, generator=g)
        X[r0:r1, :D] = mt[st] + sd[st] * torch.randn(r1 - r0, D, device=dev, generator=g)
    offs = np.arange(0, B + 1, dtype=np.int64) * T
    batch = eng.PackedBatch(X, torch.from_numpy(offs).to(dev), D, offs)
    a = _np(m.score_words(batch, eng.FP32))
    b = _np(m.score_words(batch, eng.FP32))
    for k in ("best_word", "best_score", "scores"):
        assert np.array_equal(a[k], b[k]), k
    for u in np.random.default_rng(0).choice(B, 256, replace=False):
        x = X[offs[u]:offs[u + 1], :D].cpu().numpy().T
        lps = _oracle_scores(x, means, var, tm, sp)
        assert a["best_word"][u] == int(np.argmax(lps))
        assert_close(a["scores"][u], lps, 1e-6, what=f"utterance {u}")


@pytest.fixture(scope="module")
def corpus_dir(tmp_path_factory):
    from sapr_b200 import synth
    root = tmp_path_factory.mktemp("dense_score_corpus")
    fs = root / "feature_set"; fs.mkdir()
    feats, labels, mu, sd = synth.make_corpus(11 * 8, 11, 8, 13, 40, 60, seed=4243)
    for u, (x, w) in enumerate(zip(feats, labels)):
        np.save(fs / f"sp{u // 11:02d}a_w{u:03d}_{WORDS[w]}.npy", x)
    return root


def test_score_batch_end_to_end(eng, corpus_dir, monkeypatch):
    from sapr_b200.decoder import Decoder
    from sapr_b200.eval import calculate_metrics
    from sapr_b200.mfcc_extract import load_mfccs_by_word
    from sapr_b200.train import train_hmm
    root = corpus_dir
    monkeypatch.chdir(root)
    fs, md = str(root / "feature_set"), str(root / "trained_models")
    train_hmm("hmmlearn", 8, 13, n_iter=3, feature_set_path=fs, models_dir=md, batched=True)
    ev, truth = [], []
    for i, w in enumerate(WORDS):
        fw = load_mfccs_by_word(fs, w)
        ev += fw; truth += [i] * len(fw)
    for prec in ("fp32", "fp64"):
        d = Decoder(models_dir=md, implementation="hmmlearn", n_iter=3, vocab_order=WORDS, precision=prec)
        words, best, ll = d.score_batch(ev, true_labels=truth)
        loop = np.array([[d.models[w].score(f.T) for w in WORDS] for f in ev])
        assert words == [WORDS[int(np.argmax(r))] for r in loop]
        if prec == "fp64":
            assert np.array_equal(ll, loop) and np.array_equal(best, loop.max(axis=1))
        else:
            assert_close(ll, loop, 1e-6, what="loglik")
        cm, acc = d.last_confusion
        ref_cm, ref_acc = calculate_metrics([WORDS[t] for t in truth], words, WORDS)
        present = np.unique(np.concatenate([truth, [WORDS.index(w) for w in words]]))
        assert np.array_equal(cm[np.ix_(present, present)], ref_cm) and cm[:, -1].sum() == 0
        assert acc == ref_acc
    with pytest.raises(ValueError):
        Decoder.score_batch(type("D", (), {"implementation": "custom"})(), ev)
