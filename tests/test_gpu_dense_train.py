"""Batched training of hmmlearn-style word models (DENSE topology): sapr_estep on a DENSE set against sapr_hl_estep per model
(GaussianHMM.fit's E-step), the fp32 fused kernel (csrc/estep_dense.cu) against the float64 verification mode and the oracle,
far-from-model utterances, determinism, the refusals, hmmlearn_hmm.fit_vocabulary against per-model GaussianHMM.fit, and
train_hmm(..., batched=True) -> eval_hmm."""
import copy
import ctypes as C

import numpy as np
import pytest

from conftest import split_features
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
    A = np.zeros((S, S))
    A[0, 1] = 1.0
    for i in range(1, S - 1):
        A[i, i] = aii; A[i, i + 1] = 1 - aii
    A[S - 1, S - 1] = 1.0
    return A


def _synth(M, S, D, B, T_lo, T_hi, dense, seed):
    """M random diagonal-Gaussian models and B utterances drawn from them (lengths U{T_lo..T_hi}), labels interleaved."""
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
    labels[:M] = np.arange(M)                       # every model has utterances
    feats = []
    for w, T in zip(labels, lens):
        st = np.sort(rng.integers(0, S, T)) if not dense else rng.integers(0, S, T)
        feats.append((means[w, st] + np.sqrt(var[w, st]) * rng.standard_normal((T, D))).T.astype(np.float32))
    return feats, labels, (means, var, tm, sp)


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


def _estep(eng, m, feats, labels, precision, want_gamma=False):
    import torch
    batch = eng.PackedBatch.from_features(feats)
    lab = torch.as_tensor(np.asarray(labels, dtype=np.int32), device=batch.X.device)
    stats, ll, gamma = m.estep(batch, lab, None, precision, want_gamma=want_gamma)
    return (stats.cpu().numpy(), ll.cpu().numpy(), None if gamma is None else gamma.cpu().numpy(), batch)


def _hl_estep(eng, m, mi, feats):
    """sapr_hl_estep (GaussianHMM.fit's E-step kernel) on model mi's utterances packed alone."""
    import torch
    b = eng.PackedBatch.from_features(feats)
    st = torch.zeros(m.stats_stride(), dtype=torch.float64, device=b.X.device)
    lp = torch.zeros(b.B, dtype=torch.float64, device=b.X.device)
    m.ctx.check(m.lib.sapr_hl_estep(m.ctx.h, m.h, mi, C.c_void_p(b.X.data_ptr()), b.ldx, C.c_void_p(b.offsets.data_ptr()), b.B,
                                    b.total_frames, C.c_void_p(st.data_ptr()), C.c_void_p(lp.data_ptr())))
    return st.cpu().numpy(), lp.cpu().numpy()


def _model_sets(rung1_d13):
    means, var, tm, sp = _rung1_models(rung1_d13)
    feats = [f.astype(np.float32) for f in split_features(rung1_d13)]
    feats += [feats[0][:, :1], feats[1][:, :2], feats[2][:, :1], feats[3][:, :2]]        # T = 1 and 2
    labels = np.random.default_rng(11).integers(0, 11, len(feats))
    labels[:11] = np.arange(11)
    yield feats, labels, (means, var, tm, sp)
    f2, l2, p2 = _synth(11, 10, 13, 400, 1, 60, True, seed=12)                          # Dirichlet-dense
    yield f2, l2, p2


def test_fp64_equals_per_model_hl_estep(eng, rung1_d13):
    for feats, labels, prm in _model_sets(rung1_d13):
        m = _dense(eng, *prm)
        stats, ll, gamma, _ = _estep(eng, m, feats, labels, eng.FP64, want_gamma=True)
        assert len(set(labels[:40])) > 5                                                  # models interleaved in the batch
        for mi in range(m.M):
            idx = np.nonzero(labels == mi)[0]
            st, lp = _hl_estep(eng, m, mi, [feats[u] for u in idx])
            assert np.array_equal(stats[mi], st), mi                                     # bit for bit
            assert np.array_equal(ll[idx], lp), mi
        assert np.all(np.isfinite(gamma))


def _check_fp32(eng, m, feats, labels, prm, st32, ll32, g32, st64, ll64, g64, gamma_tol=2e-5, occ_frac=0.0):
    means, var, tm, sp = prm
    M, S, D = means.shape
    assert np.all(np.isfinite(st32)) and np.all(np.isfinite(ll32)) and np.all(np.isfinite(g32))
    assert np.max(np.abs(ll32 - ll64) / np.abs(ll64)) <= 1e-6
    assert np.max(np.abs(g32 - g64)) <= gamma_tol
    u32, u64 = m.unpack_stats(st32), m.unpack_stats(st64)
    lens = np.array([f.shape[1] for f in feats])
    from sapr_b200.hmmlearn_hmm import GaussianHMM
    for mi in range(M):
        n_utt, n_fr = np.sum(labels == mi), lens[labels == mi].sum()
        assert np.max(np.abs(u32["start"][mi] - u64["start"][mi])) <= 1e-5 * n_utt
        assert np.max(np.abs(u32["post"][mi] - u64["post"][mi])) <= 1e-5 * n_fr
        assert np.max(np.abs(u32["trans"][mi] - u64["trans"][mi])) <= 1e-5 * n_fr
        hs = []
        for u in (u32, u64):
            h = GaussianHMM(n_components=S, covariance_type="diag", init_params="")
            h.means_, h.covars_, h.transmat_, h.startprob_ = means[mi].copy(), var[mi].copy(), tm[mi].copy(), sp[mi].copy()
            h._do_mstep({k: v[mi] for k, v in u.items()})
            hs.append(h)
        occ = u64["post"][mi] >= max(1.0, occ_frac * n_fr)     # a state without posterior mass has no mean (NaN on both sides)
        sd = np.sqrt(hs[1]._covars[occ])
        assert np.max(np.abs(hs[0].means_[occ] - hs[1].means_[occ]) / sd) <= 1e-4, mi
        assert np.max(np.abs(hs[0]._covars[occ] - hs[1]._covars[occ]) / hs[1]._covars[occ]) <= 1e-3, mi
        assert np.max(np.abs(hs[0].transmat_[occ] - hs[1].transmat_[occ])) <= 1e-5, mi


@pytest.mark.parametrize("S", [4, 10, 16, 32])
@pytest.mark.parametrize("D", [13, 39])
@pytest.mark.parametrize("dense", [False, True])
def test_fp32_against_fp64(eng, S, D, dense):
    feats, labels, prm = _synth(11, S, D, 1100, 20, 90, dense, seed=S * 100 + D + dense)
    m = _dense(eng, *prm)
    st32, ll32, g32, _ = _estep(eng, m, feats, labels, eng.FP32, want_gamma=True)
    st64, ll64, g64, _ = _estep(eng, m, feats, labels, eng.FP64, want_gamma=True)
    # gamma: 2e-5 (the fp32 E-step tolerance of DESIGN §2) except left-to-right models with 16+ states, where the fp32 emission's
    # rounding accumulates along the forced chain (measured worst 1.2e-4; log-likelihoods and M-step results stay in tolerance)
    _check_fp32(eng, m, feats, labels, prm, st32, ll32, g32, st64, ll64, g64, gamma_tol=2e-5 if dense or S <= 10 else 2e-4)


@pytest.mark.parametrize("dense", [False, True])
def test_fp32_far_from_model(eng, dense):
    S, D = 10, 39
    feats, labels, prm = _synth(11, S, D, 440, 20, 80, dense, seed=7 + dense)
    means, var, tm, sp = prm
    sd = np.sqrt(var).max(axis=(0, 1))                                                   # largest state sigma per dim
    feats = [(f + 50.0 * sd[:, None]).astype(np.float32) for f in feats]
    m = _dense(eng, *prm)
    st32, ll32, g32, _ = _estep(eng, m, feats, labels, eng.FP32, want_gamma=True)
    st64, ll64, g64, _ = _estep(eng, m, feats, labels, eng.FP64, want_gamma=True)
    # at 50 sigma an emission is ~5e4 nats, which fp32 resolves to ~3e-3 nats: gamma agrees to 5e-3 (measured worst 2.7e-3), and
    # the M-step is compared on states holding >= 1 % of the model's frames (a state with ~1 frame of mass: variance 2.4e-2 off)
    _check_fp32(eng, m, feats, labels, prm, st32, ll32, g32, st64, ll64, g64, gamma_tol=5e-3, occ_frac=0.01)


def test_large_batch_deterministic_and_oracle(eng):
    M, S, D, B = 11, 10, 13, 20000
    feats, labels, (means, var, tm, sp) = _synth(M, S, D, B, 80, 120, False, seed=31)
    m = _dense(eng, means, var, tm, sp)
    a = _estep(eng, m, feats, labels, eng.FP32)
    b = _estep(eng, m, feats, labels, eng.FP32)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    # a 256-utterance sample against the oracle's float64 E-step (hmmlearn semantics)
    idx = np.sort(np.random.default_rng(0).choice(B, 256, replace=False))
    sf, sl = [feats[u] for u in idx], labels[idx]
    st, ll, _, _ = _estep(eng, m, sf, sl, eng.FP32)
    u32 = m.unpack_stats(st)
    for mi in range(M):
        sel = np.nonzero(sl == mi)[0]
        if len(sel) == 0:
            continue
        X, offs = orc.pack([sf[k] for k in sel])
        o = orc.hl_estep(X, offs, sp[mi], tm[mi], means[mi], var[mi])
        assert np.max(np.abs(ll[sel] - o["loglik"]) / np.abs(o["loglik"])) <= 1e-6
        nfr = offs[-1]
        assert np.max(np.abs(u32["post"][mi] - o["post"])) <= 1e-5 * nfr
        assert np.max(np.abs(u32["trans"][mi] - o["trans"])) <= 1e-5 * nfr
        assert np.max(np.abs(u32["start"][mi] - o["start"])) <= 1e-5 * len(sel)
        mu32, mu = u32["obs"][mi] / u32["post"][mi][:, None], o["obs"] / o["post"][:, None]
        assert np.max(np.abs(mu32 - mu) / np.sqrt(var[mi])) <= 1e-4


def test_refusals(eng):
    import torch
    from sapr_b200._lib import SaprError
    feats, labels, prm = _synth(3, 10, 13, 40, 20, 30, True, seed=1)
    m = _dense(eng, *prm)
    batch = eng.PackedBatch.from_features(feats)
    with pytest.raises(SaprError):
        m.estep(batch, None, None, eng.FP32)
    big = _synth(2, 33, 13, 4, 5, 6, True, seed=2)
    mb = _dense(eng, *big[2])
    bb = eng.PackedBatch.from_features(big[0])
    lab = torch.as_tensor(big[1].astype(np.int32), device=bb.X.device)
    with pytest.raises(SaprError) as ei:
        mb.estep(bb, lab, None, eng.FP32)
    assert ei.value.args[0] == -4 or "S > 32" in str(ei.value)
    mb.estep(bb, lab, None, eng.FP64)                                                    # float64 takes any S sapr_hl_estep takes
    from sapr_b200.hmmlearn_hmm import GaussianHMM, fit_vocabulary
    hs = []
    for mi in range(3):
        h = GaussianHMM(n_components=10, covariance_type="diag", init_params="", n_iter=2)
        h.means_, h.covars_, h.transmat_, h.startprob_ = prm[0][mi], prm[1][mi], prm[2][mi], prm[3][mi]
        hs.append(h)
    with pytest.raises(ValueError):
        fit_vocabulary(hs, [feats[:5], [], feats[5:10]])
    from sapr_b200.train import train_hmm
    with pytest.raises(ValueError):
        train_hmm("custom", batched=True)


def _init_models(prm, n_iter, seed):
    means, var, tm, sp = prm
    rng = np.random.default_rng(seed)
    from sapr_b200.hmmlearn_hmm import GaussianHMM
    hs = []
    for mi in range(means.shape[0]):
        h = GaussianHMM(n_components=means.shape[1], covariance_type="diag", init_params="", n_iter=n_iter, tol=1e-2,
                        params="mc" if mi == 3 else "stmc")
        if mi == 5:
            h.tol = 1e12                                                                 # converges after 2 iterations
        h.means_ = means[mi] + 0.3 * np.sqrt(var[mi]) * rng.standard_normal(means[mi].shape)
        h.covars_ = var[mi] * 1.5
        h.transmat_, h.startprob_ = tm[mi].copy(), sp[mi].copy()
        hs.append(h)
    return hs


def test_fit_vocabulary_fp64_equals_per_model_fit(eng):
    from sapr_b200.hmmlearn_hmm import fit_vocabulary
    feats, labels, prm = _synth(11, 6, 13, 330, 20, 60, False, seed=21)
    per = _init_models(prm, 5, 1)
    bat = copy.deepcopy(per)
    words = [[feats[u] for u in np.nonzero(labels == mi)[0]] for mi in range(11)]
    for h, fs in zip(per, words):
        h.fit(np.concatenate([f.T for f in fs], axis=0), [f.shape[1] for f in fs])
    fit_vocabulary(bat, words, precision="fp64")
    assert per[5].monitor_.iter == 2 and any(h.monitor_.iter == 5 for h in per)
    for a, b in zip(per, bat):
        assert list(a.monitor_.history) == list(b.monitor_.history)
        assert a.monitor_.iter == b.monitor_.iter
        for k in ("means_", "_covars", "transmat_", "startprob_"):
            assert np.array_equal(getattr(a, k), getattr(b, k)), k


def _corpus(n_per_word, seed):
    from sapr_b200 import synth
    feats, labels, _, _ = synth.make_corpus(11 * n_per_word, 11, 8, 13, 40, 60, seed=seed)
    return feats, np.asarray(labels)


def test_fit_vocabulary_fp32_against_fp64(eng, tmp_path):
    import pickle
    from sapr_b200.decoder import Decoder
    from sapr_b200.hmmlearn_hmm import HMMLearnModel, fit_vocabulary
    feats, labels = _corpus(30, 777)
    words = [[feats[u] for u in np.nonzero(labels == w)[0]] for w in range(11)]
    base = [HMMLearnModel(num_states=8, model_name=WORDS[w], n_iter=3, feature_set=feats).model for w in range(11)]
    fits = {}
    for prec in ("fp64", "fp32"):
        ms = fit_vocabulary(copy.deepcopy(base), words, precision=prec)
        d = tmp_path / prec / "hmmlearn"
        d.mkdir(parents=True)
        for w, h in zip(WORDS, ms):
            with open(d / f"{w}_hmmlearn_3.pkl", "wb") as f:
                pickle.dump(h, f)
        fits[prec] = ms
    for a, b in zip(fits["fp32"], fits["fp64"]):
        ha, hb = np.array(a.monitor_.history), np.array(b.monitor_.history)
        assert len(ha) == len(hb) == 3
        assert np.max(np.abs(ha - hb) / np.abs(hb)) <= 1e-5
    test_feats, _ = _corpus(8, 4243)
    rec = {}
    for prec in ("fp64", "fp32"):
        dec = Decoder(models_dir=str(tmp_path / prec), implementation="hmmlearn", n_iter=3, vocab_order=WORDS)
        rec[prec] = dec.decode_batch(test_feats)[0]
    assert rec["fp32"] == rec["fp64"]


@pytest.fixture(scope="module")
def corpus_dir(tmp_path_factory):
    from sapr_b200 import synth
    root = tmp_path_factory.mktemp("dense_train_corpus")
    fs = root / "feature_set"; fs.mkdir()
    feats, labels, mu, sd = synth.make_corpus(11 * 8, 11, 8, 13, 40, 60, seed=4243)
    for u, (x, w) in enumerate(zip(feats, labels)):
        np.save(fs / f"sp{u // 11:02d}a_w{u:03d}_{WORDS[w]}.npy", x)
    return root


def test_train_hmm_batched_end_to_end(corpus_dir, monkeypatch):
    from sapr_b200.eval import eval_hmm
    from sapr_b200.train import train_hmm
    root = corpus_dir
    monkeypatch.chdir(root)
    fs = str(root / "feature_set")
    md_loop, md_bat = str(root / "loop_models"), str(root / "batched_models")
    train_hmm("hmmlearn", 8, 13, n_iter=3, feature_set_path=fs, models_dir=md_loop)
    h_loop = dict(train_hmm.histories)
    out = train_hmm("hmmlearn", 8, 13, n_iter=3, feature_set_path=fs, models_dir=md_bat, batched=True)
    h_bat = dict(train_hmm.histories)
    assert sorted(out) == sorted(WORDS)
    for w in WORDS:
        assert (root / "batched_models" / "hmmlearn" / f"{w}_hmmlearn_3.pkl").exists()
        a, b = np.array(h_bat[w]), np.array(h_loop[w])
        assert len(a) == len(b) and np.max(np.abs(a - b) / np.abs(b)) <= 1e-5, w
    loop = eval_hmm("hmmlearn", fs, model_iter=3, models_dir=md_loop, vocab_order=WORDS, batched=True)
    bat = eval_hmm("hmmlearn", fs, model_iter=3, models_dir=md_bat, vocab_order=WORDS, batched=True)
    assert bat["true_labels"] == loop["true_labels"]
    assert bat["predicted_labels"] == loop["predicted_labels"]
