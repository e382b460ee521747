"""Batched recognition with hmmlearn-style word models (DENSE topology: every state emits, S x S transmat + startprob):
sapr_viterbi on a DENSE set against GaussianHMM.decode / sapr_hl_decode per model + the strict-'>' arg-max of
decoder.py:42-47, the fp32 fused kernel (csrc/viterbi_dense.cu) against the float64 verification mode, the near-tie
re-decoding, the edges of the fp32 range (utterances 50 sigma from every model, transitions below the fp32 range), the host
entry point, the refusals, and train -> evaluate through Decoder / eval_hmm."""
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
    """The reference's initial left-to-right pattern (hmmlearn_hmm.py initialize_transmat): 2S - 2 finite arcs."""
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


def _per_model_fp64(m, batch):
    """sapr_hl_decode (GaussianHMM.decode's kernel) for every model: scores [B, M], int32 paths [M, sum_T]."""
    import torch
    dev = batch.X.device
    sc = np.empty((batch.B, m.M)); paths = []
    for mi in range(m.M):
        lp = torch.zeros(batch.B, dtype=torch.float64, device=dev)
        p = torch.zeros(batch.total_frames, dtype=torch.int32, device=dev)
        m.ctx.check(m.lib.sapr_hl_decode(m.ctx.h, m.h, mi, C.c_void_p(batch.X.data_ptr()), batch.ldx,
                                         C.c_void_p(batch.offsets.data_ptr()), batch.B, batch.total_frames,
                                         C.c_void_p(lp.data_ptr()), C.c_void_p(p.data_ptr())))
        sc[:, mi] = lp.cpu().numpy(); paths.append(p.cpu().numpy())
    return sc, np.stack(paths)


def _argmax_first(sc):
    bw = np.full(sc.shape[0], -1, dtype=np.int32); bs = np.full(sc.shape[0], -np.inf)
    for mi in range(sc.shape[1]):
        take = sc[:, mi] > bs
        bw[take] = mi; bs[take] = sc[take, mi]
    return bw, bs


def _path_score(x_TD, p, means, var, tm, sp):
    lf = orc.emission_diag(x_TD.T.astype(np.float64), means, var, all_emit=True)
    with np.errstate(divide="ignore"):
        lA, lpi = np.log(tm), np.log(sp)
    return lpi[p[0]] + lf[0, p[0]] + float(np.sum(lA[p[:-1], p[1:]] + lf[np.arange(1, len(p)), p[1:]]))


def _rung1_models(g):
    """11 DENSE models from the Rung-1 goldens, built as test_gpu_hmmlearn_mfcc._setup builds one (entry / exit rows made
    emitting next to their neighbours); model 4 starts spread over two states, the rest in state 0 (startprob zeros)."""
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


def test_fp64_equals_per_model_decode(eng, rung1_d13):
    g = rung1_d13
    means, var, tm, sp = _rung1_models(g)
    feats = [f.astype(np.float32) for f in split_features(g)]
    feats += [feats[0][:, :1], feats[1][:, :2], feats[2][:, :1]]         # T = 1 and 2
    m = _dense(eng, means, var, tm, sp)
    batch = eng.PackedBatch.from_features(feats)
    out = m.viterbi(batch, None, eng.FP64, 0, want_scores=True, want_path=True)
    sc, paths = _per_model_fp64(m, batch)
    bw, bs = _argmax_first(sc)
    assert np.array_equal(out["scores"].cpu().numpy(), sc)                      # bit for bit
    assert np.array_equal(out["best_word"].cpu().numpy(), bw)
    assert np.array_equal(out["best_score"].cpu().numpy(), bs)
    got = out["path"].cpu().numpy()
    offs = batch.offsets_host
    for u in range(batch.B):
        a, b = offs[u], offs[u + 1]
        assert np.array_equal(got[a:b], paths[max(bw[u], 0), a:b])
    # GaussianHMM.decode (one model at a time, decoder.py:43) and the oracle restatement
    from sapr_b200.hmmlearn_hmm import GaussianHMM
    for u in list(range(0, batch.B, 17)) + [batch.B - 3, batch.B - 2, batch.B - 1]:
        x = feats[u].T
        lps = []
        for mi in range(11):
            h = GaussianHMM(n_components=10, covariance_type="diag", init_params="")
            h.means_, h.covars_, h.transmat_, h.startprob_ = means[mi], var[mi], tm[mi], sp[mi]
            lp, p = h.decode(x)
            assert lp == sc[u, mi]
            lf = orc.emission_diag(x.T.astype(np.float64), means[mi], var[mi], all_emit=True)
            olp, op = orc.hl_viterbi(lf, sp[mi], tm[mi])
            assert abs(olp - lp) <= 1e-10 * abs(olp)
            assert np.array_equal(op, p)
            lps.append(lp)
        assert int(np.argmax(lps)) == bw[u]


def _check_fp32(ref, out, batch, feats, prm):
    """fp32 against float64: identical words, scores within 1e-6, and paths identical except float64 near-ties: at most 2 % of
    the paths differ, each scoring within 2e-3 of the float64 optimum.  Prints the measured worst cases."""
    means, var, tm, sp = prm
    B = batch.B
    rw, ow = ref["best_word"].cpu().numpy(), out["best_word"].cpu().numpy()
    assert np.array_equal(ow, rw)
    rsc, osc = ref["scores"].cpu().numpy(), out["scores"].cpu().numpy()
    assert_close(osc, rsc, 1e-6, what="scores")
    assert_close(out["best_score"].cpu().numpy(), ref["best_score"].cpu().numpy(), 1e-6, what="best scores")
    fin = np.isfinite(rsc)
    rp, op = ref["path"].cpu().numpy(), out["path"].cpu().numpy()
    offs = batch.offsets_host
    differ = [u for u in range(B) if not np.array_equal(rp[offs[u]:offs[u + 1]], op[offs[u]:offs[u + 1]])]
    rbs = ref["best_score"].cpu().numpy()
    gap = 0.0
    for u in differ:        # float64 near-ties only: the fp32 path scores within 2e-3 of the optimum in float64
        w = rw[u]
        ps = _path_score(feats[u].T, op[offs[u]:offs[u + 1]].astype(np.int64), means[w], var[w], tm[w], sp[w])
        gap = max(gap, rbs[u] - ps)
    print(f"fp32 vs fp64 worst: score {np.max(np.abs(osc[fin] - rsc[fin]) / np.maximum(1.0, np.abs(rsc[fin])), initial=0.0):.2e}, "
          f"paths differing {len(differ)} of {B}, path score gap {gap:.2e}")
    assert len(differ) <= 0.02 * B, len(differ)
    assert gap <= 2e-3


@pytest.mark.parametrize("S", [1, 2, 4, 8, 9, 10, 16, 17, 32])
@pytest.mark.parametrize("D", [13, 39])
@pytest.mark.parametrize("dense", [False, True])
@pytest.mark.parametrize("ragged", [False, True])
@pytest.mark.parametrize("M", [1, 11, 17])
def test_fp32_against_fp64(eng, S, D, dense, ragged, M):
    """The bucket edges 8 / 16 / 32; M = 17 sends model 16 to a second blockIdx.y group of 16 models."""
    B = 300
    feats, labels, (means, var, tm, sp) = _synth(M, S, D, B, 30 if ragged else 60, 90 if ragged else 60, dense,
                                                 seed=S * 1000 + D * 10 + M + 7 * dense + 3 * ragged)
    if M > 1:
        # model M-1 can never score for T >= 2: all start mass on a state with no outgoing arcs (GaussianHMM._check refuses it)
        k = S - 1
        tm[M - 1, k] = 0.0
        sp[M - 1] = 0.0; sp[M - 1, k] = 1.0
    m = _dense(eng, means, var, tm, sp)
    batch = eng.PackedBatch.from_features(feats)
    ref = m.viterbi(batch, None, eng.FP64, 0, want_scores=True, want_path=True)
    out = m.viterbi(batch, None, eng.FP32, 0, want_scores=True, want_path=True)
    if M > 1:
        assert np.all(ref["scores"].cpu().numpy()[:, M - 1] == -np.inf)
    _check_fp32(ref, out, batch, feats, (means, var, tm, sp))


def test_fp32_far_from_every_model(eng):
    """Utterances 50 sigma from every model (emissions of ~5e4 nats per frame), as the scoring suite has them."""
    M, S, D = 11, 10, 39
    feats, _, (means, var, tm, sp) = _synth(M, S, D, 400, 40, 100, False, seed=8)
    sd = np.sqrt(var).mean(axis=(0, 1))
    far = [f + (50.0 * sd * np.sign(np.random.default_rng(u).standard_normal(D)))[:, None].astype(np.float32)
           for u, f in enumerate(feats)]
    m = _dense(eng, means, var, tm, sp)
    batch = eng.PackedBatch.from_features(far)
    ref = m.viterbi(batch, None, eng.FP64, 0, want_scores=True, want_path=True)
    out = m.viterbi(batch, None, eng.FP32, 0, want_scores=True, want_path=True)
    assert np.all(np.isfinite(out["scores"].cpu().numpy()))
    _check_fp32(ref, out, batch, far, (means, var, tm, sp))


@pytest.mark.parametrize("tiny", [1e-50, 1e-45])
def test_fp32_transitions_below_the_fp32_range(eng, tiny):
    """The only arc into state k + 1 has probability 1e-50 (0 in fp32) or 1e-45 (its smallest denormal); the Viterbi reads
    ln A from float64, so the arc stays on the path."""
    M, S, D, k = 11, 10, 13, 4
    feats, _, (means, var, tm, sp) = _synth(M, S, D, 500, 30, 90, False, seed=13)
    for mi in range(M):
        tm[mi, k] = 0.0; tm[mi, k, k] = 1.0 - tiny; tm[mi, k, k + 1] = tiny
        tm[mi, k + 1] = 0.0; tm[mi, k + 1, k + 2] = 1.0
    m = _dense(eng, means, var, tm, sp)
    batch = eng.PackedBatch.from_features(feats)
    ref = m.viterbi(batch, None, eng.FP64, 0, want_scores=True, want_path=True)
    out = m.viterbi(batch, None, eng.FP32, 0, want_scores=True, want_path=True)
    assert np.all(np.isfinite(ref["scores"].cpu().numpy()))
    op, offs = out["path"].cpu().numpy(), batch.offsets_host
    crossed = sum(np.any(op[offs[u]:offs[u + 1]] == k + 1) for u in range(batch.B))
    assert crossed >= 0.5 * batch.B                                             # the case exercises the arc
    _check_fp32(ref, out, batch, feats, (means, var, tm, sp))


def test_no_model_scores_gives_minus_one(eng):
    S, D = 6, 13
    feats, _, (means, var, tm, sp) = _synth(2, S, D, 70, 2, 9, False, seed=5)
    tm[:, S - 1] = 0.0
    sp[:] = 0.0; sp[:, S - 1] = 1.0
    m = _dense(eng, means, var, tm, sp)
    batch = eng.PackedBatch.from_features(feats)
    outs = [m.viterbi(batch, None, p, 0, want_scores=True, want_path=True) for p in (eng.FP64, eng.FP32)]
    for o in outs:
        assert np.all(o["best_word"].cpu().numpy() == -1)
        assert np.all(o["best_score"].cpu().numpy() == -np.inf)
        assert np.all(o["scores"].cpu().numpy() == -np.inf)
    assert np.array_equal(outs[0]["path"].cpu().numpy(), outs[1]["path"].cpu().numpy())


def test_fp32_near_ties_are_redecoded_in_float64(eng, monkeypatch):
    M, S, D, B = 11, 10, 13, 900
    feats, labels, (means, var, tm, sp) = _synth(M, S, D, B, 40, 64, False, seed=77)
    rng = np.random.default_rng(5)
    means[5] = means[3] + 1e-7 * np.sqrt(var[3]) * rng.standard_normal(means[3].shape)
    var[5] = var[3]; tm[5] = tm[3]; sp[5] = sp[3]
    m = _dense(eng, means, var, tm, sp)
    batch = eng.PackedBatch.from_features(feats)
    ref = m.viterbi(batch, None, eng.FP64, 0, want_scores=True, want_path=True)
    out = m.viterbi(batch, None, eng.FP32, 0, want_scores=True, want_path=True)
    flagged = m.ctx.viterbi_flagged()
    rw, ow = ref["best_word"].cpu().numpy(), out["best_word"].cpu().numpy()
    near = np.isin(rw, (3, 5))
    assert near.sum() > 30 and flagged >= near.sum()
    assert np.array_equal(ow, rw)
    assert np.array_equal(out["best_score"].cpu().numpy()[near], ref["best_score"].cpu().numpy()[near])
    assert np.array_equal(out["scores"].cpu().numpy()[near], ref["scores"].cpu().numpy()[near])
    offs = batch.offsets_host
    rp, op = ref["path"].cpu().numpy(), out["path"].cpu().numpy()
    for u in np.nonzero(near)[0]:
        assert np.array_equal(op[offs[u]:offs[u + 1]], rp[offs[u]:offs[u + 1]])
    monkeypatch.setenv("SAPR_EXACT_WORDS", "0")
    raw = m.viterbi(batch, None, eng.FP32, 0, want_scores=False, want_path=False)["best_word"].cpu().numpy()
    assert m.ctx.viterbi_flagged() == 0
    assert np.mean(raw[near] != rw[near]) > 0.05


def test_viterbi_host_dense(eng):
    feats, _, prm = _synth(11, 10, 13, 3000, 40, 120, False, seed=9)
    m = _dense(eng, *prm)
    batch = eng.PackedBatch.from_features(feats)
    dev = m.viterbi(batch, None, eng.FP32, 0, want_path=True)
    Xh = batch.X.cpu().numpy(); offs = batch.offsets_host
    host = m.viterbi_host(Xh, offs, eng.FP32, 0, chunk_utts=1000)
    assert np.array_equal(host["best_word"], dev["best_word"].cpu().numpy())
    assert np.array_equal(host["best_score"], dev["best_score"].cpu().numpy())
    assert np.array_equal(host["path"], dev["path"].cpu().numpy())


def test_dense_refusals(eng):
    from sapr_b200._lib import SaprError
    feats, _, prm = _synth(3, 10, 13, 40, 20, 30, True, seed=1)
    m = _dense(eng, *prm)
    batch = eng.PackedBatch.from_features(feats)
    with pytest.raises(SaprError):
        m.viterbi(batch, None, eng.FP32, 5)
    with pytest.raises(SaprError):
        m.viterbi(batch, None, eng.FP32, 0, all_paths=True)
    import torch
    mou = torch.zeros(batch.B, dtype=torch.int32, device=batch.X.device)
    with pytest.raises(SaprError):
        m.viterbi(batch, mou, eng.FP32, 0)
    big = _synth(2, 33, 13, 4, 5, 6, True, seed=2)[2]
    mb = _dense(eng, *big)
    with pytest.raises(SaprError):
        mb.viterbi(batch, None, eng.FP32, 0)


def test_large_batch_deterministic_and_oracle(eng):
    M, S, D, B = 11, 10, 13, 20000
    feats, _, (means, var, tm, sp) = _synth(M, S, D, B, 80, 120, False, seed=31)
    m = _dense(eng, means, var, tm, sp)
    batch = eng.PackedBatch.from_features(feats)
    a = m.viterbi(batch, None, eng.FP32, 0, want_scores=True, want_path=True)
    b = m.viterbi(batch, None, eng.FP32, 0, want_scores=True, want_path=True)
    for k in ("best_word", "best_score", "scores", "path"):
        assert np.array_equal(a[k].cpu().numpy(), b[k].cpu().numpy()), k
    rng = np.random.default_rng(0)
    offs = batch.offsets_host
    bw, bs, p = a["best_word"].cpu().numpy(), a["best_score"].cpu().numpy(), a["path"].cpu().numpy()
    same = 0
    sample = rng.choice(B, 256, replace=False)
    for u in sample:
        x = feats[u].astype(np.float64)
        res = [orc.hl_viterbi(orc.emission_diag(x, means[mi], var[mi], all_emit=True), sp[mi], tm[mi]) for mi in range(M)]
        lps = np.array([r[0] for r in res])
        assert bw[u] == int(np.argmax(lps))
        assert abs(bs[u] - lps.max()) <= 1e-6 * abs(lps.max())
        same += np.array_equal(p[offs[u]:offs[u + 1]], res[bw[u]][1])
    assert same >= 0.98 * len(sample)


@pytest.fixture(scope="module")
def corpus_dir(tmp_path_factory):
    from sapr_b200 import synth
    root = tmp_path_factory.mktemp("dense_corpus")
    fs = root / "feature_set"; fs.mkdir()
    feats, labels, mu, sd = synth.make_corpus(11 * 8, 11, 8, 13, 40, 60, seed=4243)
    for u, (x, w) in enumerate(zip(feats, labels)):
        np.save(fs / f"sp{u // 11:02d}a_w{u:03d}_{WORDS[w]}.npy", x)
    return root, feats, labels


def test_train_eval_hmmlearn_batched(corpus_dir, monkeypatch):
    from sklearn.metrics import confusion_matrix
    from sapr_b200.decoder import Decoder
    from sapr_b200.eval import eval_hmm
    from sapr_b200.mfcc_extract import load_mfccs_by_word
    from sapr_b200.train import train_hmm
    root, feats, labels = corpus_dir
    monkeypatch.chdir(root)
    fs, md = str(root / "feature_set"), str(root / "trained_models")
    train_hmm("hmmlearn", 8, 13, n_iter=3, feature_set_path=fs, models_dir=md)
    loop = eval_hmm("hmmlearn", fs, model_iter=3, models_dir=md, vocab_order=WORDS)
    bat = eval_hmm("hmmlearn", fs, model_iter=3, models_dir=md, vocab_order=WORDS, batched=True)
    assert bat["true_labels"] == loop["true_labels"]
    assert bat["predicted_labels"] == loop["predicted_labels"]
    assert bat["confusion_matrix"].equals(loop["confusion_matrix"])
    for w in WORDS:
        for a, b in zip(loop["results"][w], bat["results"][w]):
            assert abs(a["log_likelihood"] - b["log_likelihood"]) <= 1e-6 * abs(a["log_likelihood"])
    t_idx = [WORDS.index(w) for w in bat["true_labels"]]
    p_idx = [WORDS.index(w) for w in bat["predicted_labels"]]
    assert np.array_equal(bat["confusion_matrix"].values, confusion_matrix(t_idx, p_idx))
    # the float64 verification mode equals the per-sequence loop exactly
    d = Decoder(models_dir=md, implementation="hmmlearn", n_iter=3, vocab_order=WORDS, precision="fp64")
    ev = [f for w in WORDS for f in load_mfccs_by_word(fs, w)]
    words, scores, paths = d.decode_batch(ev)
    for u, f in enumerate(ev):
        w, s, st = d.decode_sequence(f.T)
        assert words[u] == w and scores[u] == s and paths[u] == list(st)
