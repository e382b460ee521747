"""Parity of the fused CUDA kernels (through the C ABI) against the reference-generated golden vectors and
the CPU oracle.  Run with ``-m gpu`` on a B200."""
import numpy as np
import pytest

from conftest import assert_close, split_features
from oracle import oracle as orc

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from sapr_b200 import engine
    return engine


def _models(eng, g, M=None):
    A, means, var = g["A"], g["means"], g["var"]
    M = M or means.shape[0]
    m = eng.WordModels(M, int(g["N"]), int(g["D"]))
    m.set(means[:M], var[:M], A[:M])
    return m


def path_score(E, A, path):
    """Score of a given state path under the reference's decode rules (custom_hmm.py:469-503)."""
    S = E.shape[1]
    with np.errstate(divide="ignore"):
        lA = np.log(A)
    s = 0.0
    prev = path[0]
    s += 0.0 if prev == 0 else (lA[0, 1] + E[0, 1] if prev == 1 else -np.inf)
    for t in range(1, len(path)):
        j = path[t]
        s += lA[prev, j] + (E[t, j] if 0 < j < S - 1 else 0.0)
        prev = j
    return s


def _P(eng, prec):
    return {"fp64": eng.FP64, "fp32": eng.FP32, "fp32_simt": eng.FP32_SIMT}[prec]


@pytest.mark.parametrize("name", ["rung1_d39", "rung1_d13"])
def test_tensor_core_emission_tile(eng, name, request):
    """The tcgen05 emission (fp16 hi/lo split operands, fp32 TMEM accumulate) against the float64 oracle
    emission of every model: absolute error of the log-density."""
    g = request.getfixturevalue(name)
    feats = split_features(g)
    m = _models(eng, g)
    batch = eng.PackedBatch.from_features(feats)
    E = m.tc_emission(batch).cpu().numpy()
    offs = batch.offsets_host
    worst = 0.0
    for u in range(batch.B):
        for w in range(m.M):
            ref = orc.emission_diag(feats[u], g["means"][w], g["var"][w])[:, 1:-1]
            got = E[offs[u]:offs[u + 1], w * 8:(w + 1) * 8]
            worst = max(worst, float(np.max(np.abs(got - ref) / (1e-4 + 5e-7 * np.abs(ref)))))
    # stated tolerance: |E_tc - E_f64| <= 1e-4 + 5e-7 |E|.  The tensor core truncates its fp32 accumulator on every
    # K step (observed bias ~ +2e-7 |E|); measured worst case on these sets: 2.2e-4 at |E| ~ 900 (D = 39), 5.5e-5 (D = 13).
    assert worst < 1.0, worst


@pytest.mark.parametrize("name", ["rung1_d39", "rung1_d13"])
@pytest.mark.parametrize("prec", ["fp64", "fp32", "fp32_simt"])
def test_viterbi_all_models_vs_reference(eng, name, prec, request):
    g = request.getfixturevalue(name)
    feats = split_features(g)
    m = _models(eng, g)
    batch = eng.PackedBatch.from_features(feats)
    P = _P(eng, prec)
    out = m.viterbi(batch, None, P, 0, want_scores=True, want_path=True, all_paths=True)
    sc = out["scores"].cpu().numpy(); bw = out["best_word"].cpu().numpy()
    allp = out["all_paths"].cpu().numpy(); bp = out["path"].cpu().numpy()
    offs = batch.offsets_host
    # float64 verification mode: rel 1e-12; fp32 production mode: rel 1e-6 (stated tolerance, SURVEY 8c)
    assert_close(sc, g["dec_scores"], 1e-12 if prec == "fp64" else 1e-6, what="scores")
    assert np.array_equal(bw, g["dec_best"])
    assert_close(out["best_score"].cpu().numpy(), g["dec_scores"][np.arange(len(bw)), bw],
                 1e-12 if prec == "fp64" else 1e-6, what="best_score")
    near_ties = 0
    for u in range(batch.B):
        T = feats[u].shape[1]
        assert np.array_equal(bp[offs[u]:offs[u + 1]], allp[bw[u], offs[u]:offs[u + 1]])
        for w in range(m.M):
            got = allp[w, offs[u]:offs[u + 1]].astype(np.int32)
            ref = g["dec_paths"][u, w, :T].astype(np.int32)
            if np.array_equal(got, ref):
                continue
            assert prec != "fp64", f"float64 path differs for utt {u} model {w}"
            # documented near-tie policy: the fp32 path must score within 2e-3 of the optimum in float64
            E = orc.emission_diag(feats[u], g["means"][w], g["var"][w])
            assert abs(path_score(E, g["A"][w], got) - g["dec_scores"][u, w]) < 2e-3, (u, w)
            near_ties += 1
    assert near_ties <= 0.02 * batch.B * m.M


def test_viterbi_first_frames_and_own_model(eng, rung1_d13):
    """SURVEY D3: the reference walks only features.shape[0] = D frames; and the own-model mode."""
    import torch
    g = rung1_d13
    feats = split_features(g)
    m = _models(eng, g)
    batch = eng.PackedBatch.from_features(feats)
    D = int(g["D"])
    out = m.viterbi(batch, None, eng.FP64, D, want_scores=True, want_path=True)
    X, offs = orc.pack(feats)
    bw, bs, sc, bp = orc.viterbi_batch(X, offs, g["A"], g["means"], g["var"], first_frames=D)
    assert np.array_equal(out["best_word"].cpu().numpy(), bw)
    assert_close(out["scores"].cpu().numpy(), sc, 1e-12, what="scores")
    p = out["path"].cpu().numpy()
    for u in range(batch.B):
        assert np.array_equal(p[offs[u]:offs[u] + D], bp[offs[u]:offs[u] + D])
    # own-model mode: each utterance against its label's model only
    lab = torch.as_tensor(g["labels"].astype(np.int32), device="cuda")
    out2 = m.viterbi(batch, lab, eng.FP64, 0, want_scores=True, want_path=True)
    assert np.array_equal(out2["best_word"].cpu().numpy(), g["labels"])
    assert_close(out2["best_score"].cpu().numpy(), g["dec_scores"][np.arange(batch.B), g["labels"]], 1e-12, what="own")
    p2 = out2["path"].cpu().numpy()
    for u in range(batch.B):
        T = feats[u].shape[1]
        assert np.array_equal(p2[offs[u]:offs[u + 1]], g["dec_paths"][u, g["labels"][u], :T])
    with pytest.raises(IndexError):
        m.viterbi(batch, None, eng.FP64, 10 ** 6)


@pytest.mark.parametrize("T", [2, 5, 8, 9, 10])
def test_viterbi_short_utterances(eng, edge, T):
    """T <= N: the exit state is never reachable -> score -inf, path = zeros + [S-1] (custom_hmm.py:505-512)."""
    x = edge[f"T{T}_x"].astype(np.float64).T
    m = eng.WordModels(2, 8, 13)
    m.set(edge["means"], edge["var"], edge["A"])
    batch = eng.PackedBatch.from_features([x])
    for P in (eng.FP64, eng.FP32, eng.FP32_SIMT):
        out = m.viterbi(batch, None, P, 0, want_scores=True, want_path=True, all_paths=True)
        assert np.array_equal(out["all_paths"].cpu().numpy()[0], edge[f"T{T}_dec_path"])
        assert_close(out["scores"].cpu().numpy()[0, 0], edge[f"T{T}_dec_score"], 1e-12 if P == eng.FP64 else 1e-6, what="score")
    # ragged tile: the same short utterance next to longer ones in one 128-row tensor-core tile
    long_x = np.tile(x, (1, 20))[:, :37]
    b2 = eng.PackedBatch.from_features([long_x, x, long_x[:, :21]])
    o_tc = m.viterbi(b2, None, eng.FP32, 0, want_scores=True, all_paths=True)
    o_64 = m.viterbi(b2, None, eng.FP64, 0, want_scores=True, all_paths=True)
    assert_close(o_tc["scores"].cpu().numpy(), o_64["scores"].cpu().numpy(), 1e-6, what="ragged scores")
    assert np.array_equal(o_tc["all_paths"].cpu().numpy()[0, 37:37 + T], edge[f"T{T}_dec_path"])


@pytest.mark.parametrize("name", ["rung1_d39", "rung1_d13", "rung1_mismatch_d39"])
@pytest.mark.parametrize("prec", ["fp64", "fp32"])
def test_estep_vs_reference(eng, name, prec, request):
    import torch
    g = request.getfixturevalue(name)
    if name == "rung1_mismatch_d39":
        assert int((g["es_xi_rows_zero"] >= 39).sum()) >= 1      # the golden exercises the D10 underflow (whole utterances without xi)
    feats = split_features(g)
    m = _models(eng, g)
    batch = eng.PackedBatch.from_features(feats)
    lab = torch.as_tensor(g["labels"].astype(np.int32), device="cuda")
    P = eng.FP64 if prec == "fp64" else eng.FP32
    for order in (None, eng.group_by_model(lab)):
        stats, ll, gamma = m.estep(batch, lab, order, P, want_gamma=True)
        st = m.unpack_stats(stats)
        rl, ra = (1e-12, 1e-10) if prec == "fp64" else (1e-6, 1e-5)
        assert_close(ll.cpu().numpy(), g["es_loglik"], rl, what="loglik")
        assert_close(gamma.cpu().numpy(), g["es_gamma"][:, 1:-1], 0, ra, what="gamma")
        S = m.S
        emit = (np.arange(S) > 0) & (np.arange(S) < S - 1)
        for w in range(m.M):
            sel = g["labels"] == w
            n = max(1, int(sel.sum()))
            assert_close(st["G"][w], g["es_G"][sel].sum(0) * emit, 0, ra * 50 * n, what="G")
            assert_close(st["Xi"][w], g["es_xi_self"][sel].sum(0) * emit, 0, ra * 50 * n, what="Xi")
            assert_close(st["occ"][w], g["es_occ"][sel].sum(0) * emit, 0, ra * 50 * n, what="occ")
        # feature sums against the oracle's batched leg (same pivot = current mean)
        X, offs = orc.pack(feats)
        ost, _ = orc.estep_batch(X, offs, g["labels"], g["A"], g["means"], g["var"])
        D = m.D
        o1 = ost[:, 3 * S:3 * S + S * D].reshape(m.M, S, D); o2 = ost[:, 3 * S + S * D:].reshape(m.M, S, D)
        scale = np.sqrt(g["var"])                       # per-dim sigma: sums scale with it
        tol = 1e-9 if prec == "fp64" else 2e-4
        assert np.max(np.abs(st["s1"] - o1) / scale) < tol * 60
        assert np.max(np.abs(st["s2"] - o2) / scale ** 2) < tol * 60 * 10


@pytest.mark.parametrize("name", ["rung1_d39", "rung1_d13", "rung1_mismatch_d39"])
@pytest.mark.parametrize("prec", ["fp64", "fp32"])
def test_mstep_vs_reference_baum_welch_iteration(eng, name, prec, request):
    """One E-step + M-step for all words at once == the reference's baum_welch(max_iter=1) per word
    (Rung-1 ladder): A, means and the DIAGONAL of the reference's full covariances."""
    import torch
    g = request.getfixturevalue(name)
    feats = split_features(g)
    m = _models(eng, g)
    batch = eng.PackedBatch.from_features(feats)
    lab = torch.as_tensor(g["labels"].astype(np.int32), device="cuda")
    floor_v = 0.001 * float(np.mean(np.diag(g["global_cov"])))
    hist = eng.train_words(m, batch, lab, 1, floor_v, eng.FP64 if prec == "fp64" else eng.FP32)
    means, var, A, _ = m.get()
    rt = 1e-10 if prec == "fp64" else 1e-5
    assert_close(hist[0], g["bw1_hist"], 1e-12 if prec == "fp64" else 1e-6, what="hist")
    assert_close(A, g["bw1_A"], rt, atol=rt, what="A")
    sig = np.sqrt(g["var"])
    assert np.max(np.abs(means - g["bw1_mean"]) / sig) < (1e-9 if prec == "fp64" else 1e-4), "means"
    ref_var = np.diagonal(g["bw1_cov"], axis1=2, axis2=3)
    emit = slice(1, m.S - 1)
    assert np.max(np.abs(var[:, emit] - ref_var[:, emit]) / g["var"][:, emit]) < (1e-8 if prec == "fp64" else 1e-3), "variances"
    assert np.all(var[:, 0] == 0) and np.all(var[:, -1] == 0) and np.all(means[:, 0] == 0)


def test_moderate_batch_against_oracle(eng):
    """2048 ragged utterances x 11 models (seconds on the oracle): words/paths bit-exact in float64,
    near-tie accounting in fp32; E-step statistics; host-buffer call equals the device call."""
    import torch
    from sapr_b200 import synth
    feats, labels, mu, sd = synth.make_corpus(2048, 11, 8, 39, 60, 90, seed=7)
    A, means, var = synth.truth_models(mu, sd, 0.9)
    m = eng.WordModels(11, 8, 39)
    m.set(means, var, A)
    batch = eng.PackedBatch.from_features(feats)
    X, offs = orc.pack(feats)
    bw, bs, sc, bp = orc.viterbi_batch(X, offs, A, means, var)
    o64 = m.viterbi(batch, None, eng.FP64, 0, want_scores=True)
    assert np.array_equal(o64["best_word"].cpu().numpy(), bw)
    assert np.array_equal(o64["path"].cpu().numpy().astype(np.int32), bp)
    assert_close(o64["scores"].cpu().numpy(), sc, 1e-12, what="scores64")
    for P in (eng.FP32_SIMT, eng.FP32):          # SIMT emission, then the tensor-core emission (kept as o32)
        o32 = m.viterbi(batch, None, P, 0, want_scores=True)
        assert_close(o32["scores"].cpu().numpy(), sc, 1e-6, what="scores32")
        w32 = o32["best_word"].cpu().numpy()
        bad = np.nonzero(w32 != bw)[0]
        for u in bad:   # a different word is only acceptable on a float64 near-tie between the two words
            assert abs(sc[u, w32[u]] - sc[u, bw[u]]) < 1e-5 * abs(sc[u, bw[u]]), u
        assert len(bad) <= 2
        pm = np.mean(o32["path"].cpu().numpy().astype(np.int32) == bp)
        assert pm > 0.9995, f"fp32 path agreement {pm}"
    # host-buffer entry: same answers
    Xh, offh = synth.pack_frame_major(feats)
    oh = m.viterbi_host(Xh, offh, eng.FP32, 0, chunk_utts=500)
    assert np.array_equal(oh["best_word"], w32)
    assert np.array_equal(oh["path"], o32["path"].cpu().numpy())
    assert np.array_equal(oh["best_score"], o32["best_score"].cpu().numpy())
    # E-step
    lab = torch.as_tensor(labels, device="cuda")
    ost, oll = orc.estep_batch(X, offs, labels, A, means, var)
    for P, rl, ra in ((eng.FP64, 1e-12, 1e-9), (eng.FP32, 1e-6, 3e-5)):
        stats, ll, _ = m.estep(batch, lab, None, P)
        assert_close(ll.cpu().numpy(), oll, rl, what="loglik")
        st = stats.cpu().numpy()
        S = 10
        occ = ost[:, 2 * S:3 * S]
        assert np.max(np.abs(st[:, :3 * S] - ost[:, :3 * S])) < ra * 200 * 10
        d1 = np.abs(st[:, 3 * S:] - ost[:, 3 * S:])
        assert np.max(d1) < ra * 200 * 50
    # 1-vs-2 shard equality of the reduced statistics (what the NCCL all-reduce sums)
    from sapr_b200.dist import shard_bounds
    tot = None
    for (a, b) in shard_bounds(offh, 2):
        sub = eng.PackedBatch.from_features(feats[a:b])
        s, _, _ = m.estep(sub, torch.as_tensor(labels[a:b], device="cuda"), None, eng.FP64)
        tot = s if tot is None else tot + s
    full, _, _ = m.estep(batch, lab, None, eng.FP64)
    assert_close(tot.cpu().numpy(), full.cpu().numpy(), 1e-12, atol=1e-9, what="sharded stats")


@pytest.mark.parametrize("B,M,D,T,first", [(300, 11, 39, 37, 0), (129, 5, 13, 24, 0), (128, 11, 39, 9, 0), (77, 3, 20, 8, 0),
                                           (260, 11, 13, 40, 13), (300, 11, 30, 37, 0), (260, 8, 24, 24, 0)])
def test_viterbi_equal_length_batch_tma_vs_oracle(eng, B, M, D, T, first, monkeypatch):
    """Equal-length batches (the BASELINE cfg-2 shape) take one of the TMA-fed kernels, chosen by shape: k_viterbi_v4 for
    10 or 4 feature chunks (D 32-39, 8-15) and M >= 4; k_viterbi_v3 for 8 chunks (D 24-31) and 8 <= M <= 12 (the last two
    shapes); k_viterbi_tma otherwise (M = 3).  Words, scores and paths against the CPU oracle (custom_hmm.py:462-514 x all
    models + decoder.py:42-47); batch sizes that are not a multiple of the 128-utterance tile (zero-filled rows), T down to N
    (exit never reachable: -inf), first_frames (D3); and the call with SAPR_TMA=0 (per-row bulk-copy kernel where k_viterbi_tma
    ran) must agree with it on words and to 1e-6 on scores."""
    from sapr_b200 import synth
    feats, labels, mu, sd = synth.make_corpus(B, M, 8, D, T, T, seed=1000 + B + T)
    A, means, var = synth.truth_models(mu, sd, 0.9)
    m = eng.WordModels(M, 8, D)
    m.set(means, var, A)
    batch = eng.PackedBatch.from_features(feats)
    X, offs = orc.pack(feats)
    bw, bs, sc, bp = orc.viterbi_batch(X, offs, A, means, var, first_frames=first)
    l0 = m.ctx.launches()
    out = m.viterbi(batch, None, eng.FP32, first, want_scores=True, want_path=True)
    assert m.ctx.launches() > l0
    got = out["scores"].cpu().numpy()
    assert_close(got, sc, 1e-6, what="scores (tma)")
    w = out["best_word"].cpu().numpy()
    for u in np.nonzero(w != bw)[0]:
        assert abs(sc[u, w[u]] - sc[u, bw[u]]) < 1e-5 * abs(sc[u, bw[u]]), u
    assert np.sum(w != bw) <= 1
    walked = first if first else T
    pg = out["path"].cpu().numpy().astype(np.int32).reshape(B, T)[:, :walked]
    pr = bp.reshape(B, T)[:, :walked] if bp.size == B * T else bp.reshape(B, -1)[:, :walked]
    if np.isfinite(sc).all():
        assert np.mean(pg == pr) > 0.999, np.mean(pg == pr)
    monkeypatch.setenv("SAPR_TMA", "0")
    out0 = m.viterbi(batch, None, eng.FP32, first, want_scores=True, want_path=True)
    assert_close(out0["scores"].cpu().numpy(), got, 1e-6, what="scores (bulk-copy kernel vs tma kernel)")
    assert np.mean(out0["best_word"].cpu().numpy() == w) > 0.995


def test_estep_short_and_ragged_utterances_tc_vs_float64(eng):
    """The tensor-core E-step (fp32) against the float64 verification kernel on the shapes the reference's own
    recursions treat specially: T = 1, 2 (gamma rows NaN / one-hot, custom_hmm.py:252-255), T <= N (exit state
    unreachable), T = N + 1, ragged lengths inside one 128-utterance tile, several models per tile."""
    import torch
    from sapr_b200 import synth
    rng = np.random.default_rng(5)
    lens = [1, 2, 5, 8, 9, 10, 17, 33, 64, 3, 9, 12] + list(rng.integers(9, 70, size=200))
    feats, labels, mu, sd = synth.make_corpus(len(lens), 11, 8, 39, 70, 70, seed=3)
    feats = [f[:, :T] for f, T in zip(feats, lens)]
    A, means, var = synth.truth_models(mu, sd, 0.9)
    m = eng.WordModels(11, 8, 39)
    m.set(means, var, A)
    batch = eng.PackedBatch.from_features(feats)
    lab = torch.as_tensor(labels, device="cuda")
    s64, l64, g64 = m.estep(batch, lab, None, eng.FP64, want_gamma=True)
    s32, l32, g32 = m.estep(batch, lab, None, eng.FP32, want_gamma=True)
    assert_close(l32.cpu().numpy(), l64.cpu().numpy(), 1e-6, what="loglik")
    assert_close(g32.cpu().numpy(), g64.cpu().numpy(), 0, 2e-5, what="gamma")
    a, b = s32.cpu().numpy(), s64.cpu().numpy()
    assert np.array_equal(np.isnan(a), np.isnan(b))
    ok = ~np.isnan(b)
    assert np.max(np.abs(a[ok] - b[ok]) / (1.0 + np.abs(b[ok]))) < 2e-4


def test_launch_counter_and_errors(eng):
    from sapr_b200 import _lib
    ctx = _lib.default_context()
    n0 = ctx.launches()
    m = eng.WordModels(1, 8, 13)
    with pytest.raises(_lib.SaprError):
        m.viterbi(eng.PackedBatch.from_features([np.zeros((13, 20), dtype=np.float32)]))   # parameters not set
    assert ctx.launches() >= n0
    with pytest.raises(_lib.SaprError):
        eng.WordModels(1, 0, 13)


@pytest.mark.parametrize("D", [12, 13, 40, 44])
def test_estep_feature_dims_vs_oracle(eng, D):
    """E-step statistics for feature dimensions with (13) and without (12, 40, 44: D a multiple of 4) a padding column: the
    statistics kernel takes sum_t gamma from a constant-1 padding dim when there is one and from explicit sums otherwise.
    Several tiles per model, ragged lengths; tensor-core path against the float64 oracle."""
    import torch
    from sapr_b200 import synth
    feats, labels, mu, sd = synth.make_corpus(1500, 11, 8, D, 30, 50, seed=100 + D)
    A, means, var = synth.truth_models(mu, sd, 0.9)
    m = eng.WordModels(11, 8, D)
    m.set(means, var, A)
    batch = eng.PackedBatch.from_features(feats)
    X, offs = orc.pack(feats)
    lab = torch.as_tensor(labels, device="cuda")
    ost, oll = orc.estep_batch(X, offs, labels, A, means, var)
    S = 10
    scale = np.maximum(1.0, np.abs(ost))
    for P, rl, ra in ((eng.FP64, 1e-12, 1e-9), (eng.FP32, 1e-6, 2e-4)):
        stats, ll, _ = m.estep(batch, lab, None, P)
        assert_close(ll.cpu().numpy(), oll, rl, what=f"loglik D={D}")
        st = stats.cpu().numpy()
        assert np.max(np.abs(st[:, :3 * S] - ost[:, :3 * S]) / scale[:, :3 * S]) < ra, "occupancies"
        assert np.max(np.abs(st[:, 3 * S:] - ost[:, 3 * S:]) / scale[:, 3 * S:]) < ra * 10, "feature sums"


@pytest.mark.parametrize("ragged", [False, True])
def test_fp32_word_near_ties_are_redecoded_in_float64(eng, ragged, monkeypatch):
    """fp32 production mode: an utterance whose two best word scores are closer than fp32 resolves is flagged by the arg-max
    kernel and re-decoded in float64 inside the same call, so the recognised word (decoder.py:42-47, strict > over the models),
    its score and its path are the verification mode's.  Two word models that differ by 1e-7 sigma make most margins far smaller
    than the fp32 score error; equal-length batches take k_viterbi_v4, ragged ones k_viterbi_tc."""
    import torch
    from sapr_b200 import synth
    B, M, D = 900, 11, 39
    feats, labels, mu, sd = synth.make_corpus(B, M, 8, D, 40, 64 if ragged else 40, seed=77)
    A, means, var = synth.truth_models(mu, sd, 0.9)
    rng = np.random.default_rng(5)
    means[5] = means[3] + 1e-7 * np.sqrt(var[3]) * rng.standard_normal(means[3].shape)
    var[5] = var[3]; A[5] = A[3]
    m = eng.WordModels(M, 8, D)
    m.set(means, var, A)
    batch = eng.PackedBatch.from_features(feats)
    ref = m.viterbi(batch, None, eng.FP64, 0, want_scores=True, want_path=True)
    out = m.viterbi(batch, None, eng.FP32, 0, want_scores=True, want_path=True)
    flagged = m.ctx.viterbi_flagged()
    rw, ow = ref["best_word"].cpu().numpy(), out["best_word"].cpu().numpy()
    near = np.isin(rw, (3, 5))
    assert near.sum() > 30 and flagged >= near.sum()                        # every 3-vs-5 utterance is a near-tie
    assert np.array_equal(ow, rw)                                           # words: exactly the float64 ones
    rs, os_ = ref["best_score"].cpu().numpy(), out["best_score"].cpu().numpy()
    assert np.array_equal(os_[near], rs[near])                              # re-decoded utterances carry the float64 score ...
    offs = batch.offsets_host
    rp, op = ref["path"].cpu().numpy(), out["path"].cpu().numpy()
    for u in np.nonzero(near)[0][:200]:
        assert np.array_equal(op[offs[u]:offs[u + 1]], rp[offs[u]:offs[u + 1]])   # ... and the float64 path
    assert_close(out["scores"].cpu().numpy(), ref["scores"].cpu().numpy(), 1e-6, what="scores")
    monkeypatch.setenv("SAPR_EXACT_WORDS", "0")                             # without the pass fp32 cannot tell the two models apart
    raw = m.viterbi(batch, None, eng.FP32, 0, want_scores=False, want_path=False)["best_word"].cpu().numpy()
    assert m.ctx.viterbi_flagged() == 0
    assert np.mean(raw[near] != rw[near]) > 0.05


def test_viterbi_blocked_forward_arc_scores_minus_inf(eng):
    """A word model whose chain is cut (A[j, j+1] = 0) cannot reach the exit state: custom_hmm.py:462-514 returns -inf for it and
    decoder.py:42-47 never picks it.  The equal-length fp32 kernel folds the transition constants out of its recursion (their sum
    is added to the final score only), so this is the case where that sum is -inf; words / scores of the other models must not
    be disturbed."""
    from sapr_b200 import synth
    B, M, D, T = 384, 11, 39, 48
    feats, labels, mu, sd = synth.make_corpus(B, M, 8, D, T, T, seed=91)
    A, means, var = synth.truth_models(mu, sd, 0.9)
    A[4, 3, 3] += A[4, 3, 4]; A[4, 3, 4] = 0.0                  # model 4: state 3 can no longer advance
    m = eng.WordModels(M, 8, D)
    m.set(means, var, A)
    batch = eng.PackedBatch.from_features(feats)
    X, offs = orc.pack(feats)
    with np.errstate(divide="ignore"):
        bw, bs, sc, bp = orc.viterbi_batch(X, offs, A, means, var)
    assert np.all(np.isneginf(sc[:, 4])) and np.all(bw != 4)
    out = m.viterbi(batch, None, eng.FP32, 0, want_scores=True, want_path=True)
    got = out["scores"].cpu().numpy()
    assert np.all(np.isneginf(got[:, 4]))
    assert_close(got, sc, 1e-6, what="scores")
    assert np.array_equal(out["best_word"].cpu().numpy(), bw)
    assert np.mean(out["path"].cpu().numpy() == bp) > 0.999


def test_viterbi_equal_length_multi_chunk(eng, monkeypatch):
    """Batches whose back-pointer scratch exceeds 1 GB are decoded in chunks of utterances (335 k at cfg 2); SAPR_V_CHUNK forces
    that path at a small size: words, scores, paths and the near-tie re-decoding must equal the single-chunk call."""
    from sapr_b200 import synth
    feats, labels, mu, sd = synth.make_corpus(1000, 11, 8, 39, 40, 40, seed=17)
    A, means, var = synth.truth_models(mu, sd, 0.9)
    means[7] = means[2] + 1e-7 * np.sqrt(var[2]); var[7] = var[2]; A[7] = A[2]        # some near-ties in every chunk
    m = eng.WordModels(11, 8, 39)
    m.set(means, var, A)
    batch = eng.PackedBatch.from_features(feats)
    one = m.viterbi(batch, None, eng.FP32, 0, want_scores=True, want_path=True)
    f1 = m.ctx.viterbi_flagged()
    monkeypatch.setenv("SAPR_V_CHUNK", "256")
    many = m.viterbi(batch, None, eng.FP32, 0, want_scores=True, want_path=True)
    assert m.ctx.viterbi_flagged() == f1 and f1 > 0
    for k in ("best_word", "best_score", "scores", "path"):
        assert np.array_equal(one[k].cpu().numpy(), many[k].cpu().numpy()), k


@pytest.mark.parametrize("M,D", [(11, 39), (7, 36), (5, 13), (12, 15)])
def test_viterbi_partial_round_two_launches(eng, monkeypatch, M, D):
    """A batch whose tile count is not a multiple of the SM count runs as two launches (full rounds, then the partial round, with
    the first part's arg-max / back-trace on a second stream beside it; the partial round as two CTAs per tile, one accumulator
    column half each, when the model groups split at a multiple of 16 columns -- not for M = 5).  Words, scores, paths and the
    near-tie re-decoding must equal the single-launch call bit for bit, and utterances on both sides of the split must agree
    with the CPU oracle."""
    import torch
    from sapr_b200 import synth
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    B, T = sms * 128 + 300, 16                                         # one full round + three tiles (the last one partial)
    feats, labels, mu, sd = synth.make_corpus(B, M, 8, D, T, T, seed=23 + M)
    A, means, var = synth.truth_models(mu, sd, 0.9)
    means[3] = means[2] + 1e-7 * np.sqrt(var[2]); var[3] = var[2]; A[3] = A[2]        # near-ties in both parts
    m = eng.WordModels(M, 8, D)
    m.set(means, var, A)
    batch = eng.PackedBatch.from_features(feats)
    two = m.viterbi(batch, None, eng.FP32, 0, want_scores=True, want_path=True)
    f2 = m.ctx.viterbi_flagged()
    monkeypatch.setenv("SAPR_V_TAIL", "0")
    one = m.viterbi(batch, None, eng.FP32, 0, want_scores=True, want_path=True)
    assert m.ctx.viterbi_flagged() == f2 and f2 > 0
    for k in ("best_word", "best_score", "scores", "path"):
        assert np.array_equal(one[k].cpu().numpy(), two[k].cpu().numpy()), k
    split = sms * 128
    pick = np.r_[0:150, split - 150:split + 150, B - 150:B]
    sub = [feats[i] for i in pick]
    X, offs = orc.pack(sub)
    with np.errstate(all="ignore"):
        bw, bs, sc, bp = orc.viterbi_batch(X, offs, A, means, var)
    assert_close(two["scores"].cpu().numpy()[pick], sc, 1e-6, what="scores on both sides of the split")
    assert np.array_equal(two["best_word"].cpu().numpy()[pick], bw)
    got = two["path"].cpu().numpy().astype(np.int32).reshape(B, T)[pick].reshape(-1)
    assert np.mean(got == bp) > 0.995


@pytest.mark.parametrize("M,D", [(4, 39), (7, 36), (12, 38), (11, 12), (12, 15), (5, 13)])
def test_viterbi_equal_length_shape_sweep_vs_oracle(eng, M, D):
    """k_viterbi_v4 over the shapes it takes (4 <= M <= 12 models split 1-3 per recursion group, D in the 10- and 4-chunk
    classes) and the lengths around its special frames (t = 0, 1; exit closed below 8 frames; padding frames when T is not a
    multiple of four; one and 130 utterances = partial tiles): words, scores and paths against the CPU oracle."""
    from sapr_b200 import synth
    for T, B in ((2, 130), (3, 1), (5, 130), (8, 33), (9, 130), (13, 1), (16, 130), (30, 257)):
        Tg = max(T, 16)                                        # the generator needs a frame per state; short cases are truncated
        feats, labels, mu, sd = synth.make_corpus(B, M, 8, D, Tg, Tg, seed=7 * T + B + M)
        feats = [np.ascontiguousarray(f[:, :T]) for f in feats]
        A, means, var = synth.truth_models(mu, sd, 0.85)
        m = eng.WordModels(M, 8, D)
        m.set(means, var, A)
        batch = eng.PackedBatch.from_features(feats)
        X, offs = orc.pack(feats)
        with np.errstate(all="ignore"):
            bw, bs, sc, bp = orc.viterbi_batch(X, offs, A, means, var)
        out = m.viterbi(batch, None, eng.FP32, 0, want_scores=True, want_path=True)
        assert_close(out["scores"].cpu().numpy(), sc, 1e-6, what=f"scores T={T} B={B}")
        assert np.array_equal(out["best_word"].cpu().numpy(), bw), (T, B)            # near-ties are re-decoded in float64
        got = out["path"].cpu().numpy().astype(np.int32)
        if T >= 9:
            assert np.mean(got == bp) > 0.995, (T, B, np.mean(got == bp))
        else:
            # no model reaches the exit below 9 frames: every score is -inf, decoder.py:42-47 picks no word and returns no path
            assert np.all(out["best_word"].cpu().numpy() == -1) and np.all(np.isneginf(sc))
