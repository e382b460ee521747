"""The float64 hmmlearn kernels (sapr_hl_score / sapr_hl_decode / sapr_hl_estep, csrc/hmmlearn.cu) against the CPU oracle's
restatement (orc.emission_diag + orc.hl_forward / hl_viterbi / hl_estep) over the range include/sapr_b200.h promises: 1 to 1024
states, both mappings (thread per utterance for S <= 32 and B >= 16 * SMs, one CTA per utterance otherwise), zeros in
startprob_ / transmat_, an unreachable state, empty and one-frame utterances, frame totals that cut the 512-frame chunks of the
observation sums inside utterances, exact Viterbi ties, and one E-step over more than 65 535 such chunks.

Tolerances, float64 against float64 with the same formulas (the device and the C library round exp / log differently in the last
bit): log-likelihoods and scores 1e-12 * max(1, |ref|), statistics 1e-10 * max(1, |ref|), paths exact."""
import numpy as np
import pytest

from conftest import assert_close
from oracle import oracle as orc

pytestmark = pytest.mark.gpu

LL_TOL, STAT_TOL = 1e-12, 1e-10
STATS = ("start", "trans", "post", "obs", "obs2")


@pytest.fixture(scope="module")
def cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


@pytest.fixture(scope="module")
def thread_batch(cuda):
    """the smallest batch that runs thread per utterance (hl_thread_per_utt in csrc/hmmlearn.cu), plus 7"""
    return 16 * cuda.cuda.get_device_properties(cuda.cuda.current_device()).multi_processor_count + 7


def _model(S, D, seed, left_to_right=False):
    rng = np.random.default_rng(seed)
    means = rng.normal(0.0, 3.0, (S, D))
    var = rng.uniform(0.5, 1.5, (S, D)) ** 2
    tm = rng.dirichlet(np.ones(S), size=S)
    sp = rng.dirichlet(np.ones(S))
    if left_to_right:                                  # zeros in startprob_ and transmat_
        tm = np.zeros((S, S))
        for i in range(S - 1):
            a = rng.uniform(0.6, 0.95)
            tm[i, i], tm[i, i + 1] = a, 1.0 - a
        tm[S - 1, S - 1] = 1.0
        sp = np.zeros(S); sp[0] = 1.0
    return means, var, tm, sp


def _frames(rng, means, var, lengths, sorted_states=False):
    """float32 frames (sum T, D) drawn around the model's states (in state order per utterance for left-to-right models)"""
    S, D = means.shape
    parts = []
    for T in lengths:
        st = rng.integers(0, S, T)
        if sorted_states:
            st = np.sort(st)
        parts.append(means[st] + np.sqrt(var[st]) * rng.standard_normal((T, D)))
    return np.concatenate(parts, axis=0).astype(np.float32)


class _Dev:
    """one DENSE + DIAG model on the device; the C entry points called as GaussianHMM calls them, with per-utterance outputs"""

    def __init__(self, means, var, tm, sp):
        from sapr_b200 import engine
        S, D = means.shape
        self.S, self.D = S, D
        self.m = engine.WordModels(1, S, D, engine.EMIT_DIAG, engine.TOPO_DENSE)
        self.m.set(means, var, tm, sp)

    def _batch(self, X, lengths):
        from sapr_b200.engine import PackedBatch
        return PackedBatch.from_frames(X, lengths)

    def score(self, X, lengths):
        import torch
        from sapr_b200._lib import ptr
        b = self._batch(X, lengths)
        lp = torch.full((b.B,), np.nan, dtype=torch.float64, device=b.X.device)
        self.m.ctx.check(self.m.lib.sapr_hl_score(self.m.ctx.h, self.m.h, 0, ptr(b.X), b.ldx, ptr(b.offsets), b.B,
                                                  b.total_frames, ptr(lp)))
        return lp.cpu().numpy()

    def decode(self, X, lengths):
        import torch
        from sapr_b200._lib import ptr
        b = self._batch(X, lengths)
        lp = torch.full((b.B,), np.nan, dtype=torch.float64, device=b.X.device)
        path = torch.full((b.total_frames,), -1, dtype=torch.int32, device=b.X.device)
        self.m.ctx.check(self.m.lib.sapr_hl_decode(self.m.ctx.h, self.m.h, 0, ptr(b.X), b.ldx, ptr(b.offsets), b.B,
                                                   b.total_frames, ptr(lp), ptr(path)))
        return lp.cpu().numpy(), path.cpu().numpy()

    def estep(self, X, lengths):
        import torch
        from sapr_b200._lib import ptr
        b = self._batch(X, lengths)
        n = int(self.m.lib.sapr_hl_stats_len(self.S, self.D))
        stats = torch.full((n,), np.nan, dtype=torch.float64, device=b.X.device)
        lp = torch.full((b.B,), np.nan, dtype=torch.float64, device=b.X.device)
        self.m.ctx.check(self.m.lib.sapr_hl_estep(self.m.ctx.h, self.m.h, 0, ptr(b.X), b.ldx, ptr(b.offsets), b.B,
                                                  b.total_frames, ptr(stats), ptr(lp)))
        return self.m.unpack_stats(stats.cpu().numpy()[None]), lp.cpu().numpy()

    def estep_words(self, X, lengths):
        """WordModels.estep(..., FP64): the route the dense-topology tests take to these kernels"""
        import torch
        from sapr_b200 import engine
        b = self._batch(X, lengths)
        lab = torch.zeros(b.B, dtype=torch.int32, device=b.X.device)
        stats, ll, _ = self.m.estep(b, lab, None, engine.FP64)
        return self.m.unpack_stats(stats), ll.cpu().numpy()


def _oracle(X, lengths, means, var, tm, sp):
    """per-utterance forward score, Viterbi log-probability and path, and the E-step; empty utterances get a score of 0 and no
    path, and stay out of the E-step (orc_hl_forward writes frame 0 even when T = 0)"""
    X64 = X.astype(np.float64)
    offs = np.concatenate([[0], np.cumsum(lengths)]).astype(np.int64)
    score, vlp, paths = np.zeros(len(lengths)), np.zeros(len(lengths)), []
    for u, (a, b) in enumerate(zip(offs[:-1], offs[1:])):
        if b == a:
            continue
        lf = orc.emission_diag(X64[a:b].T, means, var, all_emit=True)
        score[u] = orc.hl_forward(lf, sp, tm)[0]
        vlp[u], p = orc.hl_viterbi(lf, sp, tm)
        paths.append(p)
    keep = np.asarray(lengths) > 0
    st = orc.hl_estep(X64, np.concatenate([[0], np.cumsum(np.asarray(lengths)[keep])]).astype(np.int64), sp, tm, means, var)
    ll = np.zeros(len(lengths)); ll[keep] = st["loglik"]
    st["loglik"] = ll
    return score, vlp, np.concatenate(paths) if paths else np.zeros(0, np.int32), st


def _check_stats(got, ll, ref, what):
    for k in STATS:
        assert_close(np.asarray(got[k]).reshape(ref[k].shape), ref[k], STAT_TOL, what=f"{what} {k}")
    assert_close(ll, ref["loglik"], LL_TOL, what=f"{what} loglik")


def _check_all(dev, X, lengths, ref, what):
    """score, decode and E-step against the oracle's results ``ref``; returns the device's (score, decode logprob, path)"""
    score, vlp, path, st = ref
    sc = dev.score(X, lengths)
    assert_close(sc, score, LL_TOL, what=f"{what} score")
    lp, p = dev.decode(X, lengths)
    assert_close(lp, vlp, LL_TOL, what=f"{what} decode logprob")
    assert np.array_equal(p, path), f"{what}: Viterbi path differs at {np.flatnonzero(p != path)[:10]}"
    got, ll = dev.estep(X, lengths)
    _check_stats({k: v[0] for k, v in got.items()}, ll, st, what)
    return sc, lp, p


STATE_RANGE = [(1, 1), (2, 13), (31, 39), (32, 1), (33, 13), (64, 39), (65, 1), (255, 13), (257, 39), (800, 1), (801, 13),
               (1024, 39)]


@pytest.mark.parametrize("S,D", STATE_RANGE)
def test_state_range_vs_oracle(cuda, S, D):
    """Warp-boundary state counts, one and two states, and the E-step above 800 states (whose CTA kernel must fit 1024 threads
    in the register file): per-utterance scores, Viterbi log-probabilities and paths, the five statistics and the per-utterance
    log-likelihoods, directly through the C entry points and through WordModels.estep(FP64) (bit for bit the same call)."""
    means, var, tm, sp = _model(S, D, seed=7000 + S)
    rng = np.random.default_rng(S * 10 + D)
    lengths = [1, 2, 30, 17] if S >= 255 else [1, 2, 57, 33, 8, 64, 20]
    X = _frames(rng, means, var, lengths)
    dev = _Dev(means, var, tm, sp)
    ref = _oracle(X, lengths, means, var, tm, sp)
    _check_all(dev, X, lengths, ref, f"S={S} D={D}")
    st, ll = dev.estep(X, lengths)
    sw, llw = dev.estep_words(X, lengths)
    for k in STATS:
        assert np.array_equal(sw[k], st[k]), f"WordModels.estep(FP64) {k} differs from sapr_hl_estep"
    assert np.array_equal(llw, ll)


def _kernels(torch, fn):
    """names of the CUDA kernels fn() launches"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {e.key for e in prof.key_averages()}


def _mapping_kernels(torch, dev, X, lengths):
    names = _kernels(torch, lambda: dev.score(X, lengths))
    return {"thread" if any("k_hl_forward" in n and "cta" not in n for n in names) else None,
            "cta" if any("k_hl_forward_cta" in n for n in names) else None} - {None}


def _chunks(lengths, n):
    """split the utterances into n consecutive chunks: (frame range, lengths) per chunk"""
    offs = np.concatenate([[0], np.cumsum(lengths)])
    cut = np.linspace(0, len(lengths), n + 1).astype(int)
    return [((offs[a], offs[b]), lengths[a:b]) for a, b in zip(cut[:-1], cut[1:])]


@pytest.mark.parametrize("S,D", [(2, 13), (32, 39)])
def test_both_mappings_vs_oracle(cuda, thread_batch, S, D):
    """16 * SMs + 7 utterances run thread per utterance; the same utterances in three smaller calls run one CTA per utterance.
    Score and decode are the same arithmetic in both (the header of csrc/hmmlearn.cu): equal bit for bit.  The E-step sums
    the posteriors in different orders, so each mapping is held to the oracle."""
    means, var, tm, sp = _model(S, D, seed=8000 + S)
    rng = np.random.default_rng(S + 1)
    lengths = [int(t) for t in rng.integers(1, 20, thread_batch)]
    lengths[:3] = [1, 2, 0]
    X = _frames(rng, means, var, lengths)
    dev = _Dev(means, var, tm, sp)
    parts = _chunks(lengths, 3)
    assert all(len(lc) < thread_batch - 7 for _, lc in parts)
    assert _mapping_kernels(cuda, dev, X, lengths) == {"thread"}
    assert _mapping_kernels(cuda, dev, X[:parts[0][0][1]], parts[0][1]) == {"cta"}
    refs = [_oracle(X[a:b], lc, means, var, tm, sp) for (a, b), lc in parts]
    whole = (np.concatenate([r[0] for r in refs]), np.concatenate([r[1] for r in refs]), np.concatenate([r[2] for r in refs]),
             {k: sum(r[3][k] for r in refs) for k in STATS})
    whole[3]["loglik"] = np.concatenate([r[3]["loglik"] for r in refs])
    score_t, lp_t, path_t = _check_all(dev, X, lengths, whole, f"thread S={S}")
    score_c, lp_c, path_c = [], [], []
    for ((a, b), lc), ref in zip(parts, refs):
        sc, lp, p = _check_all(dev, X[a:b], lc, ref, f"cta S={S} frames {a}:{b}")
        score_c.append(sc); lp_c.append(lp); path_c.append(p)
    assert np.concatenate(score_c).tobytes() == score_t.tobytes(), "score: thread and CTA mappings differ"
    assert np.concatenate(lp_c).tobytes() == lp_t.tobytes(), "decode logprob: thread and CTA mappings differ"
    assert np.array_equal(np.concatenate(path_c), path_t), "decode path: thread and CTA mappings differ"


@pytest.mark.parametrize("S,D,mapping,edge", [(6, 13, "thread", 1), (6, 13, "cta", -1), (40, 1, "cta", 1)])
def test_structure_vs_oracle(cuda, thread_batch, S, D, mapping, edge):
    """A left-to-right model (zeros in startprob_ and transmat_) with one extra state that no transition enters (a zero column:
    posterior exactly 0); one- and two-frame utterances; an empty utterance between two others, given as a repeated offset
    (log-likelihood 0, no statistics, its neighbours' results the same bits as without it); an utterance of more than 512
    frames, with the batch total 512 k + edge so that the chunks of the observation sums start and end inside utterances."""
    means, var, tm, sp = _model(S, D, seed=9000 + S, left_to_right=True)
    tm = np.pad(tm, ((0, 1), (0, 1)))                   # state S: no way in, leaves to state 0
    tm[S, 0] = 1.0
    sp = np.pad(sp, (0, 1))
    rng = np.random.default_rng(S + 2)
    means = np.vstack([means, rng.normal(0.0, 3.0, (1, D))])
    var = np.vstack([var, rng.uniform(0.5, 1.5, (1, D)) ** 2])
    lengths = [1, 2, 37, 0, 700, 5]
    if mapping == "thread":
        lengths += [int(t) for t in rng.integers(3, 12, thread_batch - len(lengths))]
    lengths.append(512 * (sum(lengths) // 512 + 2) + edge - sum(lengths))
    assert sum(lengths) % 512 == edge % 512
    X = _frames(rng, means[:S], var[:S], lengths, sorted_states=True)
    dev = _Dev(means, var, tm, sp)
    assert _mapping_kernels(cuda, dev, X, lengths) == {mapping}
    ref = _oracle(X, lengths, means, var, tm, sp)
    sc, lp, path = _check_all(dev, X, lengths, ref, f"S={S + 1} {mapping}")
    got, ll = dev.estep(X, lengths)
    assert ll[3] == 0.0 and sc[3] == 0.0 and lp[3] == 0.0
    assert got["post"][0, S] == 0.0 and got["start"][0, S] == 0.0
    assert not got["trans"][0, :, S].any() and not got["obs"][0, S].any() and not got["obs2"][0, S].any()
    assert (path != S).all()
    # the same batch without the empty utterance: every other utterance's results keep their bits
    rest = lengths[:3] + lengths[4:]
    keep = np.r_[0:3, 4:len(lengths)]
    assert dev.score(X, rest).tobytes() == sc[keep].tobytes()
    lp_r, path_r = dev.decode(X, rest)
    assert lp_r.tobytes() == lp[keep].tobytes() and np.array_equal(path_r, path)
    assert dev.estep(X, rest)[1].tobytes() == ll[keep].tobytes()


def _tied_model(S, D, seed):
    """S states of which the last ndup duplicate states 0 .. ndup-1: identical rows, columns (halved: exact in binary), start
    probabilities, means and variances, so every Viterbi comparison between a state and its duplicate is an exact tie"""
    K = (S + 1) // 2
    ndup = S - K
    means, var, P, p0 = _model(K, D, seed)
    base = np.r_[np.arange(K), np.arange(ndup)]        # state -> the base state it copies
    mult = np.where(np.arange(K) < ndup, 2.0, 1.0)
    tm = P[np.ix_(base, base)] / mult[base][None, :]
    sp = p0[base] / mult[base]
    return means[base], var[base], tm, sp, K


@pytest.mark.parametrize("S,D", [(4, 13), (257, 13)])
def test_viterbi_ties_vs_oracle(cuda, thread_batch, S, D):
    """Exact ties: the path must be the oracle's, where the lowest index wins every tie, so no duplicate state ever appears.
    S = 4 in both mappings (a thread-per-utterance batch and the same utterances in CTA-per-utterance calls), S = 257 in the
    CTA mapping (the only one above 32 states)."""
    means, var, tm, sp, K = _tied_model(S, D, seed=9500 + S)
    for a in (tm, tm.T, sp, means, var):
        assert a[K:].tobytes() == a[:S - K].tobytes()
    rng = np.random.default_rng(S + 3)
    lengths = [int(t) for t in rng.integers(1, 25, thread_batch if S <= 32 else 6)]
    X = _frames(rng, means, var, lengths)
    dev = _Dev(means, var, tm, sp)
    offs = np.concatenate([[0], np.cumsum(lengths)])
    vlp, paths = [], []
    for a, b in zip(offs[:-1], offs[1:]):
        lp, p = orc.hl_viterbi(orc.emission_diag(X[a:b].T.astype(np.float64), means, var, all_emit=True), sp, tm)
        vlp.append(lp); paths.append(p)
    vlp, path = np.array(vlp), np.concatenate(paths)
    assert (path < K).all()
    runs = [(X, lengths)]
    if S <= 32:
        assert _mapping_kernels(cuda, dev, X, lengths) == {"thread"}
        runs += [(X[a:b], lc) for (a, b), lc in _chunks(lengths, 3)]
    got_lp, got_path = [], []
    for Xr, lr in runs:
        lp, p = dev.decode(Xr, lr)
        got_lp.append(lp); got_path.append(p)
    if S <= 32:
        assert _mapping_kernels(cuda, dev, runs[1][0], runs[1][1]) == {"cta"}
        got_lp.append(np.concatenate(got_lp[1:])); got_path.append(np.concatenate(got_path[1:]))
        got_lp, got_path = [got_lp[0], got_lp[-1]], [got_path[0], got_path[-1]]
    for lp, p in zip(got_lp, got_path):
        assert_close(lp, vlp, LL_TOL, what="tied decode logprob")
        assert np.array_equal(p, path), f"tied path differs at {np.flatnonzero(p != path)[:10]}"


def test_estep_over_65536_chunks_vs_oracle(cuda):
    """33 554 432 frames in one E-step: 65 536 chunks of 512 frames, one more than a grid's y dimension holds.  S = 2, D = 1,
    256-frame utterances (thread per utterance).  Tolerance 1e-9 relative: the oracle sums 131 072 log-likelihoods and
    3.4e7 frames of statistics one after the other, the device in per-utterance slots and 512-frame chunks."""
    S, D, T, B = 2, 1, 256, 131072
    means, var, tm, sp = _model(S, D, seed=9900)
    rng = np.random.default_rng(9901)
    st = rng.integers(0, S, B * T)
    X = (means[st] + np.sqrt(var[st]) * rng.standard_normal((B * T, D))).astype(np.float32)
    del st
    lengths = [T] * B
    dev = _Dev(means, var, tm, sp)
    got, ll = dev.estep(X, lengths)
    ref = orc.hl_estep(X.astype(np.float64), np.arange(B + 1, dtype=np.int64) * T, sp, tm, means, var)
    for k in STATS:
        assert_close(got[k][0], ref[k], 1e-9, what=f"65536 chunks {k}")
    assert_close(ll.sum(), ref["logprob"], 1e-9, what="65536 chunks log-likelihood")
    assert_close(ll, ref["loglik"], LL_TOL, what="65536 chunks per-utterance log-likelihood")
