"""Batched scoring with hmmlearn-style word models (DENSE topology, csrc/score_dense.cu): prints one JSON line.

reference: 330 utterances, T ~ U{80..120}, D = 13, S = 10, M = 11 -- the per-sequence loop of GaussianHMM.score (one call per
           utterance x model, the arg-max taken in Python) against one Decoder.score_batch call, wall time around synchronised
           work, recognised words compared.
throughput: 100 000 utterances x 200 frames x 11 models, S = 10, D in {13, 39}, left-to-right (the reference's initial zero
           pattern, 2S - 2 arcs) and fully dense (Dirichlet rows) transitions.  Kernel times come from the profile classes
           (12 = dense forward, 1 = its arg-max, 13 = float64 re-scoring of near-ties; 7 = the scores-only dense Viterbi at the same
           shape, in the same run), averaged over the timed calls.  The emission's SIMT bound is M*S*2D FMAs per utterance-frame at
           one FMA per lane and cycle (148 SMs x 128 lanes at the maximum SM clock), as in tools/dense_bench.py.  The float64 call
           is SAPR_FP64 (sapr_hl_score per model); the fp32 scores and words are compared with it over the whole batch.

usage: python tools/dense_score_bench.py [--utts 100000] [--frames 200] [--calls 5] [--out FILE]
"""
import argparse
import json
import os
import pickle
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tools.dense_bench import LANES, SMS, gpu_info, make_models  # noqa: E402


def reference_size(M=11, S=10, D=13, B=330):
    from sapr_b200.decoder import Decoder
    from sapr_b200.hmmlearn_hmm import GaussianHMM
    from sapr_b200.synth import VOCAB
    import torch
    means, var, tm, sp = make_models(M, S, D, False, 11)
    rng = np.random.default_rng(12)
    feats = []
    for _ in range(B):
        w, T = rng.integers(0, M), rng.integers(80, 121)
        st = np.sort(rng.integers(0, S, T))
        feats.append((means[w, st] + np.sqrt(var[w, st]) * rng.standard_normal((T, D))).T.astype(np.float32))
    with tempfile.TemporaryDirectory() as tmp:
        os.makedirs(os.path.join(tmp, "hmmlearn"))
        for i in range(M):
            h = GaussianHMM(n_components=S, covariance_type="diag", init_params="")
            h.means_, h.covars_, h.transmat_, h.startprob_ = means[i], var[i], tm[i], sp[i]
            with open(os.path.join(tmp, "hmmlearn", f"{VOCAB[i]}_hmmlearn_15.pkl"), "wb") as f:
                pickle.dump(h, f)
        dec = Decoder(models_dir=tmp, implementation="hmmlearn", n_iter=15, vocab_order=VOCAB)
        models = [dec.models[w] for w in dec.vocab]
        for f in feats[:3]:
            [h.score(f.T) for h in models]            # warm-up: module load, per-model uploads
        dec.score_batch(feats)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        loop_words = []
        for f in feats:
            lps = [h.score(f.T) for h in models]
            loop_words.append(dec.vocab[int(np.argmax(lps))])
        torch.cuda.synchronize()
        t_loop = time.perf_counter() - t0
        t_b = []
        for _ in range(5):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            words, _, _ = dec.score_batch(feats)
            torch.cuda.synchronize()
            t_b.append(time.perf_counter() - t0)
    return {"utterances": B, "loop_s": round(t_loop, 4), "loop_calls": B * M, "batch_s_median": round(float(np.median(t_b)), 5),
            "speedup": round(t_loop / float(np.median(t_b)), 1), "words_identical": words == loop_words}


def throughput(B, T, D, dense, calls, clock_mhz, M=11, S=10):
    import torch
    from sapr_b200 import engine
    means, var, tm, sp = make_models(M, S, D, dense, 21 + D)
    m = engine.WordModels(M, S, D, engine.EMIT_DIAG, engine.TOPO_DENSE)
    m.set(means, var, tm, sp)
    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev); g.manual_seed(D + 2 * dense)
    Dp = (D + 3) // 4 * 4
    X = torch.zeros(B * T, Dp, dtype=torch.float32, device=dev)
    mt = torch.tensor(means.reshape(M * S, D), dtype=torch.float32, device=dev)
    sd = torch.tensor(np.sqrt(var).reshape(M * S, D), dtype=torch.float32, device=dev)
    w = torch.randint(0, M, (B,), device=dev, generator=g).repeat_interleave(T)
    for r0 in range(0, B * T, 1 << 22):       # generated in slices: bounded temporaries
        r1 = min(B * T, r0 + (1 << 22))
        st = w[r0:r1] * S + torch.randint(0, S, (r1 - r0,), device=dev, generator=g)
        X[r0:r1, :D] = mt[st] + sd[st] * torch.randn(r1 - r0, D, device=dev, generator=g)
    offsets = torch.arange(0, B + 1, device=dev, dtype=torch.int64) * T
    batch = engine.PackedBatch(X, offsets, D, np.arange(0, B + 1, dtype=np.int64) * T)

    out32 = m.score_words(batch, engine.FP32)     # warm-up, and the fp32 result compared below
    flagged = m.ctx.viterbi_flagged()
    m.ctx.profile(True)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(calls):
        m.score_words(batch, engine.FP32)
    torch.cuda.synchronize()
    wall = (time.perf_counter() - t0) / calls
    k12, n12 = m.ctx.profile_read(12); k1, _ = m.ctx.profile_read(1); k13, _ = m.ctx.profile_read(13)
    m.ctx.profile(False)

    m.viterbi(batch, None, engine.FP32, 0, want_path=False)
    m.ctx.profile(True)
    for _ in range(calls):
        m.viterbi(batch, None, engine.FP32, 0, want_path=False)
    k7, _ = m.ctx.profile_read(7)
    m.ctx.profile(False)

    out64 = m.score_words(batch, engine.FP64)     # warm-up (workspace growth), and the float64 reference
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    m.score_words(batch, engine.FP64)
    torch.cuda.synchronize()
    t64 = time.perf_counter() - t0

    s32, s64 = out32["scores"].cpu().numpy(), out64["scores"].cpu().numpy()
    fin = np.isfinite(s64)
    rel = float(np.max(np.abs(s32[fin] - s64[fin]) / np.maximum(1.0, np.abs(s64[fin])))) if fin.any() else 0.0
    agree = float(np.mean(out32["best_word"].cpu().numpy() == out64["best_word"].cpu().numpy()))
    fwd_ms = k12 / calls
    fma = B * T * M * S * 2 * D
    simt_ms = fma / (SMS * LANES * clock_mhz * 1e6) * 1e3 if clock_mhz else None
    return {"D": D, "transitions": "dense" if dense else "left_to_right", "finite_arcs_per_model": int(np.sum(tm > 0)) // M,
            "utterances": B, "frames": T, "models": M, "states": S,
            "forward_ms": round(fwd_ms, 4), "forward_launches_per_call": n12 // calls, "argmax_ms": round(k1 / calls, 4),
            "rescore_ms": round(k13 / calls, 4), "flagged": flagged, "call_wall_ms": round(wall * 1e3, 3),
            "viterbi_scores_only_ms": round(k7 / calls, 4), "forward_over_viterbi": round(fwd_ms / (k7 / calls), 3),
            "updates_per_s": float(f"{B * T * S * M / (fwd_ms * 1e-3):.4g}"),
            "emission_simt_bound_ms": round(simt_ms, 4) if simt_ms else None,
            "fraction_of_simt_bound": round(simt_ms / fwd_ms, 4) if simt_ms else None,
            "fp64_call_ms": round(t64 * 1e3, 2), "fp32_vs_fp64_max_rel": float(f"{rel:.3g}"), "word_agreement": agree}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--utts", type=int, default=100_000)
    ap.add_argument("--frames", type=int, default=200)
    ap.add_argument("--calls", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("dense_score_bench needs a CUDA device")
    torch.cuda.set_device(0)
    info = gpu_info()
    line = {"bench": "dense_score", **info, "reference_size": reference_size(), "throughput": []}
    for D in (13, 39):
        for dense in (False, True):
            line["throughput"].append(throughput(a.utts, a.frames, D, dense, a.calls, info.get("sm_max_mhz")))
            torch.cuda.empty_cache()
    s = json.dumps(line)
    print(s)
    if a.out:
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
