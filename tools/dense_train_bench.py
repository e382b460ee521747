"""Batched training of hmmlearn-style word models (DENSE topology, csrc/estep_dense.cu): prints one JSON line.

reference: 330 utterances, T ~ U{80..120}, D = 13, S = 10, M = 11, 15 iterations -- train_hmm("hmmlearn") per word (one
           GaussianHMM.fit per word, float64 E-steps) against train_hmm(..., batched=True) (one fp32 dense E-step per iteration for
           the whole vocabulary), wall time around synchronised work, per-word log-likelihood histories compared.
throughput: 100 000 utterances x 200 frames, 11 models, S = 10, D in {13, 39}, left-to-right (2S - 2 arcs) and Dirichlet-dense
           transitions, utterances grouped by word.  The fp32 E-step's kernel time comes from the profile classes (9 = forward /
           backward, 10 = feature statistics), averaged over the timed calls; the float64 path (SAPR_FP64 = sapr_hl_estep per
           model) is timed on the same batch, and the two are compared.  The SIMT FMA bound counts 2*S*D emission FMAs twice
           (forward, and the backward's recomputation) + 2*S*D statistics FMAs + 3 per finite arc (forward, backward, xi) per
           utterance-frame at one FMA per lane and cycle (148 SMs x 128 lanes at the maximum SM clock).

usage: python tools/dense_train_bench.py [--utts 100000] [--frames 200] [--calls 5] [--out FILE]
"""
import argparse
import json
import os
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tools.dense_bench import LANES, SMS, gpu_info, make_models   # noqa: E402

WORDS = ["heed", "hid", "head", "had", "hard", "hud", "hod", "hoard", "hood", "whod", "heard"]


def reference_size(tmp):
    import torch
    from sapr_b200 import synth
    from sapr_b200.train import train_hmm
    feats, labels, _, _ = synth.make_corpus(330, 11, 8, 13, 80, 120, seed=2024)
    fs = os.path.join(tmp, "feature_set")
    os.makedirs(fs)
    for u, (x, w) in enumerate(zip(feats, labels)):
        np.save(os.path.join(fs, f"sp{u // 11:02d}a_w{u:03d}_{WORDS[w]}.npy"), x)
    out = {}
    for name, batched in (("warmup", True), ("per_word", False), ("batched", True)):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        train_hmm("hmmlearn", 8, 13, n_iter=15, feature_set_path=fs, models_dir=os.path.join(tmp, name), batched=batched)
        torch.cuda.synchronize()
        out[name] = (time.perf_counter() - t0, dict(train_hmm.histories))
    hp, hb = out["per_word"][1], out["batched"][1]
    n = {w: min(len(hp[w]), len(hb[w])) for w in WORDS}          # a word may converge (tol) one iteration apart
    rel = max(float(np.max(np.abs(np.array(hb[w][:n[w]]) - np.array(hp[w][:n[w]])) / np.abs(np.array(hp[w][:n[w]]))))
              for w in WORDS)
    return {"utts": 330, "iters": 15, "per_word_s": round(out["per_word"][0], 4), "batched_s": round(out["batched"][0], 4),
            "speedup": round(out["per_word"][0] / out["batched"][0], 2), "history_max_rel_diff": rel,
            "iterations_per_word": [len(hp[w]) for w in WORDS], "iterations_batched": [len(hb[w]) for w in WORDS]}


def device_batch(eng, means, var, tm, B, T, seed):
    """B equal-length utterances grouped by word, drawn on the device (state = position along the utterance)."""
    import torch
    M, S, D = means.shape
    g = torch.Generator(device="cuda").manual_seed(seed)
    counts = np.bincount(np.random.default_rng(seed).integers(0, M, B), minlength=M)
    labels = torch.as_tensor(np.repeat(np.arange(M), counts).astype(np.int32), device="cuda")
    mu = torch.as_tensor(means, dtype=torch.float32, device="cuda")
    sd = torch.as_tensor(np.sqrt(var), dtype=torch.float32, device="cuda")
    st = (torch.arange(T, device="cuda") * S // T)
    dp = (D + 3) // 4 * 4
    X = torch.zeros((B * T, dp), dtype=torch.float32, device="cuda")
    step = 8192
    for u0 in range(0, B, step):
        lab = labels[u0:u0 + step].long()
        n = lab.numel()
        x = mu[lab[:, None], st[None, :]] + sd[lab[:, None], st[None, :]] * torch.randn((n, T, D), generator=g, device="cuda")
        X[u0 * T:(u0 + n) * T, :D] = x.reshape(n * T, D)
    offs = np.arange(B + 1, dtype=np.int64) * T
    return eng.PackedBatch(X, torch.as_tensor(offs, device="cuda"), D, offs), labels


def throughput(eng, B, T, D, dense, calls, clock_mhz):
    import torch
    M, S = 11, 10
    means, var, tm, sp = make_models(M, S, D, dense, seed=D + dense)
    m = eng.WordModels(M, S, D, eng.EMIT_DIAG, eng.TOPO_DENSE)
    m.set(means, var, tm, sp)
    batch, labels = device_batch(eng, means, var, tm, B, T, seed=5 + D)
    m.estep(batch, labels, None, eng.FP32)                                    # warm-up
    a = m.estep(batch, labels, None, eng.FP32)
    b = m.estep(batch, labels, None, eng.FP32)
    deterministic = bool(torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]))
    m.ctx.profile(True)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(calls):
        st32, ll32, _ = m.estep(batch, labels, None, eng.FP32)
    torch.cuda.synchronize()
    wall32 = (time.perf_counter() - t0) / calls
    fb_ms, fb_n = m.ctx.profile_read(9)
    ob_ms, ob_n = m.ctx.profile_read(10)
    m.ctx.profile(False)
    m.estep(batch, labels, None, eng.FP64)                                    # warm-up
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    st64, ll64, _ = m.estep(batch, labels, None, eng.FP64)
    torch.cuda.synchronize()
    wall64 = time.perf_counter() - t0
    u32, u64 = m.unpack_stats(st32), m.unpack_stats(st64)
    l32, l64 = ll32.cpu().numpy(), ll64.cpu().numpy()
    frames = u64["post"].sum(axis=1)
    k_ms = (fb_ms + ob_ms) / calls
    arcs = int(np.count_nonzero(tm)) / M
    fma = 4 * S * D + 2 * S * D + 3 * arcs
    bound_ms = B * T * fma / (SMS * LANES * clock_mhz * 1e6) * 1e3 if clock_mhz else None
    return {"D": D, "transitions": "dense" if dense else "left-to-right", "arcs_per_model": arcs,
            "fp32_fb_ms": round(fb_ms / calls, 4), "fp32_stats_ms": round(ob_ms / calls, 4), "fp32_kernel_ms": round(k_ms, 4),
            "fp32_call_wall_ms": round(wall32 * 1e3, 3), "fp64_call_wall_ms": round(wall64 * 1e3, 3),
            "fp64_over_fp32_kernels": round(wall64 * 1e3 / k_ms, 1),
            "updates_per_s": B * T * S / (k_ms * 1e-3), "simt_fma_bound_ms": bound_ms,
            "frac_of_simt_fma_bound": (bound_ms / k_ms) if bound_ms else None, "deterministic": deterministic,
            "loglik_max_rel": float(np.max(np.abs(l32 - l64) / np.abs(l64))),
            "post_max_abs_over_frames": float(np.max(np.abs(u32["post"] - u64["post"]).max(axis=1) / frames)),
            "trans_max_abs_over_frames": float(np.max(np.abs(u32["trans"] - u64["trans"]).reshape(M, -1).max(axis=1) / frames)),
            "mean_max_diff_over_sigma": float(np.max(np.abs(u32["obs"] / u32["post"][..., None] - u64["obs"] / u64["post"][..., None])
                                                     / np.sqrt(var))),
            "profile_launches": [fb_n, ob_n]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--utts", type=int, default=100000)
    ap.add_argument("--frames", type=int, default=200)
    ap.add_argument("--calls", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("dense_train_bench needs a CUDA device")
    from sapr_b200 import engine as eng
    info = gpu_info()
    res = {"bench": "dense_train", **info}
    with tempfile.TemporaryDirectory() as tmp:
        res["reference"] = reference_size(tmp)
    res["throughput"] = [throughput(eng, args.utts, args.frames, D, dense, args.calls, info.get("sm_max_mhz"))
                         for D in (13, 39) for dense in (False, True)]
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
