"""Batched training of hmmlearn-style word models (DENSE topology, csrc/estep_dense.cu): prints one JSON line.

reference: 330 utterances, T ~ U{80..120}, D = 13, S = 10, M = 11, 15 iterations -- train_hmm("hmmlearn") per word (one
           GaussianHMM.fit per word, float64 E-steps) against train_hmm(..., batched=True) (one fp32 dense E-step per iteration for
           the whole vocabulary), wall time around synchronised work, per-word log-likelihood histories compared.  The batched run
           alternates the parent's fit_vocabulary (host M-step, parameters re-uploaded every iteration) with the device-resident
           one, and one profiled run of each splits an iteration into E-step kernels, M-step kernel and the remainder.
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


def parent_fit_vocabulary(models, features, precision="fp32"):
    """fit_vocabulary as it was before the device M-step, for the comparison: every iteration uploads every model's parameters
    (dev.set), downloads the statistics and runs one numpy _do_mstep per active model."""
    from sapr_b200._lib import EMIT_DIAG, FP32, FP64, TOPO_DENSE
    from sapr_b200.decoder import stack_hmmlearn_models
    from sapr_b200.engine import PackedBatch, WordModels
    from sapr_b200.hmmlearn_hmm import ConvergenceMonitor
    for mdl in models:
        mdl._check()
    means, _, _, _ = stack_hmmlearn_models(models)
    M, S, D = means.shape
    feats = [np.asarray(x, dtype=np.float32) for f in features for x in f]
    counts = np.array([len(f) for f in features])
    bounds = np.concatenate([[0], np.cumsum(counts)])
    batch = PackedBatch.from_features(feats, labels=np.repeat(np.arange(M), counts))
    dev = WordModels(M, S, D, EMIT_DIAG, TOPO_DENSE)
    prec = FP64 if precision == "fp64" else FP32
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


def reference_size(tmp, rounds=3):
    """train_hmm per word, then train_hmm(batched=True) with the parent's fit_vocabulary and with this one, alternated; the
    fit_vocabulary calls are timed on their own too, and one profiled run of each splits an iteration into E-step kernels
    (classes 9 + 10), M-step (class 11) and the remainder (launches, copies, host work)."""
    import torch
    from sapr_b200 import _lib, hmmlearn_hmm, synth, train
    from sapr_b200.train import train_hmm
    feats, labels, _, _ = synth.make_corpus(330, 11, 8, 13, 80, 120, seed=2024)
    fs = os.path.join(tmp, "feature_set")
    os.makedirs(fs)
    for u, (x, w) in enumerate(zip(feats, labels)):
        np.save(os.path.join(fs, f"sp{u // 11:02d}a_w{u:03d}_{WORDS[w]}.npy"), x)
    impls = {"parent": parent_fit_vocabulary, "this": hmmlearn_hmm.fit_vocabulary}
    fit_s = []

    def timed(fn):
        def run(*a, **k):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            r = fn(*a, **k)
            torch.cuda.synchronize()
            fit_s.append(time.perf_counter() - t0)
            return r
        return run

    def batched_run(impl, tag):
        train.fit_vocabulary = timed(impls[impl])
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        train_hmm("hmmlearn", 8, 13, n_iter=15, feature_set_path=fs, models_dir=os.path.join(tmp, tag), batched=True)
        torch.cuda.synchronize()
        return time.perf_counter() - t0, fit_s[-1], dict(train_hmm.histories)

    try:
        batched_run("this", "warmup")
        batched_run("parent", "warmup")
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        train_hmm("hmmlearn", 8, 13, n_iter=15, feature_set_path=fs, models_dir=os.path.join(tmp, "per_word"))
        torch.cuda.synchronize()
        per_word = (time.perf_counter() - t0, dict(train_hmm.histories))
        runs = {"parent": [], "this": []}
        for r in range(rounds):
            for impl in ("parent", "this"):
                runs[impl].append(batched_run(impl, f"{impl}{r}"))
        ctx = _lib.default_context()
        split = {}
        for impl in ("parent", "this"):
            ctx.profile(True)
            _, fit, hist = batched_run(impl, f"{impl}_prof")
            c9, c10, c11 = (ctx.profile_read(k)[0] for k in (9, 10, 11))
            ctx.profile(False)
            n = max(len(h) for h in hist.values())
            split[impl] = {"iterations": n, "fit_ms_per_iteration": round(fit * 1e3 / n, 3),
                           "estep_kernels_ms": round((c9 + c10) / n, 4), "mstep_kernel_ms": round(c11 / n, 4),
                           "remainder_ms": round((fit * 1e3 - c9 - c10 - c11) / n, 3)}
    finally:
        train.fit_vocabulary = hmmlearn_hmm.fit_vocabulary
    hp = per_word[1]
    hb, hq = runs["this"][-1][2], runs["parent"][-1][2]
    n = {w: min(len(hp[w]), len(hb[w])) for w in WORDS}          # a word may converge (tol) one iteration apart
    rel = max(float(np.max(np.abs(np.array(hb[w][:n[w]]) - np.array(hp[w][:n[w]])) / np.abs(np.array(hp[w][:n[w]]))))
              for w in WORDS)
    med = {k: float(np.median([x[0] for x in v])) for k, v in runs.items()}
    return {"utts": 330, "iters": 15, "per_word_s": round(per_word[0], 4), "batched_s": round(med["this"], 4),
            "parent_batched_s": round(med["parent"], 4), "batched_s_runs": [round(x[0], 4) for x in runs["this"]],
            "parent_batched_s_runs": [round(x[0], 4) for x in runs["parent"]],
            "fit_s": round(float(np.median([x[1] for x in runs["this"]])), 4),
            "parent_fit_s": round(float(np.median([x[1] for x in runs["parent"]])), 4),
            "histories_equal_parent": hb == hq, "iteration_split": split,
            "speedup": round(per_word[0] / med["this"], 2), "history_max_rel_diff": rel,
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
