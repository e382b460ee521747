"""Sharded batched training of hmmlearn-style word models (fit_vocabulary with dist): a check and one iteration's timing.

Run under torchrun, one process per GPU (NCCL through the library's own communicator):
    torchrun --nproc_per_node 8 tools/dense_train_dist.py --out FILE

check:  11 models, S = 10, D = 13, 880 utterances.  Every rank fits the whole vocabulary sharded (dist) and unsharded on its own,
        float64; the sharded fit must reproduce the unsharded one (histories within 1e-12 relative, parameters within 1e-10,
        equal iteration counts) and every rank must hold the same parameters.  A non-zero rank with an empty shard is not
        exercised here (tests/test_gpu_dense_mstep.py does that).
timing: the calls fit_vocabulary makes per iteration -- fp32 dense E-step on this rank's shard, ONE all-reduce of [stats |
        per-model log-likelihood sums], sapr_hl_mstep for every model, the copy of the M sums to the host -- on device-drawn
        utterances of 200 frames grouped by word, 11 left-to-right models, S = 10, D in {13, 39}: weak scaling (100 000
        utterances per GPU) and strong scaling (100 000 in total).  E-step kernel times are profile classes 9 and 10, the M-step
        class 11 (rank 0's, averaged over the timed iterations); wall time per iteration is the slowest rank's.
"""
import argparse
import copy
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tools.dense_bench import gpu_info, make_models          # noqa: E402
from tools.dense_train_bench import device_batch              # noqa: E402


def _init(means, var, tm, sp, n_iter, seed):
    from sapr_b200.hmmlearn_hmm import GaussianHMM
    rng = np.random.default_rng(seed)
    hs = []
    for mi in range(means.shape[0]):
        h = GaussianHMM(n_components=means.shape[1], covariance_type="diag", init_params="", n_iter=n_iter, tol=1e-3)
        h.means_ = means[mi] + 0.3 * np.sqrt(var[mi]) * rng.standard_normal(means[mi].shape)
        h.covars_ = var[mi] * 1.5
        h.transmat_, h.startprob_ = tm[mi].copy(), sp[mi].copy()
        hs.append(h)
    return hs


def _rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-300), initial=0.0))


def check(d):
    import torch
    from sapr_b200.hmmlearn_hmm import fit_vocabulary
    M, S, D = 11, 10, 13
    means, var, tm, sp = make_models(M, S, D, False, seed=77)
    rng = np.random.default_rng(78)
    words = []
    for w in range(M):
        fs = []
        for _ in range(80):
            T = int(rng.integers(40, 120))
            st = np.sort(rng.integers(0, S, T))
            fs.append((means[w, st] + np.sqrt(var[w, st]) * rng.standard_normal((T, D))).T.astype(np.float32))
        words.append(fs)
    base = _init(means, var, tm, sp, 6, 79)
    sharded = fit_vocabulary(copy.deepcopy(base), words, precision="fp64", dist=d)
    single = fit_vocabulary(copy.deepcopy(base), words, precision="fp64")
    hist = max(_rel(list(a.monitor_.history), list(b.monitor_.history)) for a, b in zip(sharded, single))
    par = max(_rel(getattr(a, k), getattr(b, k)) for a, b in zip(sharded, single)
              for k in ("means_", "_covars", "transmat_", "startprob_"))
    iters = all(a.monitor_.iter == b.monitor_.iter for a, b in zip(sharded, single))
    # every rank holds the same bytes: the maximum and minimum over ranks of every parameter agree
    flat = torch.as_tensor(np.concatenate([np.ravel(getattr(a, k)) for a in sharded for k in ("means_", "_covars", "transmat_",
                                                                                              "startprob_")]), device="cuda")
    lo, hi = flat.clone(), flat.clone()
    d.max_(hi)
    lo.neg_(); d.max_(lo); lo.neg_()
    same = bool(torch.equal(lo, hi))
    ok = hist <= 1e-12 and par <= 1e-10 and iters and same
    return {"passed": ok, "history_max_rel": hist, "params_max_rel": par, "iterations_equal": iters, "ranks_identical": same,
            "iterations": [a.monitor_.iter for a in sharded]}


def time_iteration(d, B, T, D, iters):
    import torch
    from sapr_b200 import engine as eng
    from sapr_b200._lib import ptr
    from sapr_b200.hmmlearn_hmm import GaussianHMM, expand_priors, param_flags
    M, S = 11, 10
    means, var, tm, sp = make_models(M, S, D, False, seed=D)
    m = eng.WordModels(M, S, D, eng.EMIT_DIAG, eng.TOPO_DENSE)
    m.set(means, var, tm, sp)
    hs = [GaussianHMM(n_components=S, covariance_type="diag", init_params="") for _ in range(M)]
    for h, mu in zip(hs, means):
        h.means_ = mu
    priors = torch.as_tensor(expand_priors(hs), device="cuda")
    flags = param_flags(hs)
    batch, labels = device_batch(eng, means, var, tm, B, T, seed=5 + D + 1000 * d.rank)
    lab = labels.to(torch.int64)
    ll_host = torch.empty(M, dtype=torch.float64, pin_memory=True)

    def one():
        stats, loglik, _ = m.estep(batch, labels, None, eng.FP32)
        ll_m = torch.zeros(M, dtype=torch.float64, device="cuda")
        ll_m.index_add_(0, lab, loglik)
        packed = torch.cat([stats.reshape(-1), ll_m])
        d.allreduce_(packed)
        ll_host.copy_(packed[-M:], non_blocking=True)
        ev = torch.cuda.Event()
        ev.record()
        m.ctx.check(m.lib.sapr_hl_mstep(m.ctx.h, m.h, ptr(packed), ptr(priors), ptr(flags)))
        ev.synchronize()
        return packed.numel()

    one()                                                                      # warm-up
    d.barrier(); torch.cuda.synchronize()
    m.ctx.profile(True)
    t0 = time.perf_counter()
    for _ in range(iters):
        n = one()
    torch.cuda.synchronize()
    wall = torch.tensor([(time.perf_counter() - t0) / iters], dtype=torch.float64, device="cuda")
    d.max_(wall)
    fb, _ = m.ctx.profile_read(9)
    ob, _ = m.ctx.profile_read(10)
    ms, _ = m.ctx.profile_read(11)
    m.ctx.profile(False)
    return {"D": D, "utts_per_gpu": B, "frames": T, "estep_fb_ms": round(fb / iters, 4), "estep_stats_ms": round(ob / iters, 4),
            "mstep_ms": round(ms / iters, 4), "wall_ms_per_iteration": round(float(wall.item()) * 1e3, 3),
            "allreduce_bytes": 8 * n}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--utts", type=int, default=100_000)
    ap.add_argument("--frames", type=int, default=200)
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("dense_train_dist needs a CUDA device")
    from sapr_b200.dist import Dist
    d = Dist()
    torch.cuda.set_device(d.local_rank)
    res = {"bench": "dense_train_dist", "world": d.world, **gpu_info()}
    res["check"] = check(d)
    if d.rank == 0:
        print("check", "passed" if res["check"]["passed"] else "FAILED", json.dumps(res["check"]), flush=True)
    res["weak"] = [time_iteration(d, a.utts, a.frames, D, a.iters) for D in (13, 39)]
    res["strong"] = [time_iteration(d, a.utts // d.world, a.frames, D, a.iters) for D in (13, 39)]
    d.barrier()
    if d.rank == 0:
        line = json.dumps(res)
        print(line)
        if a.out:
            with open(a.out, "w") as f:
                f.write(line + "\n")
    d.shutdown()
    if not res["check"]["passed"]:
        sys.exit(1)


if __name__ == "__main__":
    main()
