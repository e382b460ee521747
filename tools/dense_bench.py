"""Batched recognition with hmmlearn-style word models (DENSE topology, csrc/viterbi_dense.cu): prints one JSON line.

reference: 330 utterances, T ~ U{80..120}, D = 13, S = 10, M = 11 -- the reference's per-sequence loop (Decoder.decode_sequence,
           one GaussianHMM.decode per utterance x model) against one Decoder.decode_batch call, wall time around synchronised
           work, recognised words compared.
throughput: 100 000 utterances x 200 frames x 11 models, S = 10, D in {13, 39}, left-to-right (the reference's initial zero
           pattern, 2S - 2 arcs) and fully dense (Dirichlet rows) transitions.  Kernel times come from the profile classes
           (7 = dense Viterbi, 1 = its arg-max / back-trace, 8 = float64 re-decoding of near-ties), averaged over the timed calls.
           Algorithmic bytes per utterance: features T*D*4 + path T + word 4 + score 8.  The emission's SIMT bound is
           M*S*2D FMAs per utterance-frame at one FMA per lane and cycle (148 SMs x 128 lanes at the maximum SM clock).

usage: python tools/dense_bench.py [--utts 100000] [--frames 200] [--calls 5] [--out FILE]
"""
import argparse
import json
import os
import pickle
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_MEASURED_GBS = 6552.0      # measured copy bandwidth of the B200 (DESIGN §4)
SMS, LANES = 148, 128


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split(", ")
        return {"gpu": out[0], "power_limit_w": float(out[1]), "sm_max_mhz": float(out[2])}
    except Exception as e:      # noqa: BLE001 -- the line says what could not be read
        import torch
        return {"gpu": torch.cuda.get_device_name(0), "power_limit_w": None, "sm_max_mhz": None, "nvidia_smi": str(e)}


def lr_transmat(S, aii):
    A = np.zeros((S, S))
    A[0, 1] = 1.0
    for i in range(1, S - 1):
        A[i, i] = aii; A[i, i + 1] = 1 - aii
    A[S - 1, S - 1] = 1.0
    return A


def make_models(M, S, D, dense, seed):
    rng = np.random.default_rng(seed)
    scale = 10.0 if D == 13 else 1.0
    means = rng.normal(0.0, 2.0, (M, S, D)) * scale
    var = (rng.uniform(0.5, 1.5, (M, S, D)) * scale) ** 2
    if dense:
        tm = rng.dirichlet(np.ones(S), size=(M, S)); sp = rng.dirichlet(np.ones(S), size=M)
    else:
        tm = np.stack([lr_transmat(S, rng.uniform(0.8, 0.95)) for _ in range(M)])
        sp = np.zeros((M, S)); sp[:, 0] = 1.0
    return means, var, tm, sp


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
        for f in feats[:3]:
            dec.decode_sequence(f.T)                  # warm-up: module load, per-model uploads
        dec.decode_batch(feats)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        loop_words = [dec.decode_sequence(f.T)[0] for f in feats]
        torch.cuda.synchronize()
        t_loop = time.perf_counter() - t0
        t_b = []
        for _ in range(5):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            words, _, _ = dec.decode_batch(feats)
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
    res = {}
    for label, want_path in (("path", True), ("scores_only", False)):
        m.viterbi(batch, None, engine.FP32, 0, want_path=want_path)     # warm-up
        flagged = m.ctx.viterbi_flagged()
        m.ctx.profile(True)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(calls):
            m.viterbi(batch, None, engine.FP32, 0, want_path=want_path)
        torch.cuda.synchronize()
        wall = (time.perf_counter() - t0) / calls
        k7, n7 = m.ctx.profile_read(7); k1, _ = m.ctx.profile_read(1); k8, n8 = m.ctx.profile_read(8)
        m.ctx.profile(False)
        res[label] = {"viterbi_ms": round(k7 / calls, 4), "viterbi_launches_per_call": n7 // calls,
                      "finish_ms": round(k1 / calls, 4), "redecode_ms": round(k8 / calls, 4), "call_wall_ms": round(wall * 1e3, 3),
                      "flagged": flagged}
    kern_ms = res["path"]["viterbi_ms"] + res["path"]["finish_ms"]
    alg_bytes = B * (T * D * 4 + T + 4 + 8)
    fma = B * T * M * S * 2 * D
    simt_ms = fma / (SMS * LANES * clock_mhz * 1e6) * 1e3 if clock_mhz else None
    hbm_ms = alg_bytes / (HBM_MEASURED_GBS * 1e9) * 1e3
    n_arcs = int(np.sum(tm > 0))
    return {"D": D, "transitions": "dense" if dense else "left_to_right", "finite_arcs_per_model": n_arcs // M,
            "utterances": B, "frames": T, "models": M, "states": S, **res,
            "kernel_ms": round(kern_ms, 4),
            "updates_per_s": float(f"{B * T * S * M / (kern_ms * 1e-3):.4g}"),
            "alg_bytes_per_utt": alg_bytes // B, "achieved_gbs": round(alg_bytes / (kern_ms * 1e-3) / 1e9, 1),
            "fraction_of_measured_hbm": round(alg_bytes / (kern_ms * 1e-3) / 1e9 / HBM_MEASURED_GBS, 4),
            "emission_simt_bound_ms": round(simt_ms, 4) if simt_ms else None, "hbm_bound_ms": round(hbm_ms, 4),
            "bound": ("emission SIMT" if simt_ms and simt_ms > hbm_ms else "HBM"),
            "fraction_of_bound": round(max(simt_ms or 0.0, hbm_ms) / kern_ms, 4)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--utts", type=int, default=100_000)
    ap.add_argument("--frames", type=int, default=200)
    ap.add_argument("--calls", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("dense_bench needs a CUDA device")
    torch.cuda.set_device(0)
    info = gpu_info()
    line = {"bench": "dense_viterbi", **info, "reference_size": reference_size(), "throughput": []}
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
