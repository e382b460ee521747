"""Batched host layer over the C ABI: packed utterance batches and device-resident word-model sets.

This is the throughput surface (BASELINE configs 2 and 3): every utterance x every word model in one
call, utterances sharded across GPUs, only the packed per-model sufficient statistics all-reduced.
The reference-shaped classes (``custom_hmm.HMM``, ``hmmlearn_hmm.GaussianHMM``) sit on top of it.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence

import numpy as np

from . import _lib
from ._lib import EMIT_DIAG, EMIT_SAPR, FP32, FP32_SIMT, FP64, TOPO_DENSE, TOPO_ENTRY_EXIT, ptr


def _torch():
    import torch
    return torch


class PackedBatch:
    """Features in the HBM layout every kernel reads: float32 frame-major ``X[sum_T, Dpad]`` (Dpad = D
    rounded up to 4 floats = 16-byte rows), ``offsets[B+1]`` int64.  The reference keeps a Python list
    of (D, T_u) arrays (mfcc_extract.py:41-42, :63-76); hmmlearn's ``X, lengths`` (hmmlearn_hmm.py:80-81,
    :100-101) is the same thing un-padded."""

    def __init__(self, X, offsets, D, offsets_host=None, labels=None):
        torch = _torch()
        self.X, self.offsets, self.D = X, offsets, int(D)
        self.ldx = int(X.shape[1])
        self.offsets_host = (offsets.cpu().numpy() if offsets_host is None else np.asarray(offsets_host, dtype=np.int64))
        self.B = len(self.offsets_host) - 1
        self.total_frames = int(self.offsets_host[-1])
        lens = np.diff(self.offsets_host)
        self.max_T = int(lens.max()) if self.B else 0
        self.min_T = int(lens.min()) if self.B else 0
        self.labels = labels
        assert X.dtype == torch.float32 and X.is_cuda and X.is_contiguous()
        assert self.ldx % 4 == 0 and self.ldx >= self.D

    @classmethod
    def from_features(cls, features: Sequence[np.ndarray], device=None, labels=None):
        """features: list of (D, T_u) arrays, the orientation the reference stores."""
        torch = _torch()
        from .synth import pack_frame_major
        Xh, offs = pack_frame_major([np.asarray(f, dtype=np.float32) for f in features])
        dev = device if device is not None else torch.device("cuda", torch.cuda.current_device())
        X = torch.from_numpy(Xh).to(dev)
        lab = None if labels is None else torch.as_tensor(np.asarray(labels, dtype=np.int32), device=dev)
        return cls(X, torch.from_numpy(offs).to(dev), features[0].shape[0], offs, lab)

    @classmethod
    def from_frames(cls, X_TD: np.ndarray, lengths=None, device=None):
        """hmmlearn layout: X (sum_T, D) + lengths."""
        torch = _torch()
        X_TD = np.asarray(X_TD)
        T, D = X_TD.shape
        lengths = [T] if lengths is None else list(lengths)
        assert sum(lengths) == T, "lengths must sum to the number of rows of X"
        dp = (D + 3) // 4 * 4
        Xh = np.zeros((T, dp), dtype=np.float32)
        Xh[:, :D] = X_TD
        offs = np.zeros(len(lengths) + 1, dtype=np.int64)
        offs[1:] = np.cumsum(lengths)
        dev = device if device is not None else torch.device("cuda", torch.cuda.current_device())
        return cls(torch.from_numpy(Xh).to(dev), torch.from_numpy(offs).to(dev), D, offs)


class WordModels:
    """M word models resident on the GPU (parameter block of custom_hmm.py:10-33 x M)."""

    def __init__(self, M, N, D, emission=EMIT_DIAG, topology=TOPO_ENTRY_EXIT, ctx: Optional[_lib.Context] = None):
        self.ctx = ctx or _lib.default_context()
        self.lib = self.ctx.lib
        self.M, self.N, self.D, self.emission, self.topology = int(M), int(N), int(D), emission, topology
        self.S = self.N + 2 if topology == TOPO_ENTRY_EXIT else self.N
        h = C.c_void_p()
        self.ctx.check(self.lib.sapr_models_create(self.ctx.h, self.M, self.N, self.D, emission, topology, C.byref(h)))
        self.h = h

    def __del__(self):
        try:
            if getattr(self, "h", None) and getattr(self.ctx, "h", None):
                self.lib.sapr_models_destroy(self.h)
                self.h = None
        except Exception:
            pass

    # ---- parameters ----
    def cov_shape(self):
        return (self.M, self.S, self.D) if self.emission == EMIT_DIAG else (self.M, self.S, self.D, self.D)

    def set(self, means, covars, transmat, startprob=None):
        means = np.ascontiguousarray(means, dtype=np.float64).reshape(self.M, self.S, self.D)
        covars = np.ascontiguousarray(covars, dtype=np.float64).reshape(self.cov_shape())
        transmat = np.ascontiguousarray(transmat, dtype=np.float64).reshape(self.M, self.S, self.S)
        sp = None
        if self.topology == TOPO_DENSE:
            sp = np.ascontiguousarray(startprob, dtype=np.float64).reshape(self.M, self.S)
        self.ctx.check(self.lib.sapr_models_set(self.h, ptr(means), ptr(covars), ptr(transmat), ptr(sp)))

    def get(self):
        means = np.empty((self.M, self.S, self.D)); covars = np.empty(self.cov_shape())
        A = np.empty((self.M, self.S, self.S)); sp = np.empty((self.M, self.S))
        self.ctx.check(self.lib.sapr_models_get(self.h, ptr(means), ptr(covars), ptr(A), ptr(sp)))
        return means, covars, A, sp

    # ---- decoding (custom_hmm.py:462-514 / GaussianHMM.decode + decoder.py:42-47) ----
    def viterbi(self, batch: PackedBatch, model_of_utt=None, precision=FP32, first_frames=0, want_scores=False,
                want_path=True, all_paths=False):
        torch = _torch()
        dev = batch.X.device
        if first_frames > 0 and self.topology == TOPO_DENSE:
            raise _lib.SaprError(-1, "first_frames > 0 (walk only the first frames) is the custom models' as-written decode; "
                                     "dense (hmmlearn) models always decode every frame")
        if first_frames > 0 and batch.min_T < first_frames:
            raise IndexError("utterance shorter than the frames decode walks (reference: custom_hmm.py:466 with T_frames < D)")
        B, M = batch.B, self.M
        nslots = 1 if model_of_utt is not None else M
        best_word = torch.empty(B, dtype=torch.int32, device=dev)
        best_score = torch.empty(B, dtype=torch.float64, device=dev)
        scores = torch.empty((B, nslots), dtype=torch.float64, device=dev) if want_scores else None
        # every frame of every utterance is written when all frames are walked; the as-written mode (first_frames > 0) walks fewer
        path = (torch.zeros if first_frames > 0 else torch.empty)(batch.total_frames, dtype=torch.uint8, device=dev) if want_path else None
        allp = torch.zeros((nslots, batch.total_frames), dtype=torch.uint8, device=dev) if all_paths else None
        self.ctx.check(self.lib.sapr_viterbi(self.ctx.h, self.h, ptr(batch.X), batch.ldx, ptr(batch.offsets), B,
                                             batch.total_frames, batch.max_T, ptr(model_of_utt), precision, first_frames,
                                             ptr(best_word), ptr(best_score), ptr(scores), ptr(path), ptr(allp)))
        return dict(best_word=best_word, best_score=best_score, scores=scores, path=path, all_paths=allp)

    # ---- scoring (GaussianHMM.score per model + the arg-max over the models: recognition by total likelihood) ----
    def score_words(self, batch: PackedBatch, precision=FP32, want_scores=True):
        """log P(X_u | model m) for every utterance x model of a DENSE set, and the strict-'>' arg-max over the models (first
        best wins, -1 when no model can produce the utterance).  Returns dict(best_word, best_score, scores [B, M] or None).
        FP64 = GaussianHMM.score per model, bit for bit; FP32 = the fused forward of csrc/score_dense.cu (S <= 32), which
        re-scores word near-ties in float64 (``ctx.viterbi_flagged()`` counts them)."""
        torch = _torch()
        dev = batch.X.device
        B, M = batch.B, self.M
        best_word = torch.empty(B, dtype=torch.int32, device=dev)
        best_score = torch.empty(B, dtype=torch.float64, device=dev)
        scores = torch.empty((B, M), dtype=torch.float64, device=dev) if want_scores else None
        self.ctx.check(self.lib.sapr_score_words(self.ctx.h, self.h, ptr(batch.X), batch.ldx, ptr(batch.offsets), B,
                                                 batch.total_frames, precision, ptr(best_word), ptr(best_score), ptr(scores)))
        return dict(best_word=best_word, best_score=best_score, scores=scores)

    def tc_emission(self, batch: PackedBatch):
        """Debug/parity: the tensor-core emission tile, float32 [sum_T, ncols] (column m*8 + j-1)."""
        torch = _torch()
        ncols = (self.M * 8 + 15) // 16 * 16
        E = torch.zeros((batch.total_frames, ncols), dtype=torch.float32, device=batch.X.device)
        nc = C.c_int(0)
        self.ctx.check(self.lib.sapr_debug_tc_emission(self.ctx.h, self.h, ptr(batch.X), batch.ldx, ptr(batch.offsets), batch.B,
                                                       batch.total_frames, batch.max_T, ptr(E), C.byref(nc)))
        assert nc.value == ncols
        return E

    def viterbi_host(self, X_host, offsets_host, precision=FP32, first_frames=0, chunk_utts=8192, want_path=True,
                     out=None):
        """Host-buffer call (numpy or pinned torch CPU tensors in, numpy out): H2D/D2H inside."""
        B = len(offsets_host) - 1
        total = int(offsets_host[-1])
        if out is None:
            out = dict(best_word=np.empty(B, dtype=np.int32), best_score=np.empty(B, dtype=np.float64),
                       path=np.empty(total, dtype=np.uint8) if want_path else None)
        ldx = int(X_host.shape[1])
        self.ctx.check(self.lib.sapr_viterbi_host(self.ctx.h, self.h, ptr(X_host), ldx, ptr(offsets_host), B, precision,
                                                  first_frames, chunk_utts, ptr(out["best_word"]), ptr(out["best_score"]),
                                                  ptr(out.get("path"))))
        return out

    # ---- training (custom_hmm.py:402-460) ----
    def stats_stride(self):
        if self.topology == TOPO_DENSE:
            return int(self.lib.sapr_hl_stats_len(self.S, self.D))
        return int(self.lib.sapr_stats_stride(self.N, self.D))

    def estep(self, batch: PackedBatch, model_of_utt, order=None, precision=FP32, want_gamma=False):
        """One E-step, utterance u against model ``model_of_utt[u]``: (stats [M, stats_stride()], per-utterance loglik, gamma or
        None).  DENSE sets give hmmlearn's statistics per model (``unpack_stats``) and log P(X_u); fp32 = csrc/estep_dense.cu,
        FP64 = GaussianHMM.fit's E-step per model, bit for bit."""
        torch = _torch()
        dev = batch.X.device
        stats = torch.empty((self.M, self.stats_stride()), dtype=torch.float64, device=dev)
        loglik = torch.zeros(batch.B, dtype=torch.float64, device=dev)
        gamma = None
        if want_gamma:
            gamma = torch.zeros((batch.total_frames, self.N), dtype=torch.float32 if precision == FP32 else torch.float64,
                                device=dev)
        self.ctx.check(self.lib.sapr_estep(self.ctx.h, self.h, ptr(batch.X), batch.ldx, ptr(batch.offsets), batch.B,
                                           batch.total_frames, batch.max_T, ptr(model_of_utt), ptr(order), precision,
                                           ptr(stats), ptr(loglik), ptr(gamma)))
        return stats, loglik, gamma

    def mstep(self, stats, floor_var):
        fv = np.ascontiguousarray(np.broadcast_to(np.asarray(floor_var, dtype=np.float64), (self.M,)))
        self.ctx.check(self.lib.sapr_mstep(self.ctx.h, self.h, ptr(stats), ptr(fv)))

    def unpack_stats(self, stats):
        """stats tensor/array (M, stride) -> dict of numpy views: (G, Xi, occ, s1, s2) for ENTRY_EXIT sets, hmmlearn's
        (start, trans, post, obs, obs2) for DENSE sets."""
        st = stats.cpu().numpy() if hasattr(stats, "cpu") else np.asarray(stats)
        S, D = self.S, self.D
        if self.topology == TOPO_DENSE:
            o = np.cumsum([0, S, S * S, S, S * D])
            return dict(start=st[:, :o[1]], trans=st[:, o[1]:o[2]].reshape(self.M, S, S), post=st[:, o[2]:o[3]],
                        obs=st[:, o[3]:o[4]].reshape(self.M, S, D), obs2=st[:, o[4]:].reshape(self.M, S, D))
        return dict(G=st[:, :S], Xi=st[:, S:2 * S], occ=st[:, 2 * S:3 * S],
                    s1=st[:, 3 * S:3 * S + S * D].reshape(self.M, S, D),
                    s2=st[:, 3 * S + S * D:].reshape(self.M, S, D))


def group_by_model(labels):
    """order[B] (stable, utterances grouped by model) computed on device (torch: plumbing only)."""
    torch = _torch()
    return torch.sort(labels.to(torch.int64), stable=True).indices.to(torch.int32).contiguous()


def init_flat_start(batch: PackedBatch, N: int, var_floor_factor: float = 0.001, ctx=None, dist=None):
    """custom_hmm.py:35-116 on the GPU: two passes (mean, then centred second moment) exactly like
    calculate_means / calculate_covariance; with ``dist`` the two small sums are all-reduced."""
    torch = _torch()
    ctx = ctx or _lib.default_context()
    D = batch.D
    out = torch.zeros(2 * D + 2, dtype=torch.float64, device=batch.X.device)
    ctx.check(ctx.lib.sapr_init_stats(ctx.h, ptr(batch.X), batch.ldx, ptr(batch.offsets), batch.B, D, ptr(None), ptr(out)))
    if dist is not None:
        dist.allreduce_(out)
    frames, utts = float(out[2 * D]), float(out[2 * D + 1])
    mean = out[:D] / frames
    out2 = torch.zeros_like(out)
    ctx.check(ctx.lib.sapr_init_stats(ctx.h, ptr(batch.X), batch.ldx, ptr(batch.offsets), batch.B, D, ptr(mean.contiguous()),
                                      ptr(out2)))
    if dist is not None:
        dist.allreduce_(out2)
    var = (out2[D:2 * D] / frames).cpu().numpy()
    gmean = mean.cpu().numpy()
    floor_v = var_floor_factor * float(np.mean(var))
    var = np.maximum(var, floor_v)
    S = N + 2
    avg = frames / (utts * N)
    aii = float(np.exp(-1.0 / (avg - 1.0)))
    A = np.zeros((S, S))
    A[0, 1] = 1.0
    for i in range(1, N + 1):
        A[i, i] = aii
        A[i, i + 1] = 1.0 - aii
    A[-1, -1] = 1.0
    return gmean, var, A, floor_v


def train_words(models: WordModels, batch: PackedBatch, labels, n_iter: int, floor_var, precision=FP32, tol=1e-4,
                dist=None, order=None, callback=None):
    """Whole-vocabulary Baum-Welch (train.py:106-121 + custom_hmm.py:402-460): every iteration is one
    batched E-step over all utterances (each against its own word model), ONE all-reduce of the packed
    statistics when sharded, then the M-step replicated on every GPU.  Returns per-iteration per-model LL."""
    torch = _torch()
    if order is None:
        order = group_by_model(labels)
    history = []
    prev = None
    for it in range(n_iter):
        ll_m = torch.zeros(models.M, dtype=torch.float64, device=batch.X.device)
        stats, loglik, _ = models.estep(batch, labels, order, precision)
        ll_m.index_add_(0, labels.to(torch.int64), loglik)
        if dist is not None:
            packed = torch.cat([stats.reshape(-1), ll_m])
            dist.allreduce_(packed)
            stats = packed[:-models.M].reshape(models.M, -1).contiguous()
            ll_m = packed[-models.M:]
        history.append(ll_m.cpu().numpy())
        if callback:
            callback(it, history[-1])
        tot = float(history[-1].sum())
        if prev is not None and abs(tot - prev) < tol:
            break
        prev = tot
        models.mstep(stats, floor_var)
    return np.asarray(history)


def confusion_on_device(truth, pred, M: int, ctx=None):
    """eval.py:28-38 on the device: (cm int64 [M, M + 1] tensor, accuracy) from int32 label / prediction tensors that
    stay on the GPU (the predictions are the Viterbi kernel's best_word output); column M counts utterances no model reaches."""
    torch = _torch()
    ctx = ctx or _lib.default_context()
    truth = truth.to(device=pred.device, dtype=torch.int32).contiguous()
    pred = pred.to(dtype=torch.int32).contiguous()
    B = int(pred.numel())
    cm = torch.empty((M, M + 1), dtype=torch.int64, device=pred.device)
    correct = torch.empty(1, dtype=torch.int64, device=pred.device)
    ctx.check(ctx.lib.sapr_confusion(ctx.h, ptr(truth), ptr(pred), B, M, ptr(cm), ptr(correct)))
    acc = float(correct.item()) / B if B else float("nan")
    return cm, acc
