"""hmmlearn-style surface of the reference's second implementation (assignment2/hmmlearn_hmm.py).

``GaussianHMM`` mirrors the subset of ``hmmlearn.hmm.GaussianHMM`` the reference touches
(hmmlearn_hmm.py:27-43, :103-104; train.py:116-117; decoder.py:43; visualize.py:124): constructor kwargs,
settable ``means_ / covars_ / transmat_ / startprob_``, ``fit / score / decode / predict`` and
``monitor_.history``.  hmmlearn 0.3.3 itself is not vendored in the reference and not installable here, so
the arithmetic follows SURVEY.md Appendix B (parity unpinned by the reference); it runs on the DENSE-topology
float64 kernels of csrc/hmmlearn.cu.  ``HMMLearnModel`` is the reference's wrapper class, same signature.

``decode`` is one model at a time, as decoder.py:43 calls it.  To recognise many utterances against a vocabulary of such
models at once, ``Decoder.decode_batch`` stacks them into one DENSE ``WordModels`` set (fp32 fused kernel of
csrc/viterbi_dense.cu for up to 32 states; its float64 verification mode equals this class's ``decode`` bit for bit).
``fit`` is one model at a time too; ``fit_vocabulary`` fits every word's model at once: per iteration one E-step over all
utterances of the vocabulary (csrc/estep_dense.cu) and one device M-step for every active model (``sapr_hl_mstep``, bit for bit
with ``GaussianHMM._do_mstep``), with the parameters resident on the device from the first iteration to the last.  Given a
``dist.Dist`` it shards the utterances over the ranks and sums the statistics in one all-reduce per iteration.
"""
from __future__ import annotations

import logging
from collections import deque
from typing import List

import numpy as np

from ._lib import EMIT_DIAG, TOPO_DENSE, ptr
from .engine import PackedBatch, WordModels


def _torch():
    import torch
    return torch


class ConvergenceMonitor:
    """hmmlearn.base.ConvergenceMonitor: history of per-iteration total log-probability."""

    def __init__(self, tol, n_iter, verbose=False):
        self.tol, self.n_iter, self.verbose = tol, n_iter, verbose
        self.history = deque()
        self.iter = 0

    def _reset(self):
        self.iter = 0
        self.history.clear()

    def report(self, log_prob):
        if self.verbose:
            delta = log_prob - self.history[-1] if self.history else np.nan
            print(f"{self.iter + 1:>10d} {log_prob:>16.8f} {delta:>+16.8f}")
        self.history.append(log_prob)
        self.iter += 1

    @property
    def converged(self):
        return (self.iter == self.n_iter or
                (len(self.history) >= 2 and self.history[-1] - self.history[-2] < self.tol))


class GaussianHMM:
    def __init__(self, n_components=1, covariance_type="diag", min_covar=1e-3, startprob_prior=1.0,
                 transmat_prior=1.0, means_prior=0, means_weight=0, covars_prior=1e-2, covars_weight=1,
                 algorithm="viterbi", random_state=None, n_iter=10, tol=1e-2, verbose=False, params="stmc",
                 init_params="stmc", implementation="log"):
        if covariance_type != "diag":
            raise NotImplementedError("only covariance_type='diag' is built (the reference uses nothing else)")
        if implementation != "log":
            raise NotImplementedError("only implementation='log' is built (hmmlearn_hmm.py:32)")
        self.n_components, self.covariance_type, self.min_covar = n_components, covariance_type, min_covar
        self.startprob_prior, self.transmat_prior = startprob_prior, transmat_prior
        self.means_prior, self.means_weight = means_prior, means_weight
        self.covars_prior, self.covars_weight = covars_prior, covars_weight
        self.algorithm, self.random_state, self.n_iter, self.tol = algorithm, random_state, n_iter, tol
        self.verbose, self.params, self.init_params, self.implementation = verbose, params, init_params, implementation
        self.monitor_ = ConvergenceMonitor(tol, n_iter, verbose)
        self._covars = None
        self._dev = None

    # hmmlearn stores (S, D) for "diag" and the getter expands to (S, D, D)
    @property
    def covars_(self):
        return np.array([np.diag(c) for c in self._covars])

    @covars_.setter
    def covars_(self, v):
        v = np.asarray(v, dtype=np.float64)
        self._covars = np.array([np.diag(c) for c in v]) if v.ndim == 3 else v.copy()

    def __getstate__(self):
        st = dict(self.__dict__)
        st["_dev"] = None
        st.pop("_dev_key", None)
        return st

    def __setstate__(self, st):
        self.__dict__.update(st)
        self._dev = None
        self._dev_key = None

    def _check(self):
        sp = np.asarray(self.startprob_, dtype=np.float64)
        tm = np.asarray(self.transmat_, dtype=np.float64)
        S = self.n_components
        if sp.shape != (S,) or not np.isclose(sp.sum(), 1.0):
            raise ValueError("startprob_ must have length n_components and sum to 1")
        if tm.shape != (S, S) or not np.allclose(tm.sum(axis=1), 1.0):
            raise ValueError("transmat_ rows must sum to 1")
        self.means_ = np.asarray(self.means_, dtype=np.float64)
        if self._covars is None or self._covars.shape != self.means_.shape or (self._covars <= 0).any():
            raise ValueError("'diag' covars must be positive and shaped like means_")
        self.n_features = self.means_.shape[1]

    def _models(self) -> WordModels:
        self._check()
        S, D = self.means_.shape
        if self._dev is None or (self._dev.S, self._dev.D) != (S, D):
            self._dev = WordModels(1, S, D, EMIT_DIAG, TOPO_DENSE)
        # decode / score are called once per utterance and model by decoder.py: upload only when the parameters changed
        arrs = [np.ascontiguousarray(a, dtype=np.float64) for a in (self.means_, self._covars, self.transmat_, self.startprob_)]
        key = (id(self._dev),) + tuple(hash(a.tobytes()) for a in arrs)
        if getattr(self, "_dev_key", None) != key:
            self._dev.set(*arrs)
            self._dev_key = key
        return self._dev

    @staticmethod
    def _batch(X, lengths):
        return PackedBatch.from_frames(np.asarray(X), lengths)

    def score_each(self, X, lengths=None, precision="float64"):
        """Per-sequence log-probabilities (device float64 tensor).  ``precision="float64"`` is the log-domain
        verification mode; ``"tc"`` runs the fp32 tensor-core scaled forward of csrc/ergodic_tc.cu (dense models
        with 64/128/192/256 states, BASELINE cfg 4)."""
        torch = _torch()
        m = self._models()
        b = self._batch(X, lengths)
        lp = torch.zeros(b.B, dtype=torch.float64, device=b.X.device)
        if precision not in ("float64", "tc"):
            raise ValueError("precision must be 'float64' or 'tc'")
        if precision == "float64":
            m.ctx.check(m.lib.sapr_hl_score(m.ctx.h, m.h, 0, ptr(b.X), b.ldx, ptr(b.offsets), b.B, b.total_frames, ptr(lp)))
        else:
            m.ctx.check(m.lib.sapr_ergodic_score(m.ctx.h, m.h, 0, ptr(b.X), b.ldx, ptr(b.offsets), b.B, b.max_T, ptr(lp)))
        return lp

    def score(self, X, lengths=None, precision="float64"):
        return float(self.score_each(X, lengths, precision).cpu().numpy().sum())

    def decode(self, X, lengths=None, algorithm=None):
        torch = _torch()
        m = self._models()
        b = self._batch(X, lengths)
        lp = torch.zeros(b.B, dtype=torch.float64, device=b.X.device)
        path = torch.zeros(b.total_frames, dtype=torch.int32, device=b.X.device)
        m.ctx.check(m.lib.sapr_hl_decode(m.ctx.h, m.h, 0, ptr(b.X), b.ldx, ptr(b.offsets), b.B, b.total_frames,
                                         ptr(lp), ptr(path)))
        return float(lp.cpu().numpy().sum()), path.cpu().numpy().astype(np.int64)

    def predict(self, X, lengths=None):
        return self.decode(X, lengths)[1]

    def _estep(self, m, b):
        torch = _torch()
        S, D = self.means_.shape
        n = int(m.lib.sapr_hl_stats_len(S, D))
        stats = torch.zeros(n, dtype=torch.float64, device=b.X.device)
        lp = torch.zeros(b.B, dtype=torch.float64, device=b.X.device)
        m.ctx.check(m.lib.sapr_hl_estep(m.ctx.h, m.h, 0, ptr(b.X), b.ldx, ptr(b.offsets), b.B, b.total_frames,
                                        ptr(stats), ptr(lp)))
        st = stats.cpu().numpy()
        o = 0
        out = {}
        for name, size, shape in (("start", S, (S,)), ("trans", S * S, (S, S)), ("post", S, (S,)),
                                  ("obs", S * D, (S, D)), ("obs2", S * D, (S, D))):
            out[name] = st[o:o + size].reshape(shape); o += size
        return out, float(lp.cpu().numpy().sum())

    def _do_mstep(self, st):
        """hmmlearn 0.3.3 BaseHMM._do_mstep + GaussianHMM._do_mstep for 'diag' (SURVEY Appendix B)."""
        if "s" in self.params:
            sp = np.maximum(self.startprob_prior - 1 + st["start"], 0)
            sp = np.where(self.startprob_ == 0, 0, sp)
            self.startprob_ = sp / sp.sum()
        if "t" in self.params:
            tm = np.maximum(self.transmat_prior - 1 + st["trans"], 0)
            tm = np.where(self.transmat_ == 0, 0, tm)
            rs = tm.sum(axis=1, keepdims=True)
            rs[rs == 0] = 1
            self.transmat_ = tm / rs
        denom = st["post"][:, None]
        if "m" in self.params:
            self.means_ = (self.means_weight * self.means_prior + st["obs"]) / (self.means_weight + denom)
        if "c" in self.params:
            meandiff = self.means_ - self.means_prior
            c_n = (self.means_weight * meandiff ** 2 + st["obs2"] - 2 * self.means_ * st["obs"] + self.means_ ** 2 * denom)
            c_d = max(self.covars_weight - 1, 0) + denom
            self._covars = (self.covars_prior + c_n) / np.maximum(c_d, 1e-5)

    def fit(self, X, lengths=None):
        b = self._batch(X, lengths)
        self._check()
        self.monitor_ = ConvergenceMonitor(self.tol, self.n_iter, self.verbose)
        self.monitor_._reset()
        for _ in range(self.n_iter):
            m = self._models()
            st, logprob = self._estep(m, b)
            self._do_mstep(st)
            self.monitor_.report(logprob)
            if self.monitor_.converged:
                break
        return self


class _hmm_ns:
    GaussianHMM = GaussianHMM


hmm = _hmm_ns   # `from hmmlearn import hmm` look-alike used by the reference wrapper


class HMMLearnModel:
    """assignment2/hmmlearn_hmm.py:11-108, same constructor and methods; ``feature_set`` may be passed
    directly instead of being re-loaded from ./feature_set (hmmlearn_hmm.py:23)."""

    def __init__(self, num_states: int = 8, model_name: str = None, n_iter: int = 15, min_covar: float = 0.01,
                 feature_set=None):
        self.model_name = model_name
        self.num_states = num_states
        self.total_states = num_states + 2
        if feature_set is None:
            from .mfcc_extract import load_mfccs
            feature_set = load_mfccs("feature_set")
        self.all_features = feature_set
        self.global_mean = self.calc_global_mean(self.all_features)
        self.global_cov = self.calc_global_cov(self.all_features)
        self.model = GaussianHMM(n_components=self.total_states, covariance_type="diag", n_iter=n_iter, params="stmc",
                                 implementation="log", min_covar=min_covar, init_params="")
        self.model.means_ = np.tile(self.global_mean, (self.total_states, 1))
        self.model.covars_ = np.tile(self.global_cov, (self.total_states, 1))
        self.model.transmat_ = self.initialize_transmat()
        self.model.startprob_ = np.zeros(self.total_states)
        self.model.startprob_[0] = 1.0

    def initialize_transmat(self) -> np.ndarray:
        total_frames = sum(f.shape[1] for f in self.all_features)
        avg_frames_per_state = total_frames / len(self.all_features) / self.num_states
        aii = np.exp(-1 / (avg_frames_per_state - 1))
        transmat = np.zeros((self.total_states, self.total_states))
        transmat[0, 1] = 1.0
        for i in range(1, self.num_states + 1):
            transmat[i, i] = aii
            transmat[i, i + 1] = 1 - aii
        transmat[self.num_states + 1, self.num_states + 1] = 1.0
        return transmat

    def prepare_data(self, feature_set: List[np.ndarray]) -> np.ndarray:
        return np.concatenate([f.T for f in feature_set], axis=0)

    def _global_stats(self, feature_set):
        # global mean / population variance (hmmlearn_hmm.py:83-94) from the GPU flat-start sums
        from .engine import init_flat_start
        b = PackedBatch.from_features(feature_set)
        gmean, var, _, _ = init_flat_start(b, self.num_states, var_floor_factor=0.0)
        return gmean, var

    def calc_global_mean(self, feature_set):
        return self._global_stats(feature_set)[0]

    def calc_global_cov(self, feature_set):
        return self._global_stats(feature_set)[1]

    def fit(self, feature_set: List[np.ndarray]):
        logging.info(f"Training {self.model_name} HMM using hmmlearn in {self.model.n_iter} iterations...")
        X = self.prepare_data(feature_set)
        lengths = [f.shape[1] for f in feature_set]
        try:
            self.model.fit(X, lengths)
            log_likelihood = self.model.score(X, lengths)
            return self.model, log_likelihood
        except Exception as e:   # the reference swallows and returns None (hmmlearn_hmm.py:107-108)
            logging.error(f"Error occurred while training {self.model_name} HMM: {e}")


_PARAM_BITS = {"s": 1, "t": 2, "m": 4, "c": 8}


def expand_priors(models: List[GaussianHMM]) -> np.ndarray:
    """The priors of every model as the float64 block ``sapr_hl_mstep`` reads, one row per model:
    [startprob_prior S | transmat_prior S*S | means_prior S*D | means_weight S*D | covars_prior S*D | covars_weight].
    Each prior is a scalar or an array of exactly its parameter's shape (``startprob_prior`` (S,), ``transmat_prior`` (S, S),
    the means and covariance priors (S, D)); ``covars_weight`` is a scalar, as ``_do_mstep`` passes it to Python's ``max``.
    ValueError otherwise."""
    rows = []
    for i, mdl in enumerate(models):
        S, D = np.shape(mdl.means_)
        parts = []
        for name, shape in (("startprob_prior", (S,)), ("transmat_prior", (S, S)), ("means_prior", (S, D)),
                            ("means_weight", (S, D)), ("covars_prior", (S, D)), ("covars_weight", ())):
            v = np.asarray(getattr(mdl, name), dtype=np.float64)
            if v.shape not in ((), shape):
                raise ValueError(f"model {i}: {name} must be a scalar" + (f" or shaped {shape}" if shape else "") +
                                 f"; got shape {v.shape}")
            parts.append(np.broadcast_to(v, shape).ravel())
        rows.append(np.concatenate(parts))
    return np.stack(rows)


def param_flags(models: List[GaussianHMM]) -> np.ndarray:
    """int32[M]: the letters of each model's ``params`` as ``sapr_hl_mstep``'s flag bits ('s' 1, 't' 2, 'm' 4, 'c' 8)."""
    return np.array([sum(b for c, b in _PARAM_BITS.items() if c in mdl.params) for mdl in models], dtype=np.int32)


def vocabulary_shards(lengths, world: int):
    """(u_begin, u_end) per rank over the model-grouped utterance list (``lengths`` = frames per utterance, every utterance of
    model 0, then of model 1, ...): contiguous, frame-balanced ranges that cover every utterance once (``dist.shard_bounds``)."""
    from .dist import shard_bounds
    return shard_bounds(np.concatenate([[0], np.cumsum(np.asarray(lengths, dtype=np.int64))]), world)


def fit_vocabulary(models: List[GaussianHMM], features, precision: str = "fp32", dist=None) -> List[GaussianHMM]:
    """Fit every model of a vocabulary at once: ``features[m]`` is model m's list of (D, T) arrays.  The end state equals
    ``models[m].fit(X_m, lengths_m)`` for each m.  The parameters stay on the device for the whole fit: every iteration runs ONE
    dense E-step over all utterances (each against its own word's model), then ``sapr_hl_mstep`` -- hmmlearn's ``_do_mstep``
    for every model still active, bit for bit -- then each active model's ``monitor_.report``: the order ``GaussianHMM.fit``
    uses, so priors, ``params`` and the zero masks of ``startprob_`` / ``transmat_`` behave as in the per-model fit.  A model
    leaves the active set when its monitor has converged (its own ``n_iter`` and ``tol``); its parameters then stay as they
    are.  The fitted parameters are written back to the models once, at the end.  ``precision="fp64"`` runs GaussianHMM.fit's
    float64 E-step per model and is bit-identical to the per-model fits; ``"fp32"`` is the fused kernel (up to 32 states).

    ``dist`` (a ``dist.Dist``) shards the utterances over its ranks: every rank passes the whole vocabulary and runs the
    E-step on its contiguous, frame-balanced share of the model-grouped utterance list; the statistics and the per-model
    log-likelihood sums are summed over the ranks in ONE all-reduce per iteration, so every rank takes the same M-step and
    convergence decisions and ends with the same parameters and histories.  Returns ``models``."""
    from ._lib import FP32, FP64
    from .decoder import stack_hmmlearn_models
    torch = _torch()
    if precision not in ("fp32", "fp64"):
        raise ValueError("precision must be 'fp32' or 'fp64'")
    if len(models) != len(features):
        raise ValueError(f"{len(models)} models but {len(features)} feature lists")
    for i, (mdl, f) in enumerate(zip(models, features)):
        if len(f) == 0:
            raise ValueError(f"model {i} has no utterances to fit")
        mdl._check()
    means, var, tm, sp = stack_hmmlearn_models(models)
    M, S, D = means.shape
    priors, flags = expand_priors(models), param_flags(models)
    feats = [np.asarray(x, dtype=np.float32) for f in features for x in f]
    if any(x.ndim != 2 or x.shape[0] != D for x in feats):
        raise ValueError(f"every utterance must be a (D, T) array with D = {D} features")
    counts = np.array([len(f) for f in features])
    bounds = np.concatenate([[0], np.cumsum(counts)])
    labels = np.repeat(np.arange(M), counts)
    sharded = dist is not None and dist.world > 1
    u0, u1 = vocabulary_shards([x.shape[1] for x in feats], dist.world)[dist.rank] if sharded else (0, len(feats))
    # a rank whose shard is empty still takes part in every all-reduce, with zero statistics
    batch = PackedBatch.from_features(feats[u0:u1], labels=labels[u0:u1]) if u1 > u0 else None
    dev = WordModels(M, S, D, EMIT_DIAG, TOPO_DENSE)
    dev.set(means, var, tm, sp)
    device = dev.ctx.device
    d_priors = torch.as_tensor(priors, device=device)
    prec = FP64 if precision == "fp64" else FP32
    lab = None if batch is None else batch.labels.to(torch.int64)
    ll_host = torch.empty(M if sharded else u1 - u0, dtype=torch.float64, pin_memory=True)
    for mdl in models:
        mdl.monitor_ = ConvergenceMonitor(mdl.tol, mdl.n_iter, mdl.verbose)
        mdl.monitor_._reset()
    active = [i for i, mdl in enumerate(models) if mdl.n_iter > 0]
    while active:
        if batch is not None:
            stats, loglik, _ = dev.estep(batch, batch.labels, None, prec)
        else:
            stats = torch.zeros((M, dev.stats_stride()), dtype=torch.float64, device=device)
            loglik = torch.zeros(0, dtype=torch.float64, device=device)
        if sharded:
            ll_m = torch.zeros(M, dtype=torch.float64, device=device)
            if lab is not None:
                ll_m.index_add_(0, lab, loglik)
            packed = torch.cat([stats.reshape(-1), ll_m])
            dist.allreduce_(packed)
            stats, loglik = packed[:-M], packed[-M:]
        ll_host.copy_(loglik, non_blocking=True)        # the host reads it while the M-step runs
        copied = torch.cuda.Event()
        copied.record()
        step = np.zeros(M, dtype=np.int32)
        step[active] = flags[active]
        dev.ctx.check(dev.lib.sapr_hl_mstep(dev.ctx.h, dev.h, ptr(stats), ptr(d_priors), ptr(step)))
        copied.synchronize()
        ll = ll_host.numpy()
        still = []
        for i in active:
            mdl = models[i]
            mdl.monitor_.report(float(ll[i]) if sharded else float(ll[bounds[i]:bounds[i + 1]].sum()))
            if not mdl.monitor_.converged:
                still.append(i)
        active = still
    means, var, tm, sp = dev.get()
    for i, mdl in enumerate(models):
        if mdl.monitor_.iter == 0:
            continue
        if "s" in mdl.params:
            mdl.startprob_ = sp[i].copy()
        if "t" in mdl.params:
            mdl.transmat_ = tm[i].copy()
        if "m" in mdl.params:
            mdl.means_ = means[i].copy()
        if "c" in mdl.params:
            mdl._covars = var[i].copy()
    return models
