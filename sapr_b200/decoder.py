"""Drop-in for assignment2/decoder.py: same ``Decoder`` class (constructor, ``load_models``,
``decode_sequence``, ``decode_word_samples``, ``decode_vocabulary``) plus ``decode_batch``, which scores
every utterance against every word model in ONE fused Viterbi launch (the per-model Python loop of
decoder.py:42-47 becomes the in-kernel argmax).  ``decode_batch`` takes custom models trained with
semantics="standard" (left-to-right, entry/exit states) and hmmlearn-style models (every state emits,
dense transmat + startprob, up to 32 states; csrc/viterbi_dense.cu).  ``score_batch`` recognises hmmlearn-style models by
total likelihood instead (the arg-max over the models of GaussianHMM.score) and returns the whole utterance x model
log-likelihood matrix, from one fused forward launch (csrc/score_dense.cu).

Model order: the reference iterates ``impl_dir.glob(pattern)`` (filesystem order, SURVEY D8) and keeps the
first best under strict ``>``; pass ``vocab_order`` to fix the order explicitly.
"""
from __future__ import annotations

import logging
import pickle
from pathlib import Path
from typing import Dict, List, Tuple

import numpy as np

from ._lib import EMIT_DIAG, FP32, FP64, TOPO_DENSE, TOPO_ENTRY_EXIT
from .engine import PackedBatch, WordModels
from .mfcc_extract import load_mfccs_by_word

logging.basicConfig(level=logging.INFO)


def stack_hmmlearn_models(models) -> Tuple[np.ndarray, np.ndarray, np.ndarray, np.ndarray]:
    """(means [M, S, D], variances [M, S, D], transmat [M, S, S], startprob [M, S]) of hmmlearn-style GaussianHMM models with
    diagonal covariances.  Reads only the public attributes ``means_``, ``covars_`` (the getter's expanded (S, D, D) form;
    its diagonal is taken), ``transmat_`` and ``startprob_``, so pickles of hmmlearn's own class stack too.  Every model must
    have the same number of states and features (ValueError otherwise)."""
    means = [np.asarray(m.means_, dtype=np.float64) for m in models]
    shapes = {mu.shape for mu in means}
    if len(shapes) != 1:
        raise ValueError(f"batched decoding needs models of one shape (states, features); got {sorted(shapes)}")
    var = []
    for m in models:
        c = np.asarray(m.covars_, dtype=np.float64)
        var.append(np.diagonal(c, axis1=1, axis2=2) if c.ndim == 3 else c)
    return (np.stack(means), np.stack(var), np.stack([np.asarray(m.transmat_, dtype=np.float64) for m in models]),
            np.stack([np.asarray(m.startprob_, dtype=np.float64) for m in models]))


class Decoder:
    def __init__(self, models_dir: str = "trained_models", implementation: str = "hmmlearn", n_iter: int = 15,
                 vocab_order: List[str] = None, precision: str = "fp32"):
        self.models_dir = Path(models_dir)
        self.implementation = implementation
        self.n_iter = n_iter
        self.models: Dict = {}
        self.vocab: List[str] = []
        self.precision = precision
        self._vocab_order = vocab_order
        self._dev = None
        self.load_models()

    def load_models(self) -> None:
        impl_dir = self.models_dir / self.implementation
        pattern = f"*_{self.implementation}_{self.n_iter}.pkl"
        paths = list(impl_dir.glob(pattern))
        if self._vocab_order is not None:
            paths.sort(key=lambda p: self._vocab_order.index(p.stem.split("_")[0]))
        for model_path in paths:
            word = model_path.stem.split("_")[0]
            with open(model_path, "rb") as f:
                self.models[word] = pickle.load(f)
                self.vocab.append(word)
        if not self.models:
            raise ValueError(f"No models found in {impl_dir} with pattern {pattern}")
        logging.info(f"Loaded {len(self.models)} models from {impl_dir} for words: {', '.join(self.vocab)}")

    def decode_sequence(self, features: np.ndarray) -> Tuple[str, float, List[int]]:
        """features (T, D) as decoder.py:59 hands them; per-model loop exactly like the reference."""
        if self.implementation == "custom":
            features = features.T
        best_score, best_word, best_states = float("-inf"), None, None
        for word, model in self.models.items():
            log_prob, states = model.decode(features)
            if log_prob > best_score:
                best_score, best_word, best_states = log_prob, word, states
        return best_word, best_score, best_states

    # ---- batched path: custom "standard"-semantics models (diagonal emission, all frames) or hmmlearn models ----
    def _word_models(self) -> WordModels:
        if self._dev is None and self.implementation == "hmmlearn":
            means, var, tm, sp = stack_hmmlearn_models([self.models[w] for w in self.vocab])
            M, S, D = means.shape
            dev = WordModels(M, S, D, EMIT_DIAG, TOPO_DENSE)
            dev.set(means, var, tm, sp)
            self._dev = dev
        if self._dev is None:
            ms = [self.models[w] for w in self.vocab]
            if any(getattr(m, "semantics", None) != "standard" for m in ms):
                raise ValueError("decode_batch needs custom HMM models trained with semantics='standard'")
            N, D = ms[0].num_states, ms[0].num_obs
            dev = WordModels(len(ms), N, D, EMIT_DIAG, TOPO_ENTRY_EXIT)
            means = np.stack([m.B["mean"] for m in ms])
            var = np.stack([np.diagonal(m.B["covariance"], axis1=1, axis2=2) for m in ms])
            dev.set(means, var, np.stack([m.A for m in ms]))
            self._dev = dev
        return self._dev

    def decode_batch(self, features: List[np.ndarray], true_labels=None):
        """features: list of (D, T_u) arrays.  Returns (words, scores, paths) for the whole list; a word is None when no model
        can produce the utterance.  ``precision="fp64"`` (constructor) selects the float64 verification mode; the fp32
        default re-decodes word near-ties in float64, so its words are the float64 ones.  Custom models give the reference's
        decode (entry/exit states); hmmlearn models give GaussianHMM.decode per model (paths over states 0..S-1, the first
        best model wins ties as in decoder.py:42-47).  With ``true_labels``
        (vocabulary indices) the confusion counts and the accuracy of eval.py:28-38 are accumulated on the device from the
        kernel's predictions and left in ``self.last_confusion`` = (int64 [M, M + 1] array, accuracy)."""
        dev = self._word_models()
        batch = PackedBatch.from_features(features)
        out = dev.viterbi(batch, None, FP64 if self.precision == "fp64" else FP32, 0, want_path=True)
        if true_labels is not None:
            import torch
            from .engine import confusion_on_device
            cm, acc = confusion_on_device(torch.as_tensor(np.asarray(true_labels, dtype=np.int32)), out["best_word"], len(self.vocab), dev.ctx)
            self.last_confusion = (cm.cpu().numpy(), acc)
        bw = out["best_word"].cpu().numpy(); bs = out["best_score"].cpu().numpy(); p = out["path"].cpu().numpy()
        offs = batch.offsets_host
        words = [self.vocab[i] if i >= 0 else None for i in bw]
        return words, bs, [p[offs[u]:offs[u + 1]].tolist() for u in range(batch.B)]

    def score_batch(self, features: List[np.ndarray], true_labels=None):
        """Recognition by total likelihood for hmmlearn models: features is a list of (D, T_u) arrays.  Returns (words,
        best_scores, loglik): loglik is the [B, M] numpy matrix of GaussianHMM.score for every utterance and model in vocabulary
        order, words the arg-max over the models (first best wins ties; None when no model can produce the utterance).
        ``precision="fp64"`` (constructor) gives GaussianHMM.score per model bit for bit; the fp32 default re-scores word
        near-ties in float64, so its words are the float64 ones.  ``true_labels`` fills ``self.last_confusion`` as
        ``decode_batch`` does.  Custom models raise ValueError."""
        if self.implementation != "hmmlearn":
            raise ValueError("score_batch needs hmmlearn-style models (every state emits, dense transmat + startprob)")
        dev = self._word_models()
        batch = PackedBatch.from_features(features)
        out = dev.score_words(batch, FP64 if self.precision == "fp64" else FP32, want_scores=True)
        if true_labels is not None:
            import torch
            from .engine import confusion_on_device
            cm, acc = confusion_on_device(torch.as_tensor(np.asarray(true_labels, dtype=np.int32)), out["best_word"], len(self.vocab), dev.ctx)
            self.last_confusion = (cm.cpu().numpy(), acc)
        bw = out["best_word"].cpu().numpy()
        words = [self.vocab[i] if i >= 0 else None for i in bw]
        return words, out["best_score"].cpu().numpy(), out["scores"].cpu().numpy()

    def decode_word_samples(self, word: str, feature_set: str = "feature_set") -> List[Dict]:
        if word not in self.vocab:
            raise ValueError(f"Word '{word}' not in vocabulary: {self.vocab}")
        results = []
        features = load_mfccs_by_word(feature_set, word)
        for i, feat_seq in enumerate(features):
            predicted_word, log_prob, state_sequence = self.decode_sequence(feat_seq.T)
            results.append({"sample_index": i + 1, "true_word": word, "predicted_word": predicted_word,
                            "log_likelihood": log_prob, "correct": predicted_word == word,
                            "state_sequence": state_sequence})
        return results

    def _batchable(self) -> bool:
        return self.implementation == "custom" and all(getattr(m, "semantics", None) == "standard" for m in self.models.values())

    def decode_vocabulary(self, feature_set: str = "feature_set", verbose: bool = True) -> Dict[str, List[Dict]]:
        """decoder.py:79-95.  Custom models with the standard (diagonal, all-frames) semantics are recognised in ONE fused
        Viterbi launch per word list instead of utterances x models calls (same result dictionaries; SAPR_DECODE_LOOP=1 keeps the
        reference's per-sequence loop).  hmmlearn models keep the per-sequence loop here; ``decode_batch`` and
        ``eval_hmm(..., batched=True)`` are their batched route."""
        import os
        batched = self._batchable() and os.environ.get("SAPR_DECODE_LOOP", "0") != "1"
        all_results = {}
        for word in self.vocab:
            if batched:
                feats = load_mfccs_by_word(feature_set, word)
                words, scores, paths = self.decode_batch(feats) if feats else ([], [], [])
                results = [{"sample_index": i + 1, "true_word": word, "predicted_word": words[i], "log_likelihood": float(scores[i]),
                            "correct": words[i] == word, "state_sequence": paths[i]} for i in range(len(feats))]
            else:
                results = self.decode_word_samples(word, feature_set)
            all_results[word] = results
            if verbose:
                correct = sum(r["correct"] for r in results)
                print(f"\nResults for '{word}':")
                print(f"Accuracy: {correct}/{len(results)} ({correct / len(results):.1%})")
        return all_results
