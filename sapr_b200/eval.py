"""Drop-in for the metrics half of assignment2/eval.py: ``extract_labels`` (eval.py:16-25),
``calculate_metrics`` (eval.py:28-38), ``log_per_word_accuracy`` (eval.py:99-105) and ``eval_hmm``
(eval.py:108-136) with the same arguments and the same result dictionary.  Decoding goes through the drop-in
``Decoder``; with ``batched=True`` (custom models trained with semantics="standard", or hmmlearn models of one shape
with up to 32 states) the whole evaluation set is recognised in ONE fused Viterbi launch instead of utterances x models
Python calls.  The default (``batched=False``) keeps the reference's per-sequence loop for both implementations.

The confusion matrix follows sklearn.metrics.confusion_matrix as eval.py:35 calls it (no ``labels=``): rows and
columns are the sorted union of the label indices that occur, so a word that is never seen nor predicted has no
row -- restated in numpy here.  Not rebuilt: ``plot_confusion_matrix`` and the PCA / training-error figures.
"""
from __future__ import annotations

import logging
from typing import Dict, List, Literal, Tuple, Union

import numpy as np
import pandas as pd

from .decoder import Decoder
from .mfcc_extract import load_mfccs_by_word


def extract_labels(all_results: Dict) -> Tuple[List[str], List[str]]:
    true_labels, predicted_labels = [], []
    for results in all_results.values():
        for result in results:
            true_labels.append(result["true_word"])
            predicted_labels.append(result["predicted_word"])
    return true_labels, predicted_labels


def calculate_metrics(true_labels: List[str], predicted_labels: List[str], vocab: List[str]) -> Tuple[np.ndarray, float]:
    label_mapping = {word: idx for idx, word in enumerate(vocab)}
    t = np.array([label_mapping[label] for label in true_labels], dtype=np.int64)
    p = np.array([label_mapping[label] for label in predicted_labels], dtype=np.int64)
    present = np.unique(np.concatenate([t, p]))
    cm = np.zeros((len(present), len(present)), dtype=np.int64)
    np.add.at(cm, (np.searchsorted(present, t), np.searchsorted(present, p)), 1)
    accuracy = float(np.mean(t == p)) if len(t) else float("nan")
    return cm, accuracy


def log_per_word_accuracy(all_results: Dict) -> None:
    logging.info("\nPer-word accuracy:")
    for word, results in all_results.items():
        word_correct = sum(r["correct"] for r in results)
        logging.info(f"{word}: {word_correct / len(results):.2%}")


def decode_vocabulary_batched(decoder: Decoder, feature_set_path: str) -> Dict[str, List[Dict]]:
    """Same result dictionary as Decoder.decode_vocabulary, one Viterbi launch for the whole set."""
    per_word = {word: load_mfccs_by_word(feature_set_path, word) for word in decoder.vocab}
    flat = [f for word in decoder.vocab for f in per_word[word]]
    truth = [i for i, word in enumerate(decoder.vocab) for _ in per_word[word]]
    words, scores, paths = decoder.decode_batch(flat, true_labels=truth) if flat else ([], [], [])
    all_results, k = {}, 0
    for word in decoder.vocab:
        res = []
        for i in range(len(per_word[word])):
            res.append({"sample_index": i + 1, "true_word": word, "predicted_word": words[k],
                        "log_likelihood": float(scores[k]), "correct": words[k] == word, "state_sequence": paths[k]})
            k += 1
        all_results[word] = res
    return all_results


def eval_hmm(implementation: Literal["custom", "hmmlearn"] = "hmmlearn", feature_set_path: str = "eval_feature_set",
             model_iter: int = 15, models_dir: str = "trained_models", vocab_order: List[str] = None,
             batched: bool = False) -> Dict[str, Union[dict, float, pd.DataFrame]]:
    decoder = Decoder(models_dir=models_dir, implementation=implementation, n_iter=model_iter, vocab_order=vocab_order)
    if batched:
        all_results = decode_vocabulary_batched(decoder, feature_set_path)
    else:
        all_results = decoder.decode_vocabulary(feature_set_path, verbose=False)
    true_labels, predicted_labels = extract_labels(all_results)
    dev_cm = getattr(decoder, "last_confusion", None) if batched else None
    if dev_cm is not None and None not in predicted_labels:
        # counts accumulated on the device (sapr_confusion); rows / columns restricted to the labels that occur, as sklearn does
        full, accuracy = dev_cm
        present_idx = np.nonzero((full[:, :-1].sum(axis=0) + full[:, :-1].sum(axis=1)) > 0)[0]
        cm = full[np.ix_(present_idx, present_idx)]
    else:
        cm, accuracy = calculate_metrics(true_labels, predicted_labels, decoder.vocab)
    present = sorted({decoder.vocab.index(w) for w in true_labels + predicted_labels})
    names = [decoder.vocab[i] for i in present]
    cm_df = pd.DataFrame(cm, index=names, columns=names)
    logging.info(f"\nConfusion Matrix:\n{cm_df}")
    logging.info(f"\nOverall Accuracy: {accuracy:.2%}")
    log_per_word_accuracy(all_results)
    return {"results": all_results, "accuracy": accuracy, "confusion_matrix": cm_df, "true_labels": true_labels,
            "predicted_labels": predicted_labels}
