"""Drop-in for the orchestration of assignment2/train.py: ``train_hmm`` (train.py:81-124), ``save_model``
(train.py:74-78) and ``pretty_print_matrix`` (train.py:51-71), same names, arguments, file layout
(``trained_models/<impl>/<word>_<impl>_<n_iter>.pkl``) and return value.  The per-word models are the
drop-in ``HMM`` / ``HMMLearnModel`` classes, so every E-step / M-step below runs in libsaprb200.so.

Not rebuilt: ``plot_training_progress`` (train.py:16-48, matplotlib figure) -- the per-word log-likelihood
histories it would plot are returned in ``train_hmm.histories`` instead.

``batched=True`` (hmmlearn models only) fits the whole vocabulary at once with ``hmmlearn_hmm.fit_vocabulary``: one E-step over
every word's utterances per iteration instead of one per word, same pickles, return value and histories.  With ``dist`` (a
``dist.Dist``) it shards the utterances over the ranks; every rank returns the same models and histories and rank 0 alone
writes the pickles.

``semantics`` is an addition: ``"sapr"`` (default) = custom_hmm.py as written, ``"standard"`` = diagonal
Gaussian emission over all frames (SURVEY 0.1); it is forwarded to the custom ``HMM`` only.
"""
from __future__ import annotations

import logging
import pickle
from pathlib import Path
from typing import Dict, List, Literal, Union

import numpy as np
import pandas as pd

from .custom_hmm import HMM
from .hmmlearn_hmm import HMMLearnModel, fit_vocabulary
from .mfcc_extract import load_mfccs, load_mfccs_by_word

VOCABS = ["heed", "hid", "head", "had", "hard", "hud", "hod", "hoard", "hood", "whod", "heard"]   # train.py:89-92


def pretty_print_matrix(matrix: np.ndarray, precision: int = 3) -> None:
    n = matrix.shape[0]
    names = [f"S{i}" if i != 0 and i != n - 1 else ("Entry" if i == 0 else "Exit") for i in range(n)]
    df = pd.DataFrame(matrix, columns=names, index=names)
    row_sums = df.sum(axis=1).round(precision)
    df = df.replace(0, ".")
    print("\nTransition Matrix:")
    print("==================")
    print(df.round(precision))
    assert np.allclose(row_sums, 1.0), "Row sums should be equal to 1.0"


def save_model(model, model_path: Path) -> None:
    model_path = Path(model_path)
    model_path.parent.mkdir(parents=True, exist_ok=True)
    with open(model_path, "wb") as f:
        pickle.dump(model, f)
    logging.info(f"Saved model to {model_path}")


def train_hmm(implementation: Literal["custom", "hmmlearn"] = "hmmlearn", num_states: int = 8, num_features: int = 13,
              n_iter: int = 15, min_covar: float = 0.01, var_floor_factor: float = 0.001,
              feature_set_path: str = "feature_set", models_dir: str = "trained_models", vocabs: List[str] = None,
              semantics: str = "sapr", batched: bool = False, dist=None) -> Dict[str, Union[HMM, HMMLearnModel]]:
    if batched and implementation != "hmmlearn":
        raise ValueError("batched=True fits hmmlearn models; custom models train per word (engine.train_words batches them)")
    if dist is not None and not batched:
        raise ValueError("dist shards the batched fit (batched=True); the per-word loop runs in one process")
    vocabs = list(VOCABS if vocabs is None else vocabs)
    impl_dir = Path(models_dir) / implementation
    impl_dir.mkdir(parents=True, exist_ok=True)

    feature_set = load_mfccs(feature_set_path)
    features = {word: load_mfccs_by_word(feature_set_path, word) for word in vocabs}
    total_features_length = sum(len(features[word]) for word in vocabs)
    assert total_features_length == len(feature_set)

    hmms, histories = {}, {}
    if batched:
        for word in vocabs:
            hmms[word] = HMMLearnModel(num_states=num_states, model_name=word, n_iter=n_iter, min_covar=min_covar,
                                       feature_set=feature_set)
        logging.info(f"Training {len(vocabs)} hmmlearn models at once in {n_iter} iterations...")
        fit_vocabulary([hmms[w].model for w in vocabs], [features[w] for w in vocabs], dist=dist)
        for word in vocabs:
            histories[word] = list(hmms[word].model.monitor_.history)
            if dist is None or dist.rank == 0:
                save_model(hmms[word].model, impl_dir / f"{word}_{implementation}_{n_iter}.pkl")
        train_hmm.histories = histories
        return hmms
    for word in vocabs:
        logging.info(f"\nTraining model for word: {word}")
        model_path = impl_dir / f"{word}_{implementation}_{n_iter}.pkl"
        if implementation == "custom":
            hmm = HMM(num_states, num_features, feature_set, model_name=word, var_floor_factor=var_floor_factor,
                      semantics=semantics)
            log_likelihoods = hmm.baum_welch(features[word], n_iter)
            trained_model = hmm
        elif implementation == "hmmlearn":
            hmm = HMMLearnModel(num_states=num_states, model_name=word, n_iter=n_iter, min_covar=min_covar,
                                feature_set=feature_set)
            trained_model, _ = hmm.fit(features[word])
            log_likelihoods = hmm.model.monitor_.history
        else:
            raise ValueError(f"unknown implementation {implementation!r}")
        histories[word] = list(log_likelihoods)
        save_model(trained_model, model_path)
        hmms[word] = hmm
    train_hmm.histories = histories
    return hmms
