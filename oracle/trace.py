"""Compact recordings of a greedy decode's logits, for parity checks against outputs stored under tests/golden/.

A full vocabulary of logits per step is too large to keep in the repository, so each step keeps: the greedy id, max|logits|
(the denominator of the relative error), the TOP largest logits with their ids, and the logits at SAMPLE fixed, seeded
positions.  rel_err() is max|ours - recorded| / max|recorded| over the kept positions.
"""
from __future__ import annotations

import numpy as np

TOP, SAMPLE = 16, 48


def sample_ids(vocab: int) -> np.ndarray:
    return np.sort(np.random.default_rng(vocab).choice(vocab, size=min(SAMPLE, vocab), replace=False)).astype(np.int32)


class Recorder:
    def __init__(self, vocab: int):
        self.sample = sample_ids(vocab)
        self.steps: list[tuple] = []

    def add(self, logits: np.ndarray) -> None:
        top = np.argpartition(logits, -TOP)[-TOP:].astype(np.int32)
        self.steps.append((int(np.argmax(logits)), float(np.abs(logits).max()), top, logits[top], logits[self.sample]))

    def arrays(self) -> dict:
        ids, absmax, top, top_val, val = zip(*self.steps)
        return {"ids": np.array(ids, np.int32), "absmax": np.array(absmax, np.float32), "top": np.stack(top),
                "top_val": np.stack(top_val).astype(np.float32), "sample": self.sample,
                "sample_val": np.stack(val).astype(np.float32)}


class Trace:
    """A recording made by Recorder, read back step by step."""

    def __init__(self, arrays):
        self.a = {k: np.asarray(arrays[k]) for k in arrays}

    def __len__(self) -> int:
        return len(self.a["ids"])

    def greedy(self, step: int) -> int:
        return int(self.a["ids"][step])

    def rel_err(self, step: int, logits: np.ndarray) -> float:
        a = self.a
        d = max(np.abs(logits[a["top"][step]] - a["top_val"][step]).max(), np.abs(logits[a["sample"]] - a["sample_val"][step]).max())
        return float(d / a["absmax"][step])
