"""Generates tests/golden/retrieval.npz by RUNNING THE REFERENCE's own (numpy-only) retrieval metric
code (big_vision/evaluators/proj/image_text/image_text_retrieval.py) on seeded random distance
matrices without ties.  The tests do not need the reference: its outputs are committed.

  python tests/golden/make_retrieval_golden.py <directory holding the big_vision package>

Each matrix is stored as the rank of every distance among all distances of that matrix (uint32, which
compresses to well under 1 MB); the matrix the reference ran on is
(rank * (2 / rank.size)).astype(float32), as tests/test_eval_paths.py rebuilds it.
"""
import os
import sys

import numpy as np

if len(sys.argv) != 2:
  sys.exit(__doc__)
sys.path.insert(0, sys.argv[1])
from big_vision.evaluators.proj.image_text import image_text_retrieval as ref  # noqa: E402

out = {}
rng = np.random.default_rng(123)
for name, (ni, per) in {"a": (50, 5), "b": (333, 1), "c": (200, 5)}.items():
  nt = ni * per
  # distances = 1 - cosine of noisy copies, so the recalls are non-trivial; float32 like the device
  zi = rng.standard_normal((ni, 32)).astype(np.float32)
  corr = np.repeat(np.arange(ni), per)
  rng.shuffle(corr)
  zt = zi[corr] + 1.5 * rng.standard_normal((nt, 32)).astype(np.float32)
  zi_n = zi / np.linalg.norm(zi, axis=1, keepdims=True)
  zt_n = zt / np.linalg.norm(zt, axis=1, keepdims=True)
  d64 = 1.0 - zi_n.astype(np.float64) @ zt_n.astype(np.float64).T
  # replace every distance by its global rank scaled into [0, 2): same order, and all values are
  # distinct float32 numbers, so the reference's (unstable) argsort has a unique answer
  rank = np.empty(d64.size, np.uint32)
  rank[np.argsort(d64, axis=None, kind="stable")] = np.arange(d64.size, dtype=np.uint32)
  rank = rank.reshape(d64.shape)
  d = (rank.astype(np.float64) * (2.0 / rank.size)).astype(np.float32)
  assert len(np.unique(d)) == d.size, "ties would make the reference's argsort order ambiguous"
  t2i = ref.text_to_image_retrieval_eval(d, list(corr))
  i2t = ref.image_to_text_retrieval_eval(d, list(corr))
  out[f"{name}_rank"] = rank
  out[f"{name}_corr"] = corr.astype(np.int32)
  out[f"{name}_t2i"] = np.array([t2i[f"Recall@{k}"] for k in ref.RECALL_THRESHOLDS], np.float64)
  out[f"{name}_i2t"] = np.array([i2t[f"Recall@{k}"] for k in ref.RECALL_THRESHOLDS], np.float64)
  print(name, d.shape, t2i, i2t)
np.savez_compressed(os.path.join(os.path.dirname(os.path.abspath(__file__)), "retrieval.npz"), **out)
