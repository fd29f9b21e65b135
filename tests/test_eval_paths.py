"""Integer evaluation paths (SURVEY 8f rank 2).

CPU: the oracle restatement against (a) the reference's own known-answer tables
(image_text_retrieval_test.py:26-81, which contain ties) and (b) golden vectors produced by
running the reference's numpy code here (tests/golden/make_retrieval_golden.py).
GPU: the kernels, through the C ABI and the mirrored evaluator modules, against the same tables,
the golden vectors and the oracle on seeded random inputs -- bit-exact (integers; recalls are
float64 means of booleans)."""
import os

import numpy as np
import pytest

from oracle import bv_oracle as O

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "retrieval.npz")
CORR8 = [0, 0, 1, 1, 2, 2, 3, 3]
# (dist matrix, expected image->text, expected text->image or None), image_text_retrieval_test.py:26-81
M_PERFECT = np.array([[0.0, 0.0, 0.1, 0.5, 0.1, 0.2, 0.5, 0.1],
                      [0.5, 0.4, 0.0, 0.0, 0.4, 0.2, 0.6, 0.4],
                      [0.5, 0.4, 0.1, 0.5, 0.0, 0.0, 0.8, 0.3],
                      [0.5, 0.4, 0.1, 0.5, 0.3, 0.2, 0.0, 0.0]])
M_I2T = np.array([[0.8, 0.8, 0.1, 0.5, 0.1, 0.2, 0.5, 0.1],
                  [0.5, 0.4, 0.0, 0.0, 0.4, 0.2, 0.6, 0.4],
                  [0.5, 0.4, 0.1, 0.5, 0.0, 0.8, 0.8, 0.3],
                  [0.5, 0.4, 0.1, 0.5, 0.4, 0.2, 0.3, 0.3]])
M_T2I = np.array([[0.8, 0.8, 0.1, 0.5, 0.1, 0.2, 0.1, 0.1],
                  [0.5, 0.4, 0.0, 0.0, 0.4, 0.2, 0.6, 0.4],
                  [0.5, 0.4, 0.1, 0.5, 0.0, 0.8, 0.8, 0.3],
                  [0.5, 0.4, 0.1, 0.5, 0.4, 0.2, 0.3, 0.3]])
ALL1 = {"Recall@1": 1.0, "Recall@5": 1.0, "Recall@10": 1.0}
KNOWN_I2T = [(M_PERFECT, ALL1), (M_I2T, {"Recall@1": 0.5, "Recall@5": 0.75, "Recall@10": 1.0})]
KNOWN_T2I = [(M_PERFECT, ALL1), (M_T2I, {"Recall@1": 0.375, "Recall@5": 1.0, "Recall@10": 1.0})]


def _gold_cases():
  g = np.load(GOLD)
  for name in ("a", "b", "c"):
    rank = g[f"{name}_rank"]
    dist = (rank.astype(np.float64) * (2.0 / rank.size)).astype(np.float32)   # the matrix the reference ran on
    yield name, dist, g[f"{name}_corr"], g[f"{name}_t2i"], g[f"{name}_i2t"]


def _vec(d):
  return np.array([d[f"Recall@{k}"] for k in (1, 5, 10)], np.float64)


# ------------------------------------------------------------------------------------ CPU: oracle pins
def test_oracle_matches_reference_known_answers():
  for m, exp in KNOWN_I2T:
    assert O.retrieval_recalls(m, CORR8)[1] == exp
  for m, exp in KNOWN_T2I:
    assert O.retrieval_recalls(m, CORR8)[0] == exp


def test_oracle_matches_reference_generated_golden():
  for name, d, corr, t2i, i2t in _gold_cases():
    got_t2i, got_i2t = O.retrieval_recalls(d, corr)
    assert np.array_equal(_vec(got_t2i), t2i), name
    assert np.array_equal(_vec(got_i2t), i2t), name


def test_oracle_top1_first_index_and_mask():
  logits = np.array([[1., 3., 3., 0.], [2., 2., 2., 2.], [0., -1., 5., 5.], [9., 0., 0., 0.]])
  labels = np.array([[0., 1., 0., 0.], [0., 1., 0., 0.], [0., 0., 0., 1.], [0., 0., 0., 0.]])
  nc, ns, idx = O.top1_counts(logits, labels, mask=[1., 1., 1., 1.])
  assert idx.tolist() == [1, 0, 2, 0]          # ties -> first index
  assert (nc, ns) == (1.0, 3.0)                # row 3 has all-zero labels: not counted


# ------------------------------------------------------------------------------------ GPU: kernels
@pytest.mark.gpu
def test_retrieval_known_answers_on_device():
  from big_vision_b200.evaluators.proj.image_text import image_text_retrieval as ev
  for m, exp in KNOWN_I2T:
    assert ev.image_to_text_retrieval_eval(m, CORR8) == exp
  for m, exp in KNOWN_T2I:
    assert ev.text_to_image_retrieval_eval(m, CORR8) == exp


@pytest.mark.gpu
def test_retrieval_golden_on_device():
  from big_vision_b200.evaluators.proj.image_text import image_text_retrieval as ev
  for name, d, corr, t2i, i2t in _gold_cases():
    assert np.array_equal(_vec(ev.text_to_image_retrieval_eval(d, list(corr))), t2i), name
    assert np.array_equal(_vec(ev.image_to_text_retrieval_eval(d, list(corr))), i2t), name


@pytest.mark.gpu
@pytest.mark.parametrize("ni,nt,levels", [(7, 3, 0), (64, 200, 0), (33, 1000, 5), (257, 257, 3), (1, 40, 2)])
def test_retrieval_ranks_match_stable_argsort(ni, nt, levels):
  """Ranks (not only recalls) against a stable argsort, with heavy ties when levels > 0, images
  without any text and ragged sizes."""
  import torch
  from big_vision_b200 import ops
  rng = np.random.default_rng(ni * 1000 + nt)
  d = rng.random((ni, nt)).astype(np.float32)
  if levels:
    d = np.round(d * levels) / levels
  corr = rng.integers(0, ni, nt).astype(np.int32)
  r_t2i, r_i2t = ops.retrieval_ranks(torch.from_numpy(d).cuda(), torch.from_numpy(corr))
  order0 = d.argsort(axis=0, kind="stable")
  exp_t2i = np.array([int(np.nonzero(order0[:, j] == corr[j])[0][0]) for j in range(nt)])
  order1 = d.argsort(axis=1, kind="stable")
  exp_i2t = []
  for i in range(ni):
    pos = np.nonzero(corr[order1[i]] == i)[0]
    exp_i2t.append(int(pos[0]) if len(pos) else 2 ** 31 - 1)
  assert np.array_equal(r_t2i.cpu().numpy(), exp_t2i)
  assert np.array_equal(r_i2t.cpu().numpy(), np.array(exp_i2t))


@pytest.mark.gpu
@pytest.mark.parametrize("rows,C,dtype", [(5, 3, "f32"), (1000, 1000, "f32"), (257, 31, "bf16"), (64, 4097, "f32")])
def test_top1_matches_oracle(rows, C, dtype):
  import torch
  from big_vision_b200.evaluators import classification
  rng = np.random.default_rng(rows + C)
  logits = np.round(rng.standard_normal((rows, C)) * 4).astype(np.float32) / 4     # many exact ties
  labels = np.zeros((rows, C), np.float32)
  labels[np.arange(rows), rng.integers(0, C, rows)] = 1.0
  labels[::7] = 0.0                                                                # unlabeled rows
  mask = (rng.random(rows) < 0.9).astype(np.float32)
  t = torch.from_numpy(logits).cuda()
  if dtype == "bf16":
    t = t.bfloat16()            # quarter-integers are exact in bf16 at this range
  nc, ns, idx = classification.top1_counts(t, torch.from_numpy(labels).cuda(), torch.from_numpy(mask).cuda())
  enc, ens, eidx = O.top1_counts(t.float().cpu().numpy(), labels, mask)
  assert np.array_equal(idx.cpu().numpy(), eidx)
  assert (nc, ns) == (enc, ens)


@pytest.mark.gpu
def test_top1_nan_and_zero_shot():
  import torch
  from big_vision_b200 import ops
  from big_vision_b200.evaluators import classification
  x = torch.tensor([[0., float("nan"), 5., float("nan")], [float("-inf")] * 4, [1., 2., 3., float("inf")]]).cuda()
  idx, _, _ = ops.top1(x)
  assert idx.cpu().tolist() == [1, 0, 3]       # first NaN wins, as jnp.argmax; all -inf -> 0
  g = torch.Generator().manual_seed(0)
  zi = torch.nn.functional.normalize(torch.randn(300, 64, generator=g), dim=1).bfloat16()
  zt = torch.nn.functional.normalize(torch.randn(40, 64, generator=g), dim=1).bfloat16()
  best = classification.zero_shot_best_text(zi.cuda(), zt.cuda())
  scores = zi.double() @ zt.double().T       # bf16 inputs, exact products, fp32 accumulate on device
  top2 = scores.topk(2, dim=1).values
  clear = (top2[:, 0] - top2[:, 1]) > 1e-4     # rows whose winner is not an fp32-rounding coin flip
  assert clear.sum() > 250
  assert torch.equal(best.cpu().long()[clear], scores.argmax(dim=1)[clear])
