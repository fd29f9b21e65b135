"""GPU parity of the whole SigLIP step (two towers + pairwise sigmoid loss + backward + Adam)
through the product's public API against the oracle and the committed golden vectors."""
import math

import numpy as np
import pytest
import torch

import common
from oracle import bv_oracle as O

pytestmark = pytest.mark.gpu


def _relerr(a, b):
  a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
  return np.abs(a - b).max() / (np.abs(b).max() + 1e-30)


@pytest.fixture(scope="module")
def tiny():
  from big_vision_b200.models.proj.image_text import two_towers
  z, tree, image, text = common.load_golden_tiny()
  model = two_towers.Model(**common.TINY)
  P = model.init(0, common.TINY_IMAGE_SHAPE, common.TINY_TEXT_SHAPE, device="cuda")
  P.load_tree(tree)
  image = torch.from_numpy(image).cuda()
  text = torch.from_numpy(text).cuda()
  return model, P, image, text, z, tree


def test_forward_embeddings_match_golden(tiny):
  model, P, image, text, z, _ = tiny
  zimg, ztxt, out = model.apply({"params": P}, image, text)
  # against the bf16-emulating oracle: only accumulation order differs
  assert _relerr(zimg.cpu().numpy(), z["bfloat16:zimg"]) < 1e-2
  assert _relerr(ztxt.cpu().numpy(), z["bfloat16:ztxt"]) < 1e-2
  # against the float64 model: bf16 matmul tolerance
  assert _relerr(zimg.cpu().numpy(), z["float32:zimg"]) < 4e-2
  assert _relerr(ztxt.cpu().numpy(), z["float32:ztxt"]) < 4e-2
  assert float(out["t"]) == pytest.approx(10.0, rel=1e-6) and float(out["b"]) == -10.0
  assert np.allclose(np.linalg.norm(zimg.cpu().numpy(), axis=1), 1.0, atol=1e-5)


def test_loss_and_gradients_match_golden(tiny):
  from big_vision_b200.trainers.proj.image_text import siglip
  model, P, image, text, z, _ = tiny
  loss, aux = siglip.loss_and_grads(model, P, image, text)
  assert float(loss) == pytest.approx(float(z["bfloat16:loss"]), rel=2e-3)
  assert float(loss) == pytest.approx(float(z["float32:loss"]), rel=5e-3)
  grads = P.numpy_tree("g")
  gn = math.sqrt(sum(float((g.astype(np.float64) ** 2).sum()) for g in grads.values()))
  assert gn == pytest.approx(float(z["bfloat16:gradnorm"]), rel=3e-2)
  # per-tensor error relative to that tensor's scale, with an absolute floor tied to the largest
  # gradient in the model: some gradients are exactly zero in exact arithmetic (key/bias: softmax
  # is invariant to a per-query constant), so a purely relative test is meaningless for them.
  gmax = max(float(np.abs(z["float32:grad:" + k]).max()) for k in grads)
  bad = {}
  for k, g in grads.items():
    ref = z["float32:grad:" + k].astype(np.float64)
    err = float(np.abs(g.astype(np.float64) - ref).max())
    tol = 6e-2 * float(np.abs(ref).max()) + 2e-3 * gmax
    if err > tol:
      bad[k] = (err, tol)
  assert not bad, f"gradient mismatch (abs err, tol): {sorted(bad.items(), key=lambda kv: -kv[1][0])[:8]}"


def test_softmax_clip_loss_and_gradients_match_oracle(tiny):
  """config.loss_fn="softmax" (_deprecated_contrastive.py:80-101, 322-331): bidirectional InfoNCE
  through both towers against autograd through the fp64 oracle."""
  from big_vision_b200.trainers.proj.image_text import siglip
  model, P, image, text, z, tree = tiny
  loss, aux = siglip.loss_and_grads(model, P, image, text, loss_fn="softmax")
  p64 = O.to_f64_tree(tree, requires_grad=True)
  zi, zt, ex = O.two_towers_forward(p64, image.cpu(), text.cpu(), common.oracle_cfg(common.TINY), "float32")
  ref, acc = O.softmax_contrastive_loss(zi, zt, ex["t"])
  ref.backward()
  assert float(loss) == pytest.approx(float(ref), rel=5e-3)
  grads = P.numpy_tree("g")
  gmax = max(float(v.grad.abs().max()) for v in p64.values() if v.grad is not None)
  bad = {}
  for k, g in grads.items():
    r = p64[k].grad.numpy() if p64[k].grad is not None else np.zeros_like(g)
    err = float(np.abs(g.astype(np.float64) - r).max())
    tol = 6e-2 * float(np.abs(r).max()) + 3e-3 * gmax
    if err > tol:
      bad[k] = (err, tol)
  assert not bad, sorted(bad.items(), key=lambda kv: -kv[1][0])[:8]
  assert float(np.abs(grads["b"]).max()) == 0.0          # the softmax loss has no bias term


@pytest.mark.parametrize("pool", ["first", "mean", "max", "map"])
def test_text_tower_pooling_variants(pool):
  """text_transformer.py:82-93: every pooling the reference's text tower offers, through the whole
  two-tower loss against autograd through the fp64 oracle ("last" is the golden-vector case above)."""
  from big_vision_b200.models.proj.image_text import two_towers
  from big_vision_b200.trainers.proj.image_text import siglip
  kw = dict(common.TINY, text=dict(common.TINY["text"], pool_type=pool))
  model = two_towers.Model(**kw)
  P = model.init(3, common.TINY_IMAGE_SHAPE, common.TINY_TEXT_SHAPE, device="cuda")
  tree = P.numpy_tree("f")
  image, text = common.synthetic_batch(common.TINY_IMAGE_SHAPE, common.TINY_TEXT_SHAPE, 64, seed=4)
  loss, aux = siglip.loss_and_grads(model, P, torch.from_numpy(image).cuda(), torch.from_numpy(text).cuda())
  p64 = O.to_f64_tree(tree, requires_grad=True)
  zi, zt, ex = O.two_towers_forward(p64, torch.from_numpy(image), torch.from_numpy(text), common.oracle_cfg(kw),
                                    "float32")
  ref = O.siglip_loss(zi, zt, ex["t"], ex["b"])
  ref = ref[0] if isinstance(ref, tuple) else ref
  ref.backward()
  assert float(loss) == pytest.approx(float(ref), rel=5e-3)
  grads = P.numpy_tree("g")
  assert any(k.startswith("txt/MAPHead_0/") for k in grads) == (pool == "map")
  gmax = max(float(v.grad.abs().max()) for v in p64.values() if v.grad is not None)
  bad = {}
  for k, g in grads.items():
    r = p64[k].grad.numpy() if p64[k].grad is not None else np.zeros_like(g)
    err = float(np.abs(g.astype(np.float64) - r).max())
    tol = 6e-2 * float(np.abs(r).max()) + 3e-3 * gmax
    if err > tol:
      bad[k] = (err, tol)
  assert not bad, sorted(bad.items(), key=lambda kv: -kv[1][0])[:8]


def test_loss_gradient_is_consistent_with_finite_difference(tiny):
  """d loss / d t' and d loss / d b from the kernels vs a central difference of the kernel loss."""
  from big_vision_b200.trainers.proj.image_text import siglip
  model, P, image, text, _, tree = tiny
  P.load_tree(tree)
  siglip.loss_and_grads(model, P, image, text)
  gt, gb = float(P.g("t")[0]), float(P.g("b")[0])
  eps = 1e-2
  vals = {}
  for name in ("t", "b"):
    for sgn in (+1, -1):
      P.load_tree(tree)
      P.f(name).add_(sgn * eps)
      l, _ = siglip.loss_and_grads(model, P, image, text)
      vals[(name, sgn)] = float(l)
  P.load_tree(tree)
  assert (vals[("t", 1)] - vals[("t", -1)]) / (2 * eps) == pytest.approx(gt, rel=2e-2, abs=1e-4)
  assert (vals[("b", 1)] - vals[("b", -1)]) / (2 * eps) == pytest.approx(gb, rel=2e-2, abs=1e-4)


def test_update_fn_decreases_loss_and_reports_measurements(tiny):
  from big_vision_b200 import optax as bv_optax
  from big_vision_b200.trainers.proj.image_text import siglip
  model, P, image, text, _, tree = tiny
  P.load_tree(tree)
  config = dict(optax_name="scale_by_adam", optax=dict(b2=0.95, mu_dtype="bfloat16"), lr=1e-3, wd=1e-4,
                grad_clip_norm=1.0, schedule=dict(decay_type="cosine", warmup_steps=0))
  tx, _ = bv_optax.make(config, P, sched_kw=dict(total_steps=100, batch_size=8, data_size=1000))
  state = {"params": P, "opt": tx.init(P)}
  update_fn = siglip.make_update_fn(model, tx, config)
  losses = []
  for _ in range(8):
    state, m = update_fn(state, None, {"image": image, "labels": text})
    losses.append(float(m["training_loss"]))
    assert all(math.isfinite(float(m[k])) for k in ("l2_grads", "l2_params", "l2_updates"))
  assert losses[-1] < losses[0]
  assert state["opt"]["count"] == 8
  assert torch.equal(P.half.float(), P.flat.bfloat16().float())    # bf16 shadow tracks the master copy
  P.load_tree(tree)
