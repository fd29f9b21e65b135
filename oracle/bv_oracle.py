"""ORACLE -- TEST INFRASTRUCTURE ONLY.  Never imported by the product path (big_vision_b200/).

CPU restatement of the reference's algorithm for the SigLIP / ViT / MLP-Mixer hot path, in
torch-CPU float64 with autograd providing the reference gradients.  Only `tests/`,
`__graft_entry__.smoke()` and `bench.py`'s cpu_baseline / `--impl reference` legs may use it.

PARITY UNPINNED: the reference's arithmetic lives in un-vendored, un-pinned flax / jax
(requirements.txt:7-8), neither of which is installed here or on the GPU box (probed:
`import jax` -> ModuleNotFoundError on both), and the reference's own tests hold no golden
vectors for this path (SURVEY.md 8c).  What pins this file instead:
  * every function cites the reference lines it restates;
  * the flax-internal semantics it encodes are the documented defaults (LayerNorm eps=1e-6 with
    fast variance, tanh-approximate gelu, q scaled by 1/sqrt(dh) before the dot, softmax over
    keys, DenseGeneral kernel shapes) and are cross-checked in tests/test_oracle.py against
    torch.nn.functional's independent implementations of the same operators;
  * the global loss (siglip.py:287-306) is checked against the explicit per-device form
    (_deprecated_contrastive.py:117-141) -- two restatements of one quantity must agree;
  * WHOLE-MODEL pin against code this file shares nothing with (tests/test_oracle_hf_pin.py): the
    `transformers` package in the image carries SiglipModel -- whose conversion script validates it
    against the reference's released SigLIP checkpoints -- and ViTForImageClassification, the PyTorch
    port of the original ViT.  One random parameter tree mapped into both gives, in float64, the same
    image / text embeddings (1e-7, the difference being the reference's +1e-8 in the normalisation),
    logits, loss and parameter gradients (1e-6 relative) for the two-tower model with MAP head and
    last-token text pooling, and the same logits (1e-9), softmax / sigmoid cross-entropies and gradients
    (1e-8) for the cls-token classifier; the committed golden vectors the GPU tests use
    (tests/golden/siglip_tiny.npz) are reproduced by SiglipModel from the parameters and inputs whose
    digests the file stores.  This is not the reference itself, so the "unpinned" label
    stays; it does pin every flax default listed above plus the [d, h, dh] head split, the MAP head,
    the class-token / position-embedding order and both losses against an implementation that
    reproduces the reference's checkpoints.  Not covered by it: MLP-Mixer, sincos2d, gap / "0" pooling,
    the tanh pre_logits layer (torch cross-checks and source citations only).

`mm="bfloat16"` emulates the CUDA path's rounding points (bf16 matmul operands / outputs and
a bf16 residual stream, fp32-or-better everywhere else) with straight-through gradients, so
forward parity can be asserted tightly; `mm="float32"` is the plain high-precision model.
"""
import math

import numpy as np
import torch

F64 = torch.float64


# --------------------------------------------------------------------------------------------
# numerics helpers
# --------------------------------------------------------------------------------------------
class _RoundBf16(torch.autograd.Function):
  @staticmethod
  def forward(ctx, x):
    return x.to(torch.float32).to(torch.bfloat16).to(x.dtype)

  @staticmethod
  def backward(ctx, g):
    return g


def rnd(x, mm):
  """Round to bf16 (straight-through) when emulating the bf16 matmul path."""
  return _RoundBf16.apply(x) if mm == "bfloat16" else x


def gelu_tanh(x):
  """flax.linen.gelu default (approximate=True), called at models/vit.py:75, mlp_mixer.py:36."""
  return 0.5 * x * (1.0 + torch.tanh(math.sqrt(2.0 / math.pi) * (x + 0.044715 * x ** 3)))


def layer_norm(x, scale, bias, eps=1e-6):
  """flax.linen.LayerNorm defaults (models/vit.py:92,103,160,181): eps 1e-6, stats over the last
  axis, use_fast_variance: var = max(E[x^2] - E[x]^2, 0)."""
  mean = x.mean(-1, keepdim=True)
  var = torch.clamp((x * x).mean(-1, keepdim=True) - mean * mean, min=0.0)
  return (x - mean) * torch.rsqrt(var + eps) * scale + bias


def dense(x, kernel, bias, mm):
  """flax nn.Dense(dtype=mm): y = x @ kernel + bias, operands cast to mm, fp32 accumulate."""
  y = rnd(x, mm) @ rnd(kernel, mm)
  return y + bias if bias is not None else y


def mha(xq, xkv, p, heads, mm):
  """flax.linen.MultiHeadDotProductAttention (models/vit.py:93-98,176-178).
  p: query/key/value {kernel [d,h,dh], bias [h,dh]}, out {kernel [h,dh,d], bias [d]}.
  query is scaled by 1/sqrt(dh) before the dot; softmax over keys; no mask, no dropout."""
  d = xq.shape[-1]
  dh = d // heads

  def proj(x, name):
    k = p[name + "/kernel"].reshape(d, d)
    b = p[name + "/bias"].reshape(d)
    return rnd(dense(x, k, b, mm), mm)

  q, k, v = proj(xq, "query"), proj(xkv, "key"), proj(xkv, "value")
  B, Nq, Nk = xq.shape[0], xq.shape[1], xkv.shape[1]
  q = q.reshape(B, Nq, heads, dh).transpose(1, 2)
  k = k.reshape(B, Nk, heads, dh).transpose(1, 2)
  v = v.reshape(B, Nk, heads, dh).transpose(1, 2)
  s = (q @ k.transpose(-1, -2)) / math.sqrt(dh)
  w = torch.softmax(s, dim=-1)
  if mm == "bfloat16":
    # the kernel feeds un-normalised bf16 probabilities exp(s - max) to the tensor core and
    # divides by their fp32 sum afterwards
    e = torch.exp(s - s.max(-1, keepdim=True).values)
    o = (rnd(e, mm) @ v) / e.sum(-1, keepdim=True)
  else:
    o = w @ v
  o = rnd(o, mm).transpose(1, 2).reshape(B, Nq, d)
  return dense(o, p["out/kernel"].reshape(d, d), p["out/bias"], mm)


def sub(p, prefix):
  """Sub-tree of a flat 'a/b/c' dict."""
  n = len(prefix)
  return {k[n:]: v for k, v in p.items() if k.startswith(prefix)}


def mlp_block(x, p, mm):
  """vit.MlpBlock (models/vit.py:57-78)."""
  h = rnd(dense(x, p["Dense_0/kernel"], p["Dense_0/bias"], mm), mm)
  h = rnd(gelu_tanh(h), mm)
  return dense(h, p["Dense_1/kernel"], p["Dense_1/bias"], mm)


def encoder_block(x, p, heads, mm):
  """vit.Encoder1DBlock.__call__ (models/vit.py:89-112)."""
  y = rnd(layer_norm(x, p["LayerNorm_0/scale"], p["LayerNorm_0/bias"]), mm)
  y = rnd(mha(y, y, sub(p, "MultiHeadDotProductAttention_0/"), heads, mm), mm)
  x = rnd(x + y, mm)
  y = rnd(layer_norm(x, p["LayerNorm_1/scale"], p["LayerNorm_1/bias"]), mm)
  y = rnd(mlp_block(y, sub(p, "MlpBlock_0/"), mm), mm)
  return rnd(x + y, mm)


def encoder(x, p, depth, heads, mm):
  """vit.Encoder (models/vit.py:115-160), scan=False naming; returns the PRE-norm stream and
  the encoder_norm output."""
  for i in range(depth):
    x = encoder_block(x, sub(p, f"encoderblock_{i}/"), heads, mm)
  return layer_norm(x, p["encoder_norm/scale"], p["encoder_norm/bias"])


def map_head(x, p, heads, mm):
  """vit.MAPHead (models/vit.py:163-183)."""
  n = x.shape[0]
  probe = p["probe"].expand(n, -1, -1)
  a = rnd(mha(probe, rnd(x, mm), sub(p, "MultiHeadDotProductAttention_0/"), heads, mm), mm)
  y = rnd(layer_norm(a, p["LayerNorm_0/scale"], p["LayerNorm_0/bias"]), mm)
  out = a + mlp_block(y, sub(p, "MlpBlock_0/"), mm)
  return out[:, 0]


def posemb_sincos_2d(h, w, width, temperature=10_000.0):
  """models/vit.py:34-44."""
  y, x = np.mgrid[:h, :w]
  omega = np.arange(width // 4) / (width // 4 - 1)
  omega = 1.0 / (temperature ** omega)
  y = np.einsum("m,d->md", y.flatten(), omega)
  x = np.einsum("m,d->md", x.flatten(), omega)
  return np.concatenate([np.sin(x), np.cos(x), np.sin(y), np.cos(y)], axis=1)[None]


def patch_embed(image, kernel, bias, mm):
  """nn.Conv(width, patch, strides=patch, padding="VALID") (models/vit.py:212-214) followed by
  the reshape of :216-217.  kernel [ph,pw,C,width] HWIO, image NHWC."""
  ph, pw, C, width = kernel.shape
  n, H, W, _ = image.shape
  x = image.reshape(n, H // ph, ph, W // pw, pw, C).permute(0, 1, 3, 2, 4, 5)
  x = x.reshape(n, (H // ph) * (W // pw), ph * pw * C)
  return dense(x, kernel.reshape(ph * pw * C, width), bias, mm)


def vit_forward(p, image, cfg, mm="float32"):
  """vit._Model.__call__ (models/vit.py:206-276).  cfg: dict(depth, num_heads, pool_type,
  posemb, rep_size, num_classes).  p: flat dict of float64 tensors with the reference names."""
  image = image.to(F64)
  x = rnd(patch_embed(image, p["embedding/kernel"], p["embedding/bias"], mm), mm)
  n, N0, d = x.shape
  if cfg.get("posemb", "learn") == "learn":
    pe = p["pos_embedding"]
  else:
    ph, pw = p["embedding/kernel"].shape[:2]
    pe = torch.from_numpy(posemb_sincos_2d(image.shape[1] // ph, image.shape[2] // pw, d)).to(F64)
  x = rnd(x + rnd(pe, mm), mm)
  if cfg["pool_type"] == "tok":
    x = torch.cat([rnd(p["cls"], mm).expand(n, -1, -1), x], dim=1)
  x = encoder(x, sub(p, "Transformer/"), cfg["depth"], cfg["num_heads"], mm)
  if cfg["pool_type"] == "map":
    x = map_head(x, sub(p, "MAPHead_0/"), cfg["num_heads"], mm)
  elif cfg["pool_type"] == "gap":
    x = rnd(x, mm).mean(1)
  elif cfg["pool_type"] in ("0", "tok"):
    x = x[:, 0]
  elif cfg["pool_type"] == "none":            # models/vit.py:252-253: head applied to every token
    x = rnd(x, mm)
  else:
    raise ValueError(cfg["pool_type"])
  if cfg.get("rep_size"):
    x = torch.tanh(dense(x, p["pre_logits/kernel"], p["pre_logits/bias"], mm))
  if cfg.get("num_classes"):
    x = dense(x, p["head/kernel"], p["head/bias"], mm)
  return x


def text_forward(p, text, cfg, mm="float32"):
  """text_transformer._Model.__call__ (text_transformer.py:55-99); no attention mask."""
  x = p["Embed_0/embedding"][text.long()] + p["pos_embedding"]
  x = rnd(x, mm)
  x = encoder(x, sub(p, "Encoder_0/"), cfg["depth"], cfg["num_heads"], mm)
  pool = cfg.get("pool_type", "last")
  if pool == "last":
    x = x[:, -1, :]
  elif pool == "first":
    x = x[:, 0, :]
  elif pool in ("mean", "gap"):
    x = rnd(x, mm).mean(1)
  elif pool in ("max", "gmp"):                # text_transformer.py:89-90; amax splits the cotangent
    x = torch.amax(rnd(x, mm), dim=1)         # evenly between ties, as jnp.max does
  elif pool == "map":                         # text_transformer.py:91-93
    x = map_head(x, sub(p, "MAPHead_0/"), cfg["num_heads"], mm)
  else:
    raise NotImplementedError(pool)
  if cfg.get("num_classes"):
    x = dense(rnd(x, mm), p["head/kernel"], p["head/bias"], mm)
  return x


def l2_normalize(z):
  """two_towers.py:60-61,73-74: z / (||z||_2 + 1e-8)."""
  return z / (torch.linalg.norm(z, dim=1, keepdim=True) + 1e-8)


def two_towers_forward(p, image, text, cfg, mm="float32"):
  """two_towers.Model.__call__ (two_towers.py:39-90) -> (zimg, ztxt, {"t": exp(t'), "b": b})."""
  ztxt = l2_normalize(text_forward(sub(p, "txt/"), text, cfg["text"], mm))
  zimg = l2_normalize(vit_forward(sub(p, "img/"), image, cfg["image"], mm))
  return zimg, ztxt, {"t": torch.exp(p["t"]), "b": p.get("b")}


def siglip_loss(zimg, ztxt, t, b):
  """loss_fn of trainers/proj/image_text/siglip.py:287-308 (GLOBAL batch)."""
  logits = zimg @ ztxt.T
  logits = logits * t + (b if b is not None else 0.0)
  eye = torch.eye(zimg.shape[0], dtype=logits.dtype)
  m1_diag1 = -torch.ones_like(logits) + 2 * eye
  loglik = torch.nn.functional.logsigmoid(m1_diag1 * logits)
  nll = -loglik.sum(-1)
  return nll.mean()


def siglip_loss_per_device(zimg, ztxt, t, b, world):
  """sigmoid_loss of _deprecated_contrastive.py:117-141 evaluated for every "device" of a
  world-size split, then pmean-ed (:343): must equal siglip_loss on the global batch."""
  B = zimg.shape[0]
  n = B // world
  total = 0.0
  for r in range(world):
    zi = zimg[r * n:(r + 1) * n]
    zt_me = ztxt[r * n:(r + 1) * n]
    zt_ot = torch.cat([ztxt[:r * n], ztxt[(r + 1) * n:]], 0)
    bb = b if b is not None else 0.0
    logits_me = zi @ zt_me.T * t + bb
    logits_ot = zi @ zt_ot.T * t + bb
    eye = torch.eye(n, dtype=zi.dtype)
    ll_me = torch.nn.functional.logsigmoid((-torch.ones_like(logits_me) + 2 * eye) * logits_me)
    ll_ot = torch.nn.functional.logsigmoid(-logits_ot)
    total = total + (-ll_me.sum(-1)).mean() + (-ll_ot.sum(-1)).mean()
  return total / world


def softmax_contrastive_loss(zimg, ztxt, t):
  """`softmax_loss` (CLIP), trainers/proj/image_text/_deprecated_contrastive.py:80-101, on the GLOBAL
  batch: 0.5 * (mean_i -log_softmax(zimg ztxt^T t, axis=1)_ii + mean_i -log_softmax(..., axis=0)_ii);
  also the two retrieval accuracies (argmax == diagonal, :89).  t is exp(t')."""
  logits = zimg @ ztxt.T * t
  idx = torch.arange(logits.shape[0])
  l1 = -(torch.log_softmax(logits, dim=1)[idx, idx]).mean()
  l2 = -(torch.log_softmax(logits, dim=0)[idx, idx]).mean()
  acc = ((logits.argmax(1) == idx).double().mean(), (logits.argmax(0) == idx).double().mean())
  return 0.5 * (l1 + l2), acc


def sigmoid_xent(logits, labels):
  """utils.py:236-243."""
  log_p = torch.nn.functional.logsigmoid(logits)
  log_not_p = torch.nn.functional.logsigmoid(-logits)
  return (-(labels * log_p + (1.0 - labels) * log_not_p).sum(-1)).mean()


def softmax_xent(logits, labels):
  """utils.py:276-281."""
  return (-(labels * torch.log_softmax(logits, -1)).sum(-1)).mean()


def mixer_forward(p, image, cfg, mm="float32", masks=None):
  """mlp_mixer.MlpMixer.__call__ (models/mlp_mixer.py:70-84).  `masks` [num_blocks, 2, n] are the
  per-sample stochastic-depth masks 1 - Bernoulli(drop_p) of mlp_mixer.py:173-177 (None = all ones,
  i.e. stoch_depth = 0 or eval mode); the residual adds are `x + y * mask` (:52,:55), no rescale."""
  image = image.to(F64)
  x = rnd(patch_embed(image, p["stem/kernel"], p["stem/bias"], mm), mm)
  for i in range(cfg["num_blocks"]):
    bp = sub(p, f"MixerBlock_{i}/")
    y = rnd(layer_norm(x, bp["LayerNorm_0/scale"], bp["LayerNorm_0/bias"]), mm)
    y = y.transpose(1, 2)
    tm = sub(bp, "token_mixing/")
    h = rnd(gelu_tanh(rnd(dense(y, tm["Dense_0/kernel"], tm["Dense_0/bias"], mm), mm)), mm)
    y = rnd(dense(h, tm["Dense_1/kernel"], tm["Dense_1/bias"], mm), mm).transpose(1, 2)
    if masks is not None:
      y = y * torch.as_tensor(masks[i][0]).to(F64)[:, None, None]
    x = rnd(x + y, mm)
    y = rnd(layer_norm(x, bp["LayerNorm_1/scale"], bp["LayerNorm_1/bias"]), mm)
    cm = sub(bp, "channel_mixing/")
    h = rnd(gelu_tanh(rnd(dense(y, cm["Dense_0/kernel"], cm["Dense_0/bias"], mm), mm)), mm)
    y = rnd(dense(h, cm["Dense_1/kernel"], cm["Dense_1/bias"], mm), mm)
    if masks is not None:
      y = y * torch.as_tensor(masks[i][1]).to(F64)[:, None, None]
    x = rnd(x + y, mm)
  x = layer_norm(x, p["pre_head_layer_norm/scale"], p["pre_head_layer_norm/bias"])
  x = x.mean(1)
  if cfg.get("num_classes"):
    x = dense(x, p["head/kernel"], p["head/bias"], mm)
  return x


# --------------------------------------------------------------------------------------------
# driver helpers for the tests / smoke / cpu baseline
# --------------------------------------------------------------------------------------------
def to_f64_tree(np_tree, requires_grad=False):
  return {k: torch.tensor(np.asarray(v), dtype=F64, requires_grad=requires_grad)
          for k, v in np_tree.items()}


def siglip_value_and_grad(np_tree, image, text, cfg, mm="float32"):
  """jax.value_and_grad(loss_fn)(params) of siglip.py:311 on the global batch."""
  p = to_f64_tree(np_tree, requires_grad=True)
  zimg, ztxt, extras = two_towers_forward(p, torch.as_tensor(image), torch.as_tensor(text), cfg, mm)
  loss = siglip_loss(zimg, ztxt, extras["t"], extras["b"])
  loss.backward()
  grads = {k: (v.grad.numpy() if v.grad is not None else np.zeros(v.shape)) for k, v in p.items()}
  return float(loss.detach()), grads, zimg.detach().numpy(), ztxt.detach().numpy()


def adam_reference(p, g, m, v, step, *, lr, b1, b2, eps, wd, sched=1.0, clip=0.0, gnorm=None):
  """optax chain of optax.py:143-149 for one tensor (numpy, float64)."""
  if clip and gnorm is not None and not gnorm < clip:
    g = g / gnorm * clip
  m = b1 * m + (1 - b1) * g
  v = b2 * v + (1 - b2) * g * g
  mhat = m / (1 - b1 ** step)
  vhat = v / (1 - b2 ** step)
  upd = -sched * (lr * mhat / (np.sqrt(vhat) + eps) + wd * p)
  return p + upd, m, v


def adafactor_reference(p, g, state, count, *, lr, wd=0.0, sched=1.0, min_dim_size_to_factor=32,
                        decay_rate=0.8, decay_offset=0, beta2_cap=0.999, momentum=0.9, eps=1e-30):
  """`big_vision.scale_by_adafactor` (optax.py:187-214) inside the chain of optax.py:143-149 for ONE
  tensor, numpy float64 (momentum accumulator rounded to bf16 like `dtype_momentum`).  The factored
  second moment is optax's `scale_by_factored_rms` (optax is an un-vendored, un-pinned dependency of
  the reference, requirements.txt:8; restated from its published algorithm, `_factored_dims` /
  `_update` of optax/_src/factorized.py):
    d1, d0 = the second-largest and largest axes (np.argsort), factored iff shape[d1] >= min_dim_size
    v_row = ema(mean_{d0}(g^2 + eps)), v_col = ema(mean_{d1}(g^2 + eps)), decay_t = min(cap, 1 - (t+1)^-0.8)
    u = g * (v_row / mean_{d1}(v_row))^-1/2 [expanded at d0] * v_col^-1/2 [expanded at d1]
  `state` is a dict (empty on the first call); returns (new_p, new_state)."""
  g = np.asarray(g, np.float64)
  t = np.float32(count - decay_offset) + np.float32(1.0)
  decay = float(min(np.float32(beta2_cap), np.float32(1.0) - t ** np.float32(-decay_rate)))
  shape = g.shape
  order = np.argsort(shape, kind="stable") if len(shape) else []
  st = dict(state)
  if len(shape) >= 2 and shape[order[-2]] >= min_dim_size_to_factor:
    d1, d0 = int(order[-2]), int(order[-1])
    gsq = g * g + eps
    v_row = decay * st.get("v_row", 0.0) + (1 - decay) * gsq.mean(axis=d0)
    v_col = decay * st.get("v_col", 0.0) + (1 - decay) * gsq.mean(axis=d1)
    reduced_d1 = d1 - 1 if d1 > d0 else d1
    row_col_mean = v_row.mean(axis=reduced_d1, keepdims=True)
    u = g * np.expand_dims((v_row / row_col_mean) ** -0.5, d0) * np.expand_dims(v_col ** -0.5, d1)
    st.update(v_row=v_row, v_col=v_col)
  else:
    v = decay * st.get("v", 0.0) + (1 - decay) * (g * g + eps)
    u = g * v ** -0.5
    st["v"] = v
  if momentum:
    m = momentum * st.get("m", 0.0) + (1 - momentum) * u          # optax.ema, debias=False
    st["m"] = torch.tensor(m).to(torch.float32).to(torch.bfloat16).double().numpy()   # bf16 accumulator
    u = m
  return p - sched * (lr * u + wd * p), st


# ----------------------------------------------------------------------------------------------
# Integer evaluation paths (numpy; test infrastructure like the rest of this file)
# ----------------------------------------------------------------------------------------------
def top1_counts(logits, labels, mask=None):
  """evaluators/classification.py:40-52: first-index argmax, label gather, masked counts."""
  import numpy as np
  logits = np.asarray(logits, np.float64)
  labels = np.asarray(labels, np.float64)
  mask = np.ones(len(logits)) if mask is None else np.asarray(mask, np.float64)
  mask = mask * labels.max(axis=1)
  idx = np.argmax(logits, axis=1)
  correct = np.take_along_axis(labels, idx[:, None], axis=1)[:, 0]
  return float((correct * mask).sum()), float(mask.sum()), idx.astype(np.int32)


def retrieval_recalls(dist_matrix, corr, thresholds=(1, 5, 10)):
  """evaluators/proj/image_text/image_text_retrieval.py:23-85 restated with a STABLE argsort
  (the reference calls numpy's default argsort, whose tie order is unspecified for long arrays;
  without ties the two are identical).  Returns (text->image dict, image->text dict)."""
  import numpy as np
  d = np.asarray(dist_matrix)
  corr = np.asarray(corr)
  per_text = d.argsort(axis=0, kind="stable")
  per_image = d.argsort(axis=1, kind="stable")
  t2i, i2t = {}, {}
  for k in thresholds:
    t2i[f"Recall@{k}"] = (per_text[:k, :] == corr[None]).any(axis=0).mean()
    top_k = corr[per_image[:, :k]]
    i2t[f"Recall@{k}"] = (top_k == np.arange(len(per_image))[:, None]).any(axis=1).mean()
  return t2i, i2t
