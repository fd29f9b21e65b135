"""CPU: pins the oracle.  (1) its operators against torch.nn.functional's independent
implementations, (2) the global SigLIP loss against the explicit per-device form, (3) the
committed golden vectors, (4) the product's parameter tree against the reference's names."""
import math
import os

import numpy as np
import pytest
import torch

import common
from oracle import bv_oracle as O

F64 = torch.float64


def test_layer_norm_matches_torch():
  torch.manual_seed(0)
  x = torch.randn(5, 7, 64, dtype=F64) * 3 + 1
  g, b = torch.randn(64, dtype=F64), torch.randn(64, dtype=F64)
  ref = torch.nn.functional.layer_norm(x, (64,), g, b, eps=1e-6)
  assert torch.allclose(O.layer_norm(x, g, b), ref, atol=1e-10)


def test_gelu_matches_torch_tanh_approximation():
  x = torch.linspace(-6, 6, 1001, dtype=F64)
  assert torch.allclose(O.gelu_tanh(x), torch.nn.functional.gelu(x, approximate="tanh"), atol=1e-12)


def test_mha_matches_torch_sdpa():
  torch.manual_seed(1)
  B, N, d, h = 2, 9, 128, 2
  x = torch.randn(B, N, d, dtype=F64)
  p = {f"{n}/kernel": torch.randn(d, h, d // h, dtype=F64) * 0.1 for n in ("query", "key", "value")}
  p.update({f"{n}/bias": torch.randn(h, d // h, dtype=F64) * 0.1 for n in ("query", "key", "value")})
  p["out/kernel"] = torch.randn(h, d // h, d, dtype=F64) * 0.1
  p["out/bias"] = torch.randn(d, dtype=F64) * 0.1
  got = O.mha(x, x, p, h, "float32")
  q = (x @ p["query/kernel"].reshape(d, d) + p["query/bias"].reshape(d)).reshape(B, N, h, -1).transpose(1, 2)
  k = (x @ p["key/kernel"].reshape(d, d) + p["key/bias"].reshape(d)).reshape(B, N, h, -1).transpose(1, 2)
  v = (x @ p["value/kernel"].reshape(d, d) + p["value/bias"].reshape(d)).reshape(B, N, h, -1).transpose(1, 2)
  o = torch.nn.functional.scaled_dot_product_attention(q, k, v)   # scale 1/sqrt(dh), no mask
  ref = o.transpose(1, 2).reshape(B, N, d) @ p["out/kernel"].reshape(d, d) + p["out/bias"]
  assert torch.allclose(got, ref, atol=1e-9)


def test_patch_embed_matches_conv2d():
  torch.manual_seed(2)
  img = torch.randn(2, 32, 48, 3, dtype=F64)
  k = torch.randn(16, 16, 3, 8, dtype=F64)
  b = torch.randn(8, dtype=F64)
  got = O.patch_embed(img, k, b, "float32")
  ref = torch.nn.functional.conv2d(img.permute(0, 3, 1, 2), k.permute(3, 2, 0, 1), b, stride=16)
  ref = ref.permute(0, 2, 3, 1).reshape(2, -1, 8)
  assert torch.allclose(got, ref, atol=1e-9)


def test_posemb_sincos_layout():
  pe = O.posemb_sincos_2d(3, 5, 16)
  assert pe.shape == (1, 15, 16)
  # [sin x | cos x | sin y | cos y], x fastest (models/vit.py:36-43)
  assert np.allclose(pe[0, 1, 0], math.sin(1.0)) and np.allclose(pe[0, 1, 4], math.cos(1.0))
  assert np.allclose(pe[0, 5, 8], math.sin(1.0)) and np.allclose(pe[0, 1, 8], 0.0)


@pytest.mark.parametrize("world", [1, 2, 4, 8])
def test_global_loss_equals_mean_of_per_device_losses(world):
  torch.manual_seed(3)
  B, D = 16, 32
  zi = O.l2_normalize(torch.randn(B, D, dtype=F64))
  zt = O.l2_normalize(torch.randn(B, D, dtype=F64))
  t, b = torch.tensor(10.0, dtype=F64), torch.tensor(-10.0, dtype=F64)
  assert torch.allclose(O.siglip_loss(zi, zt, t, b), O.siglip_loss_per_device(zi, zt, t, b, world), atol=1e-12)


def test_classification_losses_known_answers():
  logits = torch.tensor([[0.0, 0.0], [2.0, -2.0]], dtype=F64)
  labels = torch.tensor([[1.0, 0.0], [1.0, 0.0]], dtype=F64)
  s = O.sigmoid_xent(logits, labels)
  ref = (2 * math.log(2.0) + 2 * math.log1p(math.exp(-2.0))) / 2
  assert float(s) == pytest.approx(ref, abs=1e-12)
  sm = O.softmax_xent(logits, labels)
  assert float(sm) == pytest.approx((math.log(2.0) + math.log1p(math.exp(-4.0))) / 2, abs=1e-12)


def test_adam_reference_first_step_is_sign_update():
  p, g = np.array([1.0, -2.0]), np.array([0.5, -0.25])
  p1, m, v = O.adam_reference(p, g, 0 * p, 0 * p, 1, lr=0.1, b1=0.9, b2=0.999, eps=0.0, wd=0.0)
  assert np.allclose(p1, p - 0.1 * np.sign(g))


def test_golden_vectors_reproduce():
  z, tree, image, text = common.load_golden_tiny()
  cfg = common.oracle_cfg(common.TINY)
  loss, grads, zimg, ztxt = O.siglip_value_and_grad(tree, image, text, cfg, "float32")
  assert loss == pytest.approx(float(z["float32:loss"]), rel=1e-9)
  assert np.allclose(zimg, z["float32:zimg"], atol=1e-9)
  for k in ("t", "b", "img/MAPHead_0/probe", "txt/Embed_0/embedding",
            "img/Transformer/encoderblock_0/MultiHeadDotProductAttention_0/key/kernel"):
    assert np.allclose(grads[k], z["float32:grad:" + k], rtol=1e-4, atol=1e-7), k


def test_golden_inputs_follow_the_synthetic_recipe():
  z = np.load(common.GOLDEN_TINY)
  image, text = common.synthetic_batch(common.TINY_IMAGE_SHAPE, common.TINY_TEXT_SHAPE,
                                       common.TINY["text"]["vocab_size"])
  assert common.sha256_of({"image": image}) == str(z["image_sha256"]) and np.array_equal(text, z["text"])
  assert (text[:, -1] == 1).all() and image.min() >= -1 and image.max() <= 1


def test_param_tree_names_and_shapes_match_reference_layout():
  """SURVEY.md 8b param-tree contract (names feed the optimizer's regex masks)."""
  from big_vision_b200.models.proj.image_text import two_towers
  model = two_towers.Model(**common.TINY)
  P = model.init(0, common.TINY_IMAGE_SHAPE, common.TINY_TEXT_SHAPE, device="cpu")
  tree = P.tree("f")
  d, h, m = 64, 1, 128
  blk = "img/Transformer/encoderblock_1/"
  expect = {
      "img/embedding/kernel": (16, 16, 3, d), "img/embedding/bias": (d,),
      "img/pos_embedding": (1, 16, d),
      blk + "LayerNorm_0/scale": (d,), blk + "LayerNorm_1/bias": (d,),
      blk + "MultiHeadDotProductAttention_0/query/kernel": (d, h, d // h),
      blk + "MultiHeadDotProductAttention_0/value/bias": (h, d // h),
      blk + "MultiHeadDotProductAttention_0/out/kernel": (h, d // h, d),
      blk + "MultiHeadDotProductAttention_0/out/bias": (d,),
      blk + "MlpBlock_0/Dense_0/kernel": (d, m), blk + "MlpBlock_0/Dense_1/bias": (d,),
      "img/Transformer/encoder_norm/scale": (d,),
      "img/MAPHead_0/probe": (1, 1, d),
      "img/MAPHead_0/MultiHeadDotProductAttention_0/key/kernel": (d, h, d // h),
      "img/MAPHead_0/LayerNorm_0/scale": (d,), "img/MAPHead_0/MlpBlock_0/Dense_0/bias": (m,),
      "txt/Embed_0/embedding": (64, d), "txt/pos_embedding": (1, 16, d),
      "txt/Encoder_0/encoderblock_0/MlpBlock_0/Dense_1/kernel": (m, d),
      "txt/Encoder_0/encoder_norm/bias": (d,), "txt/head/kernel": (d, 64), "txt/head/bias": (64,),
      "t": (1,), "b": (1,),
  }
  for k, shp in expect.items():
    assert k in tree, k
    assert tuple(tree[k].shape) == shp, (k, tuple(tree[k].shape), shp)
  assert not any("qkv" in k or "kernel_flat" in k or "out_proj" in k for k in tree)
  assert float(tree["t"][0]) == pytest.approx(math.log(10.0)) and float(tree["b"][0]) == -10.0
  # decayed (".*/kernel$") parameters sit in one contiguous range at the front of the flat buffer
  assert 0 < P.n_decay < P.total
  off, _ = P.offsets["img/Transformer/encoder_norm/scale"]
  assert off >= P.n_decay
  # round trip through the reference-named tree
  np_tree = P.numpy_tree("f")
  P2 = model.init(1, common.TINY_IMAGE_SHAPE, common.TINY_TEXT_SHAPE, device="cpu").load_tree(np_tree)
  assert torch.equal(P.flat, P2.flat)


def test_scan_encoder_parameter_tree_matches_reference_scan_layout():
  """scan=True (models/vit.py:129-148): ONE `encoderblock` sub-tree whose leaves carry a leading depth
  axis (what vit.pyloop_to_scan produces from the per-layer trees); DenseGeneral shapes keep [d,h,dh]."""
  from big_vision_b200 import utils as u
  from big_vision_b200.models import vit
  kw = dict(width=128, depth=3, mlp_dim=256, num_heads=2, patch_size=(16, 16), pool_type="map")
  shape = (2, 32, 32, 3)
  P_loop = vit.Model(None, **kw).init(0, shape, device="cpu")
  P_scan = vit.Model(None, scan=True, **kw).init(0, shape, device="cpu")
  flat = P_loop.numpy_tree("f")
  nested = u.recover_tree(list(flat.keys()), list(flat.values()))
  want = {k: v.shape for k, v in u.tree_flatten_with_names(vit.pyloop_to_scan(nested))[0]}
  got = {k: tuple(v.shape) for k, v in P_scan.tree("f").items()}
  assert got == want
  blk = "Transformer/encoderblock/"
  assert got[blk + "MultiHeadDotProductAttention_0/key/kernel"] == (3, 128, 2, 64)
  assert got[blk + "MultiHeadDotProductAttention_0/out/kernel"] == (3, 2, 64, 128)
  assert got[blk + "MlpBlock_0/Dense_0/bias"] == (3, 256) and got["MAPHead_0/probe"] == (1, 1, 128)
  # the decayed group (".*/kernel$") is still one contiguous prefix of the flat buffer
  assert 0 < P_scan.n_decay < P_scan.total and P_scan.total == P_loop.total


def test_mixer_stochastic_depth_schedule_and_masks():
  """mlp_mixer.py:76: drop_p_i = i / (L - 1) * stoch_depth; masks are 1 - Bernoulli(drop_p_i) per
  sample and branch (:173-177)."""
  from big_vision_b200.models import mlp_mixer
  m = mlp_mixer.Model(10, variant="B/16", stoch_depth=0.1)
  assert m.drop_p(0) == 0.0 and m.drop_p(11) == pytest.approx(0.1) and m.drop_p(5) == pytest.approx(0.1 * 5 / 11)
  masks = m.draw_masks(np.random.default_rng(0), 4096, "cpu")
  assert tuple(masks.shape) == (12, 2, 4096) and set(np.unique(masks.numpy())) <= {0.0, 1.0}
  assert float(masks[0].min()) == 1.0
  assert abs(float(1 - masks[11].mean()) - 0.1) < 0.02


def test_text_pooling_variants_and_unpooled_vit():
  """text_transformer.py:82-95 / models/vit.py:242-255: every pooling of the reference exists in the
  oracle and in the model's parameter tree; the max pool splits its cotangent between ties (the
  jnp.max rule), which is what bv_pool_max_bwd implements."""
  import common
  from big_vision_b200.models import vit
  from big_vision_b200.models.proj.image_text import text_transformer
  x = torch.tensor([[[1.0, 5.0], [3.0, 5.0], [3.0, 2.0]]], dtype=torch.float64, requires_grad=True)
  torch.amax(x, dim=1).sum().backward()
  assert x.grad.tolist() == [[[0.0, 0.5], [0.5, 0.5], [0.5, 0.0]]]
  for pool, extra in [("last", 0), ("first", 0), ("gap", 0), ("gmp", 0), ("map", 15)]:
    m = text_transformer.Model(32, **dict(common.TINY["text"], pool_type=pool))
    P = m.init(0, common.TINY_TEXT_SHAPE, device="cpu")
    names = set(P.tree("f"))
    assert sum(k.startswith("MAPHead_0/") for k in names) == extra, pool
    text = torch.from_numpy(common.synthetic_batch(common.TINY_IMAGE_SHAPE, common.TINY_TEXT_SHAPE, 64)[1])
    z = O.text_forward(O.to_f64_tree(P.numpy_tree("f")), text, dict(depth=2, num_heads=1, pool_type=pool,
                                                                    num_classes=32))
    assert tuple(z.shape) == (8, 32)
  with pytest.raises(NotImplementedError):
    text_transformer.Model(32, **dict(common.TINY["text"], pool_type="median"))
  v = vit.Model(16, width=64, depth=1, mlp_dim=128, num_heads=1, patch_size=(16, 16), pool_type="none")
  P = v.init(0, (2, 32, 48, 3), device="cpu")
  cfg = dict(depth=1, num_heads=1, pool_type="none", num_classes=16)
  assert tuple(O.vit_forward(O.to_f64_tree(P.numpy_tree("f")), torch.zeros(2, 32, 48, 3), cfg).shape) == (2, 6, 16)


def _standin():
  import importlib.util
  root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
  spec = importlib.util.spec_from_file_location("torch_gpu_standin", os.path.join(root, "baseline", "torch_gpu.py"))
  T = importlib.util.module_from_spec(spec)
  spec.loader.exec_module(T)
  return T


def test_mixer_oracle_agrees_with_the_module_style_restatement():
  """No third-party MLP-Mixer is in the image, so unlike the ViT / SigLIP rows (test_oracle_hf_pin.py) the
  Mixer oracle is only checked against a second, separately written restatement: the nn.Module model of
  baseline/torch_gpu.py (the labelled GPU stand-in), float64 on CPU.  Two restatements of
  models/mlp_mixer.py:30-84 that disagreed anywhere (token/channel transposes, LayerNorm placement, the
  [tokens, tokens_mlp] kernels, mean pooling after pre_head_layer_norm) would show up here."""
  T = _standin()
  from big_vision_b200.models import mlp_mixer
  d, blocks, tok, ch, classes = 64, 2, 32, 128, 10
  T.MIXER["tiny"] = (d, blocks, tok, ch)
  m = mlp_mixer.Model(classes, patch_size=(16, 16), num_blocks=blocks, hidden_dim=d, tokens_mlp_dim=tok,
                      channels_mlp_dim=ch)
  P = m.init(0, (3, 64, 64, 3), device="cpu")
  rng = np.random.default_rng(5)
  tree = {k: (v if np.any(v) else (rng.standard_normal(v.shape) * 0.1).astype(np.float32))
          for k, v in P.numpy_tree("f").items()}
  t = {k: torch.from_numpy(np.asarray(v, dtype=np.float64)) for k, v in tree.items()}
  ref = T.Mixer("tiny/16", 64, classes).double().eval()
  sd = {"stem.weight": t["stem/kernel"].permute(3, 2, 0, 1), "stem.bias": t["stem/bias"],
        "norm.weight": t["pre_head_layer_norm/scale"], "norm.bias": t["pre_head_layer_norm/bias"],
        "head.weight": t["head/kernel"].T, "head.bias": t["head/bias"]}
  for i in range(blocks):
    b = f"MixerBlock_{i}/"
    for ln, src in (("ln1", "LayerNorm_0"), ("ln2", "LayerNorm_1")):
      sd[f"blocks.{i}.{ln}.weight"], sd[f"blocks.{i}.{ln}.bias"] = t[b + src + "/scale"], t[b + src + "/bias"]
    for mlp, src in (("tok", "token_mixing"), ("ch", "channel_mixing")):
      for fc, dn in (("fc1", "Dense_0"), ("fc2", "Dense_1")):
        sd[f"blocks.{i}.{mlp}.{fc}.weight"] = t[f"{b}{src}/{dn}/kernel"].T
        sd[f"blocks.{i}.{mlp}.{fc}.bias"] = t[f"{b}{src}/{dn}/bias"]
  assert set(sd) == set(ref.state_dict())
  ref.load_state_dict({k: v.contiguous() for k, v in sd.items()})
  image = torch.from_numpy(rng.uniform(-1, 1, size=(3, 64, 64, 3))).double()
  p64 = O.to_f64_tree(tree, requires_grad=True)
  mine = O.mixer_forward(p64, image, dict(num_blocks=blocks, num_classes=classes))
  theirs = ref(image)
  assert float((mine - theirs).abs().max()) < 1e-10 * max(1.0, float(theirs.abs().max()))
  labels = torch.nn.functional.one_hot(torch.from_numpy(rng.integers(0, classes, size=3)), classes).double()
  O.sigmoid_xent(mine, labels).backward()
  (-(labels * torch.nn.functional.logsigmoid(theirs) + (1 - labels) * torch.nn.functional.logsigmoid(-theirs))
   .sum(-1).mean()).backward()
  g = dict(ref.named_parameters())
  TOL = 1e-9
  for name, r in [("stem/kernel", g["stem.weight"].grad.permute(2, 3, 1, 0)),
                  ("MixerBlock_0/token_mixing/Dense_0/kernel", g["blocks.0.tok.fc1.weight"].grad.T),
                  ("MixerBlock_1/token_mixing/Dense_1/bias", g["blocks.1.tok.fc2.bias"].grad),
                  ("MixerBlock_1/channel_mixing/Dense_1/kernel", g["blocks.1.ch.fc2.weight"].grad.T),
                  ("MixerBlock_0/LayerNorm_1/scale", g["blocks.0.ln2.weight"].grad)]:
    # (the token-mixing Dense_1 bias shifts all channels of a token alike and every later consumer is a
    # LayerNorm over channels: its exact gradient is zero, hence the absolute floor)
    assert float((p64[name].grad - r).abs().max()) <= TOL * float(r.abs().max()) + 1e-14, name


def test_gpu_standin_computes_the_oracles_siglip_function():
  """bench.py times baseline/torch_gpu.py beside the product as the labelled stand-in for the reference's
  GPU build.  That comparison only means something if the stand-in computes the same model and loss: mapped
  parameters, float64, CPU -- embeddings, loss and gradients must equal the oracle's (which
  test_oracle_hf_pin.py ties to transformers' SigLIP)."""
  T = _standin()
  from big_vision_b200.models.proj.image_text import two_towers
  d, depth, mlp, heads = 128, 2, 256, 2
  T.VIT["tiny"] = (d, depth, mlp, heads)
  tower = dict(width=d, depth=depth, mlp_dim=mlp, num_heads=heads)
  model = two_towers.Model(image=dict(tower, patch_size=(16, 16), pool_type="map"),
                           text=dict(tower, vocab_size=32_000), out_dim=(None, d), temperature_init=10.0,
                           bias_init=-10.0)
  P = model.init(0, (4, 64, 64, 3), (4, 64), device="cpu")
  rng = np.random.default_rng(9)
  tree = {k: (v if np.any(v) else (rng.standard_normal(v.shape) * 0.1).astype(np.float32))
          for k, v in P.numpy_tree("f").items()}
  t = {k: torch.from_numpy(np.asarray(v, dtype=np.float64)) for k, v in tree.items()}
  ref = T.TwoTowers("tiny/16", "tiny", 64, d).double().eval()
  sd = {"t": t["t"], "b": t["b"]}

  def lin(dst, kernel, bias):
    sd[dst + ".weight"], sd[dst + ".bias"] = kernel.T, bias

  def norm(dst, src):
    sd[dst + ".weight"], sd[dst + ".bias"] = t[src + "/scale"], t[src + "/bias"]

  def proj(att, names):                       # reference [d, h, dh] kernels -> one fused [d, k*d] kernel
    return (torch.cat([t[f"{att}/{n}/kernel"].reshape(d, d) for n in names], 1),
            torch.cat([t[f"{att}/{n}/bias"].reshape(d) for n in names]))

  def mlp_block(dst, src):
    lin(dst + ".fc1", t[src + "/Dense_0/kernel"], t[src + "/Dense_0/bias"])
    lin(dst + ".fc2", t[src + "/Dense_1/kernel"], t[src + "/Dense_1/bias"])

  def encoder(dst, src):
    for i in range(depth):
      b, o = f"{src}/encoderblock_{i}", f"{dst}.blocks.{i}"
      att = b + "/MultiHeadDotProductAttention_0"
      lin(o + ".attn.qkv", *proj(att, ("query", "key", "value")))
      lin(o + ".attn.out", t[att + "/out/kernel"].reshape(d, d), t[att + "/out/bias"])
      norm(o + ".ln1", b + "/LayerNorm_0")
      norm(o + ".ln2", b + "/LayerNorm_1")
      mlp_block(o + ".mlp", b + "/MlpBlock_0")
    norm(dst + ".norm", src + "/encoder_norm")

  sd["img.embed.weight"], sd["img.embed.bias"] = t["img/embedding/kernel"].permute(3, 2, 0, 1), t["img/embedding/bias"]
  sd["img.pos"] = t["img/pos_embedding"]
  encoder("img.encoder", "img/Transformer")
  m = "img/MAPHead_0"
  sd["img.probe"] = t[m + "/probe"]
  att = m + "/MultiHeadDotProductAttention_0"
  lin("img.map_attn.q", *proj(att, ("query",)))
  lin("img.map_attn.kv", *proj(att, ("key", "value")))
  lin("img.map_attn.out", t[att + "/out/kernel"].reshape(d, d), t[att + "/out/bias"])
  norm("img.map_ln", m + "/LayerNorm_0")
  mlp_block("img.map_mlp", m + "/MlpBlock_0")
  sd["txt.embed.weight"], sd["txt.pos"] = t["txt/Embed_0/embedding"], t["txt/pos_embedding"]
  encoder("txt.encoder", "txt/Encoder_0")
  lin("txt.head", t["txt/head/kernel"], t["txt/head/bias"])
  assert set(sd) == set(ref.state_dict()), set(sd) ^ set(ref.state_dict())
  ref.load_state_dict({k: v.contiguous() for k, v in sd.items()})
  image = torch.from_numpy(rng.uniform(-1, 1, size=(4, 64, 64, 3))).double()
  text = torch.from_numpy(rng.integers(0, 32_000, size=(4, 64))).int()
  p64 = O.to_f64_tree(tree, requires_grad=True)
  cfg = {"image": dict(depth=depth, num_heads=heads, pool_type="map", posemb="learn", rep_size=False, num_classes=None),
         "text": dict(depth=depth, num_heads=heads, pool_type="last", num_classes=d)}
  zi, zt, ex = O.two_towers_forward(p64, image, text, cfg, "float32")
  zi2, zt2 = ref(image, text)
  # the stand-in hands its embeddings to the loss as float32 (`.float()` after the autocast region), so the
  # agreement is float32 rounding, not float64
  assert float((zi - zi2).abs().max()) < 2e-7 and float((zt - zt2).abs().max()) < 2e-7
  mine = O.siglip_loss(zi, zt, ex["t"], ex["b"])
  theirs = T.siglip_loss(zi2, zt2, ref.t, ref.b, 0, 4)
  assert float(mine) == pytest.approx(float(theirs), rel=1e-6)
  mine.backward()
  theirs.backward()
  g = dict(ref.named_parameters())
  TOL = 1e-5
  for name, r in [("img/pos_embedding", g["img.pos"].grad), ("img/MAPHead_0/probe", g["img.probe"].grad),
                  ("txt/head/kernel", g["txt.head.weight"].grad.T), ("t", g["t"].grad), ("b", g["b"].grad),
                  ("img/Transformer/encoderblock_0/MultiHeadDotProductAttention_0/value/kernel",
                   g["img.encoder.blocks.0.attn.qkv.weight"].grad.T[:, 2 * d:].reshape(d, heads, d // heads)),
                  ("img/MAPHead_0/MultiHeadDotProductAttention_0/key/kernel",
                   g["img.map_attn.kv.weight"].grad.T[:, :d].reshape(d, heads, d // heads))]:
    assert float((p64[name].grad - r).abs().max()) <= TOL * float(r.abs().max()) + 1e-14, name
