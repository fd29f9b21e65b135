"""CPU: pins the oracle's SigLIP path against an implementation it shares no code with.

jax / flax cannot be installed here, so the oracle cannot be compared with the reference itself
(oracle/bv_oracle.py header).  The `transformers` package in this image carries `SiglipModel`, a PyTorch
implementation of the same two-tower model whose conversion script checks its outputs against the
reference's released checkpoints.  Mapping one random parameter tree into both and comparing, in float64,
image / text embeddings, the pairwise-sigmoid loss and the gradients pins what the oracle otherwise asserts
from the reference's source alone: LayerNorm epsilon, tanh-GELU, 1/sqrt(dh) query scaling and the head
split of the [d, h, dh] kernels, the MAP head, last-token text pooling, normalisation, temperature / bias
and the loss of trainers/proj/image_text/siglip.py:287-308.  Test infrastructure only."""
import numpy as np
import pytest
import torch

from oracle import bv_oracle as O

transformers = pytest.importorskip("transformers")

W, HEADS, DEPTH, MLP, VOCAB, LEN, RES, PATCH, OUT = 128, 2, 2, 256, 97, 12, 64, 16, 128


def _tree(seed):
  from big_vision_b200.models.proj.image_text import two_towers
  tower = dict(width=W, depth=DEPTH, mlp_dim=MLP, num_heads=HEADS)
  model = two_towers.Model(image=dict(tower, patch_size=(PATCH, PATCH), pool_type="map"),
                           text=dict(tower, vocab_size=VOCAB), out_dim=(None, OUT),
                           temperature_init=10.0, bias_init=-10.0)
  P = model.init(seed, (4, RES, RES, 3), (4, LEN), device="cpu")
  rng = np.random.default_rng(seed + 1)
  tree = {}
  for k, v in P.numpy_tree("f").items():       # zero-initialised biases would hide a wrong mapping
    tree[k] = v if np.any(v) else (rng.standard_normal(v.shape) * 0.1).astype(np.float32)
  tree["img/MAPHead_0/LayerNorm_0/scale"] = (1 + 0.2 * rng.standard_normal(W)).astype(np.float32)
  return tree


def _hf_state(tree, W=W, DEPTH=DEPTH):
  """The oracle's (= the reference's) parameter tree in transformers' SiglipModel layout."""
  t = {k: torch.from_numpy(np.asarray(v, dtype=np.float64)) for k, v in tree.items()}
  sd = {}

  def dense(dst, src):                                     # flax [in, out] -> torch Linear [out, in]
    sd[dst + ".weight"], sd[dst + ".bias"] = t[src + "/kernel"].T, t[src + "/bias"]

  def norm(dst, src):
    sd[dst + ".weight"], sd[dst + ".bias"] = t[src + "/scale"], t[src + "/bias"]

  def qkv(src, which):                                     # [d, h, dh] -> [h*dh, d]
    return t[f"{src}/{which}/kernel"].reshape(W, W).T, t[f"{src}/{which}/bias"].reshape(W)

  def block(dst, src):
    att = src + "/MultiHeadDotProductAttention_0"
    for hf, bv in (("q_proj", "query"), ("k_proj", "key"), ("v_proj", "value")):
      sd[f"{dst}.self_attn.{hf}.weight"], sd[f"{dst}.self_attn.{hf}.bias"] = qkv(att, bv)
    sd[f"{dst}.self_attn.out_proj.weight"] = t[att + "/out/kernel"].reshape(W, W).T      # [h, dh, d]
    sd[f"{dst}.self_attn.out_proj.bias"] = t[att + "/out/bias"]
    norm(dst + ".layer_norm1", src + "/LayerNorm_0")
    norm(dst + ".layer_norm2", src + "/LayerNorm_1")
    dense(dst + ".mlp.fc1", src + "/MlpBlock_0/Dense_0")
    dense(dst + ".mlp.fc2", src + "/MlpBlock_0/Dense_1")

  v = "vision_model."
  sd[v + "embeddings.patch_embedding.weight"] = t["img/embedding/kernel"].permute(3, 2, 0, 1)   # HWIO -> OIHW
  sd[v + "embeddings.patch_embedding.bias"] = t["img/embedding/bias"]
  sd[v + "embeddings.position_embedding.weight"] = t["img/pos_embedding"][0]
  for i in range(DEPTH):
    block(f"{v}encoder.layers.{i}", f"img/Transformer/encoderblock_{i}")
  norm(v + "post_layernorm", "img/Transformer/encoder_norm")
  m = "img/MAPHead_0"
  sd[v + "head.probe"] = t[m + "/probe"]
  ws, bs = zip(*(qkv(m + "/MultiHeadDotProductAttention_0", w) for w in ("query", "key", "value")))
  sd[v + "head.attention.in_proj_weight"], sd[v + "head.attention.in_proj_bias"] = torch.cat(ws), torch.cat(bs)
  sd[v + "head.attention.out_proj.weight"] = t[m + "/MultiHeadDotProductAttention_0/out/kernel"].reshape(W, W).T
  sd[v + "head.attention.out_proj.bias"] = t[m + "/MultiHeadDotProductAttention_0/out/bias"]
  norm(v + "head.layernorm", m + "/LayerNorm_0")
  dense(v + "head.mlp.fc1", m + "/MlpBlock_0/Dense_0")
  dense(v + "head.mlp.fc2", m + "/MlpBlock_0/Dense_1")
  x = "text_model."
  sd[x + "embeddings.token_embedding.weight"] = t["txt/Embed_0/embedding"]
  sd[x + "embeddings.position_embedding.weight"] = t["txt/pos_embedding"][0]
  for i in range(DEPTH):
    block(f"{x}encoder.layers.{i}", f"txt/Encoder_0/encoderblock_{i}")
  norm(x + "final_layer_norm", "txt/Encoder_0/encoder_norm")
  dense(x + "head", "txt/head")
  sd["logit_scale"], sd["logit_bias"] = t["t"], t["b"]
  return {k: v.contiguous() for k, v in sd.items()}


def _hf_model(tree, width, depth, mlp, heads, res, patch, vocab, length, out):
  from transformers import SiglipConfig, SiglipModel
  common_kw = dict(hidden_size=width, intermediate_size=mlp, num_hidden_layers=depth, num_attention_heads=heads,
                   layer_norm_eps=1e-6, hidden_act="gelu_pytorch_tanh", attention_dropout=0.0)
  cfg = SiglipConfig(vision_config=dict(common_kw, image_size=res, patch_size=patch, num_channels=3),
                     text_config=dict(common_kw, vocab_size=vocab, max_position_embeddings=length, projection_size=out))
  cfg._attn_implementation = "eager"
  hf = SiglipModel(cfg).double().eval()
  state = _hf_state(tree, width, depth)
  own = hf.state_dict()
  assert set(state) == set(k for k in own if "position_ids" not in k), set(state) ^ set(own)
  for k, v in state.items():
    assert tuple(v.shape) == tuple(own[k].shape), (k, v.shape, own[k].shape)
  hf.load_state_dict(state, strict=False)
  return hf


@pytest.fixture(scope="module")
def pair():
  tree = _tree(0)
  hf = _hf_model(tree, W, DEPTH, MLP, HEADS, RES, PATCH, VOCAB, LEN, OUT)
  rng = np.random.default_rng(7)
  image = torch.from_numpy(rng.uniform(-1, 1, size=(4, RES, RES, 3))).double()
  text = torch.from_numpy(rng.integers(0, VOCAB, size=(4, LEN)))
  return tree, hf, image, text


def _oracle(tree, image, text, requires_grad=False):
  p64 = O.to_f64_tree(tree, requires_grad=requires_grad)
  tower = dict(depth=DEPTH, num_heads=HEADS)
  cfg = {"image": dict(tower, pool_type="map", posemb="learn", rep_size=False, num_classes=None),
         "text": dict(tower, pool_type="last", num_classes=OUT)}
  zi, zt, ex = O.two_towers_forward(p64, image, text.int(), cfg, "float32")
  return p64, zi, zt, ex


def test_oracle_embeddings_match_transformers_siglip(pair):
  tree, hf, image, text = pair
  _, zi, zt, ex = _oracle(tree, image, text)
  with torch.no_grad():
    out = hf(input_ids=text, pixel_values=image.permute(0, 3, 1, 2), return_loss=True)
  # the oracle divides by (norm + 1e-8) (two_towers.py:60-61), transformers by the norm: 1e-8 relative
  assert float((out.image_embeds - zi).abs().max()) < 1e-7
  assert float((out.text_embeds - zt).abs().max()) < 1e-7
  logits = zi @ zt.T * ex["t"] + ex["b"]
  assert float((out.logits_per_image - logits).abs().max()) < 1e-6
  assert float(out.loss) == pytest.approx(float(O.siglip_loss(zi, zt, ex["t"], ex["b"])), rel=1e-7)


def test_oracle_gradients_match_transformers_siglip(pair):
  tree, hf, image, text = pair
  p64, zi, zt, ex = _oracle(tree, image, text, requires_grad=True)
  O.siglip_loss(zi, zt, ex["t"], ex["b"]).backward()
  hf.zero_grad()
  hf(input_ids=text, pixel_values=image.permute(0, 3, 1, 2), return_loss=True).loss.backward()
  g = dict(hf.named_parameters())
  checks = [
      ("img/embedding/kernel", g["vision_model.embeddings.patch_embedding.weight"].grad.permute(2, 3, 1, 0)),
      ("img/pos_embedding", g["vision_model.embeddings.position_embedding.weight"].grad[None]),
      ("img/Transformer/encoderblock_0/MultiHeadDotProductAttention_0/key/kernel",
       g["vision_model.encoder.layers.0.self_attn.k_proj.weight"].grad.T.reshape(W, HEADS, W // HEADS)),
      ("img/Transformer/encoderblock_1/MlpBlock_0/Dense_0/kernel", g["vision_model.encoder.layers.1.mlp.fc1.weight"].grad.T),
      ("img/MAPHead_0/probe", g["vision_model.head.probe"].grad),
      ("img/MAPHead_0/MultiHeadDotProductAttention_0/out/kernel",
       g["vision_model.head.attention.out_proj.weight"].grad.T.reshape(HEADS, W // HEADS, W)),
      ("txt/Embed_0/embedding", g["text_model.embeddings.token_embedding.weight"].grad),
      ("txt/Encoder_0/encoderblock_0/LayerNorm_1/scale", g["text_model.encoder.layers.0.layer_norm2.weight"].grad),
      ("txt/Encoder_0/encoderblock_1/MultiHeadDotProductAttention_0/out/bias",
       g["text_model.encoder.layers.1.self_attn.out_proj.bias"].grad),
      ("txt/head/kernel", g["text_model.head.weight"].grad.T),
      ("t", g["logit_scale"].grad),
      ("b", g["logit_bias"].grad),
  ]
  for name, ref in checks:
    mine = p64[name].grad
    scale = float(ref.abs().max()) + 1e-30
    assert float((mine - ref).abs().max()) <= 1e-6 * scale + 1e-12, name


def test_committed_golden_vectors_equal_transformers_outputs():
  """tests/golden/siglip_tiny.npz is what the GPU parity tests (tests/test_model_gpu.py) compare the CUDA path
  with.  It was written by the oracle (tests/golden/make_golden.py); here the parameters and inputs it was
  computed from go through transformers' SiglipModel and must reproduce the file's float32-mode embeddings, loss and every
  stored gradient -- which ties the GPU tests' reference values to an implementation other than the oracle."""
  import common
  z, tree, image, text = common.load_golden_tiny()
  kw = common.TINY
  hf = _hf_model(tree, kw["image"]["width"], kw["image"]["depth"], kw["image"]["mlp_dim"], kw["image"]["num_heads"],
                 common.TINY_IMAGE_SHAPE[1], kw["image"]["patch_size"][0], kw["text"]["vocab_size"],
                 common.TINY_TEXT_SHAPE[1], kw["out_dim"][1])
  image = torch.from_numpy(image).double().permute(0, 3, 1, 2)
  out = hf(input_ids=torch.from_numpy(text).long(), pixel_values=image, return_loss=True)
  assert float((out.image_embeds.detach() - torch.from_numpy(z["float32:zimg"])).abs().max()) < 1e-7
  assert float((out.text_embeds.detach() - torch.from_numpy(z["float32:ztxt"])).abs().max()) < 1e-7
  assert float(out.loss) == pytest.approx(float(z["float32:loss"]), rel=1e-7)
  out.loss.backward()
  g = dict(hf.named_parameters())
  w = kw["image"]["width"]
  checks = {
      "img/pos_embedding": g["vision_model.embeddings.position_embedding.weight"].grad[None],
      "img/embedding/bias": g["vision_model.embeddings.patch_embedding.bias"].grad,
      "img/Transformer/encoderblock_0/MlpBlock_0/Dense_0/kernel": g["vision_model.encoder.layers.0.mlp.fc1.weight"].grad.T,
      "img/Transformer/encoderblock_1/MultiHeadDotProductAttention_0/out/kernel":
          g["vision_model.encoder.layers.1.self_attn.out_proj.weight"].grad.T.reshape(1, w, w),
      "img/MAPHead_0/probe": g["vision_model.head.probe"].grad,
      "img/MAPHead_0/MlpBlock_0/Dense_1/kernel": g["vision_model.head.mlp.fc2.weight"].grad.T,
      "txt/Embed_0/embedding": g["text_model.embeddings.token_embedding.weight"].grad,
      "txt/Encoder_0/encoderblock_0/MultiHeadDotProductAttention_0/query/kernel":
          g["text_model.encoder.layers.0.self_attn.q_proj.weight"].grad.T.reshape(w, 1, w),
      "txt/Encoder_0/encoder_norm/scale": g["text_model.final_layer_norm.weight"].grad,
      "txt/head/bias": g["text_model.head.bias"].grad,
      "t": g["logit_scale"].grad, "b": g["logit_bias"].grad,
  }
  for name, ref in checks.items():
    gold = torch.from_numpy(z["float32:grad:" + name]).double()
    assert float((gold - ref).abs().max()) <= 1e-6 * float(ref.abs().max()) + 1e-12, name


# ---------------------------------------------------------------------------------------------------
# The classification ViT (models/vit.py with pool_type="tok") against transformers' ViTForImageClassification,
# the PyTorch port of the original ViT.  The one structural difference is where the class token meets the
# position embedding: the reference adds the embedding to the patches and THEN prepends the token
# (models/vit.py:219-225); transformers prepends first and adds an [N+1]-row embedding.  A zero first row
# makes the two identical.
# ---------------------------------------------------------------------------------------------------
def _vit_pair(seed, classes=10):
  from transformers import ViTConfig, ViTForImageClassification
  from big_vision_b200.models import vit
  model = vit.Model(classes, width=W, depth=DEPTH, mlp_dim=MLP, num_heads=HEADS, patch_size=(PATCH, PATCH),
                    pool_type="tok", posemb="learn")
  P = model.init(seed, (3, RES, 48, 3), device="cpu")
  rng = np.random.default_rng(seed + 1)
  tree = {k: (v if np.any(v) else (rng.standard_normal(v.shape) * 0.1).astype(np.float32))
          for k, v in P.numpy_tree("f").items()}
  t = {k: torch.from_numpy(np.asarray(v, dtype=np.float64)) for k, v in tree.items()}
  sd = {}

  def dense(dst, src):
    sd[dst + ".weight"], sd[dst + ".bias"] = t[src + "/kernel"].T, t[src + "/bias"]

  def norm(dst, src):
    sd[dst + ".weight"], sd[dst + ".bias"] = t[src + "/scale"], t[src + "/bias"]

  e = "vit.embeddings."
  sd[e + "cls_token"] = t["cls"]
  sd[e + "position_embeddings"] = torch.cat([torch.zeros(1, 1, W, dtype=torch.float64), t["pos_embedding"]], 1)
  sd[e + "patch_embeddings.projection.weight"] = t["embedding/kernel"].permute(3, 2, 0, 1)
  sd[e + "patch_embeddings.projection.bias"] = t["embedding/bias"]
  for i in range(DEPTH):
    src, dst = f"Transformer/encoderblock_{i}", f"vit.encoder.layer.{i}"
    att = src + "/MultiHeadDotProductAttention_0"
    for which in ("query", "key", "value"):
      sd[f"{dst}.attention.attention.{which}.weight"] = t[f"{att}/{which}/kernel"].reshape(W, W).T
      sd[f"{dst}.attention.attention.{which}.bias"] = t[f"{att}/{which}/bias"].reshape(W)
    sd[f"{dst}.attention.output.dense.weight"] = t[att + "/out/kernel"].reshape(W, W).T
    sd[f"{dst}.attention.output.dense.bias"] = t[att + "/out/bias"]
    norm(dst + ".layernorm_before", src + "/LayerNorm_0")
    norm(dst + ".layernorm_after", src + "/LayerNorm_1")
    dense(dst + ".intermediate.dense", src + "/MlpBlock_0/Dense_0")
    dense(dst + ".output.dense", src + "/MlpBlock_0/Dense_1")
  norm("vit.layernorm", "Transformer/encoder_norm")
  dense("classifier", "head")
  cfg = ViTConfig(hidden_size=W, num_hidden_layers=DEPTH, num_attention_heads=HEADS, intermediate_size=MLP,
                  hidden_act="gelu_pytorch_tanh", hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0,
                  layer_norm_eps=1e-6, image_size=(RES, 48), patch_size=PATCH, num_channels=3, qkv_bias=True,
                  num_labels=classes)
  cfg._attn_implementation = "eager"
  hf = ViTForImageClassification(cfg).double().eval()
  own = hf.state_dict()
  assert set(sd) == set(own), set(sd) ^ set(own)
  for k, v in sd.items():
    assert tuple(v.shape) == tuple(own[k].shape), (k, v.shape, own[k].shape)
  hf.load_state_dict({k: v.contiguous() for k, v in sd.items()})
  return tree, hf


def test_oracle_vit_classifier_matches_transformers_vit():
  classes = 10
  tree, hf = _vit_pair(3, classes)
  rng = np.random.default_rng(11)
  image = torch.from_numpy(rng.uniform(-1, 1, size=(3, RES, 48, 3))).double()
  labels = torch.from_numpy(rng.integers(0, classes, size=3))
  cfg = dict(depth=DEPTH, num_heads=HEADS, pool_type="tok", posemb="learn", rep_size=False, num_classes=classes)
  p64 = O.to_f64_tree(tree, requires_grad=True)
  logits = O.vit_forward(p64, image, cfg, "float32")
  out = hf(pixel_values=image.permute(0, 3, 1, 2), labels=labels)
  assert float((out.logits - logits).abs().max()) < 1e-9 * max(1.0, float(logits.abs().max()))
  onehot = torch.nn.functional.one_hot(labels, classes).double()
  # utils.softmax_xent (utils.py:276-281) == CrossEntropyLoss(mean); utils.sigmoid_xent (utils.py:236-243)
  # sums over classes where BCEWithLogitsLoss(mean) averages over them
  loss = O.softmax_xent(logits, onehot)
  assert float(loss) == pytest.approx(float(out.loss), rel=1e-10)
  bce = torch.nn.functional.binary_cross_entropy_with_logits(logits, onehot)
  assert float(O.sigmoid_xent(logits, onehot)) == pytest.approx(float(bce) * classes, rel=1e-10)
  loss.backward()
  out.loss.backward()
  g = dict(hf.named_parameters())
  for name, ref in [
      ("cls", g["vit.embeddings.cls_token"].grad),
      ("pos_embedding", g["vit.embeddings.position_embeddings"].grad[:, 1:]),
      ("embedding/kernel", g["vit.embeddings.patch_embeddings.projection.weight"].grad.permute(2, 3, 1, 0)),
      ("Transformer/encoderblock_0/MultiHeadDotProductAttention_0/query/kernel",
       g["vit.encoder.layer.0.attention.attention.query.weight"].grad.T.reshape(W, HEADS, W // HEADS)),
      ("Transformer/encoderblock_1/MlpBlock_0/Dense_1/kernel", g["vit.encoder.layer.1.output.dense.weight"].grad.T),
      ("Transformer/encoder_norm/scale", g["vit.layernorm.weight"].grad),
      ("head/kernel", g["classifier.weight"].grad.T)]:
    scale = float(ref.abs().max()) + 1e-30
    assert float((p64[name].grad - ref).abs().max()) <= 1e-8 * scale, name
