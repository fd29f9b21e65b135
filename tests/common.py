"""Shared tiny configurations for the tests (kept small so the CPU oracle runs in seconds)."""
import hashlib
import os

import numpy as np

GOLDEN_TINY = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "siglip_tiny.npz")

TINY = dict(
    image=dict(width=64, depth=2, mlp_dim=128, num_heads=1, patch_size=(16, 16), pool_type="map"),
    text=dict(width=64, depth=2, mlp_dim=128, num_heads=1, vocab_size=64),
    out_dim=(None, 64), temperature_init=10.0, bias_init=-10.0,
)
TINY_IMAGE_SHAPE = (8, 64, 64, 3)
TINY_TEXT_SHAPE = (8, 16)


def oracle_cfg(model_kw):
  return {
      "image": dict(depth=model_kw["image"]["depth"], num_heads=model_kw["image"]["num_heads"],
                    pool_type=model_kw["image"].get("pool_type", "gap"),
                    posemb=model_kw["image"].get("posemb", "learn"),
                    rep_size=model_kw["image"].get("rep_size", False),
                    num_classes=model_kw["out_dim"][0]),
      "text": dict(depth=model_kw["text"]["depth"], num_heads=model_kw["text"]["num_heads"],
                   pool_type=model_kw["text"].get("pool_type", "last"),
                   num_classes=model_kw["out_dim"][1]),
  }


def synthetic_batch(image_shape, text_shape, vocab, seed=0):
  """SURVEY.md 8d synthetic inputs: images U(-1,1); text ids in [2,vocab) for a random length,
  then sticky EOS / pad id 1 to the end (so the last token is always 1)."""
  rng = np.random.default_rng(seed)
  image = rng.uniform(-1, 1, size=image_shape).astype(np.float32)
  n, L = text_shape
  text = np.ones((n, L), dtype=np.int32)
  lens = rng.integers(min(4, L - 1), L, size=n)
  for i in range(n):
    text[i, :lens[i]] = rng.integers(2, vocab, size=lens[i])
  return image, text


def sha256_of(arrays):
  """Digest of a dict of arrays: names, dtypes, shapes and contents, in name order."""
  h = hashlib.sha256()
  for k in sorted(arrays):
    a = np.ascontiguousarray(arrays[k])
    h.update(f"{k}:{a.dtype.str}:{a.shape};".encode())
    h.update(a.tobytes())
  return h.hexdigest()


def tiny_inputs():
  """The TINY two-tower parameters (init seed 0, float32 numpy tree) and synthetic batch (seed 0)."""
  from big_vision_b200.models.proj.image_text import two_towers
  P = two_towers.Model(**TINY).init(0, TINY_IMAGE_SHAPE, TINY_TEXT_SHAPE, device="cpu")
  image, text = synthetic_batch(TINY_IMAGE_SHAPE, TINY_TEXT_SHAPE, TINY["text"]["vocab_size"])
  return P.numpy_tree("f"), image, text


def load_golden_tiny():
  """tests/golden/siglip_tiny.npz and the inputs its vectors were computed from: (z, params, image, text).
  The file holds the oracle's outputs and the text ids; the parameters and the image are regenerated
  from their seeds and must match the digests stored with the outputs, so a changed initialiser or
  input recipe fails here instead of comparing against outputs of other inputs."""
  z = np.load(GOLDEN_TINY)
  tree, image, text = tiny_inputs()
  regen = "; regenerate the file with tests/golden/make_golden.py if the change is intended"
  assert sha256_of(tree) == str(z["params_sha256"]), "init(seed=0) no longer gives the golden parameters" + regen
  assert sha256_of({"image": image}) == str(z["image_sha256"]), "the synthetic image recipe changed" + regen
  assert np.array_equal(text, z["text"]), "the synthetic text recipe changed" + regen
  return z, tree, image, text
