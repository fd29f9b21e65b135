"""Generates tests/golden/siglip_tiny.npz with the CPU oracle (float64).

JAX/flax are not dependencies of this project, so these vectors come from oracle/bv_oracle.py
(itself checked against torch's independent operators in tests/test_oracle.py); they pin the
oracle against drift and give the GPU tests a fixed target that does not depend on re-running it.
The parameters (init seed 0) and the image (synthetic recipe, seed 0) are not stored, only their
digests: tests/common.py:load_golden_tiny regenerates them and checks the digests.
  python tests/golden/make_golden.py
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, os.path.dirname(HERE))

from oracle import bv_oracle as O  # noqa: E402
import common  # noqa: E402


def main():
  tree, image, text = common.tiny_inputs()
  out = {"text": text, "params_sha256": np.array(common.sha256_of(tree)),
         "image_sha256": np.array(common.sha256_of({"image": image}))}
  cfg = common.oracle_cfg(common.TINY)
  for mm in ("float32", "bfloat16"):
    loss, grads, zimg, ztxt = O.siglip_value_and_grad(tree, image, text, cfg, mm)
    out[f"{mm}:loss"] = np.float64(loss)
    out[f"{mm}:zimg"] = zimg
    out[f"{mm}:ztxt"] = ztxt
    if mm == "float32":   # full gradients only for the high-precision model (keeps the file small)
      for k, g in grads.items():
        out[f"{mm}:grad:" + k] = g.astype(np.float32)
    else:
      out[f"{mm}:gradnorm"] = np.float64(np.sqrt(sum(float((g.astype(np.float64) ** 2).sum()) for g in grads.values())))
    print(mm, "loss", loss)
  np.savez_compressed(os.path.join(HERE, "siglip_tiny.npz"), **out)
  print("wrote", os.path.join(HERE, "siglip_tiny.npz"))


if __name__ == "__main__":
  main()
