"""CPU: the C-ABI library builds, loads and exports every symbol include/bv_b200.h declares;
argument validation fails loudly (no compute without a GPU)."""
import ctypes
import os
import re

import pytest

from big_vision_b200 import lib as L

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_functions():
  src = open(os.path.join(ROOT, "include", "bv_b200.h")).read()
  src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
  return sorted(set(re.findall(r"\b(bv_[a-z0-9_]+)\s*\(", src)))


def test_header_symbols_exported():
  lib = L.load()
  names = _header_functions()
  assert len(names) >= 25
  for n in names:
    assert hasattr(lib, n), f"{n} declared in include/bv_b200.h but not exported"


def test_binding_covers_header():
  declared = set(_header_functions()) - {"bv_last_error_string"}
  assert declared == set(L.SIGNATURES), (declared ^ set(L.SIGNATURES))


def test_version_and_no_gpu_support_flag():
  lib = L.load()
  assert lib.bv_version() == 100
  assert lib.bv_device_supported() in (0, 1)


def test_invalid_arguments_fail_loudly():
  lib = L.load()
  args = L.GemmArgs(M=0, N=8, K=8)
  rc = lib.bv_gemm(ctypes.byref(args), None)
  assert rc == -1
  assert b"empty" in lib.bv_last_error_string()
  args = L.GemmArgs(M=8, N=8, K=8, ldd=12, out_dtype=L.BF16)   # bf16 row stride not 16B-aligned
  assert lib.bv_gemm(ctypes.byref(args), None) == -1
  with pytest.raises(L.BvError):
    L.call("bv_layernorm_fwd", None, 1, None, None, None, 1, None, None, 4, 12, 1e-6, None)


def test_ops_refuse_cpu_tensors():
  import torch
  from big_vision_b200 import ops
  with pytest.raises(L.BvError):
    ops.layernorm_fwd(torch.zeros(4, 64), torch.ones(64), torch.zeros(64))


def test_bench_workloads_cover_the_five_baseline_configs():
  """bench.py --workload: one entry per BASELINE.json config, synthetic batches of the SURVEY 8d shapes."""
  import importlib.util
  import json
  import os
  root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
  spec = importlib.util.spec_from_file_location("bench", os.path.join(root, "bench.py"))
  bench = importlib.util.module_from_spec(spec)
  spec.loader.exec_module(bench)
  assert len(json.load(open(os.path.join(root, "BASELINE.json")))["configs"]) == len(bench.WORKLOADS) == 5
  wl = bench.WORKLOADS["siglip_b16"]
  b = bench.synthetic_batch(wl, 4, seed=0)
  assert b["image"].shape == (4, 224, 224, 3) and b["image"].dtype.name == "float32"
  assert -1.0 <= b["image"].min() and b["image"].max() < 1.0
  assert b["labels"].shape == (4, 64) and b["labels"].dtype.name == "int32" and (b["labels"][:, -1] == 1).all()
  assert bench.synthetic_batch(wl, 2, seed=0, uint8=True)["image"].dtype.name == "uint8"
  c = bench.synthetic_batch(bench.WORKLOADS["vit_b16_cls"], 4, seed=0)
  assert c["labels"].shape == (4, 1000) and (c["labels"].sum(1) == 1).all()
  assert bench.WORKLOADS["siglip_l14_336"]["per_gpu_batch"] * 8 == 16384 and wl["per_gpu_batch"] * 8 == 8192
  model = bench.build_model(bench.WORKLOADS["siglip_l14_336"])
  assert model.img.scan and model.txt.scan and model.img.width == 1024 and model.img.patch_size == (14, 14)


def test_header_is_plain_c_and_a_c_program_links(tmp_path):
  """The boundary is a C ABI: include/bv_b200.h must compile as C99 (and C++), and a C program that includes
  it links against libbv_b200.so and can call the entry points that need no GPU."""
  import shutil
  import subprocess
  if shutil.which("gcc") is None:
    pytest.skip("no gcc")
  L.load()
  hdr = os.path.join(ROOT, "include", "bv_b200.h")
  subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-fsyntax-only", "-x", "c", hdr], check=True)
  subprocess.run(["g++", "-std=c++17", "-fsyntax-only", "-x", "c++", hdr], check=True)
  src = tmp_path / "main.c"
  src.write_text('#include <stdio.h>\n#include "bv_b200.h"\n'
                 'int main(void) {\n'
                 '  int rc = bv_colsum(NULL, 1, NULL, 4, 7, 7, NULL);   /* 7 columns: rejected before any launch */\n'
                 '  printf("%d %d %s\\n", bv_version(), rc, bv_last_error_string());\n'
                 '  return 0;\n}\n')
  libdir = os.path.dirname(os.path.abspath(L.LIB_PATH))
  exe = tmp_path / "main"
  subprocess.run(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe),
                  "-L", libdir, "-lbv_b200", f"-Wl,-rpath,{libdir}"], check=True)
  out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split(None, 2)
  assert out[0] == "100" and int(out[1]) < 0 and len(out[2].strip()) > 0


def test_bench_refuses_to_run_the_product_arm_without_a_gpu():
  """No CPU fallback: the product arm of bench.py exits non-zero on a box without a GPU instead of timing
  something else (the reference arm is the only thing that may run on the host cores)."""
  import subprocess
  import sys
  import torch
  if torch.cuda.is_available():
    pytest.skip("a GPU is present")
  r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1",
                      "--no-cpu-baseline", "--no-gpu-baseline"], capture_output=True, text=True, timeout=600)
  assert r.returncode != 0 and r.stdout.strip() == "" and "needs a GPU" in r.stderr


@pytest.mark.gpu
def test_bench_dumps_what_the_last_timed_step_returned(tmp_path):
  """`bench.py --dump-outputs DIR`: the last timed step's measurements, the optimizer's step count (warm-up +
  --steps updates, so --steps sets the timed steps) and a fixed sample of the train state, as float32 /
  float64 .npy files of at most 64 MB in all."""
  import json
  import subprocess
  import sys
  import numpy as np
  r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "3",
                      "--per-gpu-batch", "64", "--no-cpu-baseline", "--no-gpu-baseline",
                      "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900)
  assert r.returncode == 0, r.stderr[-2000:]
  line = json.loads(r.stdout.strip().splitlines()[-1])
  out = {p.stem: np.load(p) for p in tmp_path.iterdir()}
  assert set(out) == {"training_loss", "l2_grads", "l2_params", "l2_updates", "opt_count",
                      "params", "grads", "adam_mu", "adam_nu"}
  assert sum(p.stat().st_size for p in tmp_path.iterdir()) <= 64 << 20
  assert all(a.dtype in (np.float32, np.float64) and np.isfinite(a).all() for a in out.values())
  assert float(out["opt_count"]) == line["warmup"] + line["steps"] == 5
  assert out["params"].shape == out["grads"].shape == out["adam_mu"].shape == out["adam_nu"].shape == (1 << 21,)
  assert float(out["training_loss"]) > 0 and float(out["l2_params"]) > 0 and np.any(out["grads"] != 0)


def test_reference_arm_prints_the_contract_line():
  """`bench.py --impl reference`: the oracle port on the host cores, one JSON line with the same metric /
  unit / config keys as the product arm plus impl, cpu_baseline and an e2e block with zero copies."""
  import json
  import subprocess
  import sys
  r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                      "--warmup", "1"], capture_output=True, text=True, timeout=900)
  assert r.returncode == 0, r.stderr[-2000:]
  line = json.loads(r.stdout.strip().splitlines()[-1])
  assert line["impl"] == "reference" and line["metric"] == "siglip_vit_b16_pairs_per_sec" and line["unit"] == "pairs/s"
  assert line["higher_is_better"] is True and line["steps"] == 1 and line["value"] > 0
  assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["value"] == line["value"]
  assert line["cpu_baseline"]["cores"] >= 1 and "sample" in line["cpu_baseline"]
  assert line["e2e"] == {"value": line["value"], "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
  assert "workload" in line["config"] and "model" not in line["config"]
