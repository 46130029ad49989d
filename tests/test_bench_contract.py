"""bench.py's reference arm runs on the CPU: check the JSON contract of the line the driver parses."""
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_line_has_the_contract_keys():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "ffn_block_tokens_per_sec" and d["unit"] == "tokens/s"
    assert d["steps"] == 1
    for k in ("value", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data",
              "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["value"] > 0 and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_dump_outputs_fits_the_budget_and_samples_the_same_rows(tmp_path):
    import bench
    gen = torch.Generator().manual_seed(0)
    flat = torch.randn(8192, 4096, generator=gen)           # one 11B prefill output in fp32: 128 MiB, over the budget
    flat[:, 0] = torch.arange(8192)                         # each row carries its index
    small = torch.randn(4096, generator=gen).bfloat16()
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"y": flat.view(4, 2048, 4096), "grad_gamma": small})
    assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) <= 64_000_000
    g = np.load(tmp_path / "a" / "grad_gamma.npy")
    assert g.dtype == np.float32 and np.array_equal(g, small.float().numpy())
    ya, yb = np.load(tmp_path / "a" / "y.npy"), np.load(tmp_path / "b" / "y.npy")
    # the room grad_gamma does not use goes to y
    assert ya.dtype == np.float32 and ya.shape == ((bench.DUMP_BUDGET_BYTES - small.numel() * 4) // (4096 * 4), 4096)
    assert np.array_equal(ya, yb)
    idx = [int(r[0]) for r in ya]
    assert idx == sorted(set(idx)) and np.array_equal(ya, flat[idx].numpy())


def test_product_path_does_not_import_the_oracle():
    """The oracle is test infrastructure: nothing under the package (or the extension shims) may import it."""
    pkg = os.path.join(ROOT, "llama-3.2-multimodal_b200")
    files = [os.path.join(pkg, f) for f in os.listdir(pkg) if f.endswith(".py")]
    files += [os.path.join(ROOT, f) for f in ("rmsnorm.py", "swiglu_fused.py", os.path.join("llama32_b200", "__init__.py"))]
    for f in files:
        text = open(f).read()
        for line in text.splitlines():
            s = line.strip()
            if s.startswith(("import ", "from ")):
                assert "oracle" not in s, f"{f}: {s}"
