"""bench.py contract on CPU: the reference arm (`--impl reference`: the unmodified reference staged in oracle/_ref or, when
absent, the oracle port, on host cores) prints ONE JSON line with the keys the driver reads.  (The B200 arm needs a GPU; its
line is checked by the driver's own run.)"""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "train", "--steps", "1",
                        "--warmup", "1"], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip().startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "captions_per_sec" and d["unit"] == "captions/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 1
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["vs_baseline"] is None
    assert d["config"]["workload"].startswith("train_step")
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and abs(cb["value"] - d["value"]) < 1e-6 * d["value"]
    assert "bounded sample of 16 captions" in cb["sample"] and "bounded sample of 16 captions" in d["config"]["workload"]
    assert d["config"]["device"] == "cpu" and d["dtype"] == "f32"
    e = d["e2e"]
    assert e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0 and e["unit"] == d["unit"]
    assert abs(e["value"] - d["value"]) < 1e-6 * d["value"]


def test_dump_outputs_arrays(tmp_path):
    """--dump-outputs: float32 / float64 files, large outputs as a fixed seeded sample, decoded captions padded to arrays"""
    import numpy as np
    import torch
    import bench
    x = torch.randn(3 * bench.DUMP_SAMPLE)
    a = bench.dump_array(x)
    assert a.shape == (bench.DUMP_SAMPLE,) and a.dtype == np.float32 and np.array_equal(a, bench.dump_array(x.clone()))
    assert bench.dump_array(torch.ones(2, 3, dtype=torch.bfloat16)).shape == (2, 3)
    assert bench.dump_array(torch.ones(3, dtype=torch.float64)).dtype == np.float64
    c = bench.CFG["greedy"]
    n, S, L = 3, c["S"], c["L"]
    g = torch.Generator().manual_seed(0)
    t = {"_dims": (n, 1, S, L), "fin_count": torch.ones(n, dtype=torch.int32), "fin_len": torch.tensor([[2], [0], [S + 1]], dtype=torch.int32),
         "fin_score": torch.randn(n, 1, generator=g), "fin_ppl": torch.rand(n, 1, generator=g),
         "fin_tokens": torch.randint(0, c["V"], (n, 1, S + 1), generator=g, dtype=torch.int32),
         "fin_asrc": torch.arange(n, dtype=torch.int32).reshape(n, 1, 1).expand(n, 1, S + 1).contiguous(),
         "alpha_all": torch.rand(S + 1, n, L, generator=g)}
    out = bench.decode_outputs(t, c)
    assert out["tokens"].shape == (n, S + 1) and out["tokens"][0, :2].tolist() == t["fin_tokens"][0, 0, :2].tolist()
    assert (out["tokens"][0, 2:] == -1).all() and (out["tokens"][1] == -1).all() and out["lengths"].tolist() == [2, 0, S + 1]
    assert out["alphas"].shape == (n, S + 1, L) and np.array_equal(out["alphas"][2], t["alpha_all"][:, 2].numpy())
    bench.write_outputs(str(tmp_path), {"greedy": out})
    assert sorted(os.listdir(tmp_path)) == ["greedy.%s.npy" % k for k in sorted(out)]
    assert all(np.load(os.path.join(tmp_path, f)).dtype in (np.float32, np.float64) for f in os.listdir(tmp_path))
