"""The reference arm of bench.py (`--impl reference`: the CPU oracle port on the host cores) runs without a GPU and prints
ONE JSON line carrying the contract's keys."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    proc = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                          cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
    assert proc.returncode == 0, proc.stderr[-2000:]
    lines = [l for l in proc.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, "stdout must hold exactly one line"
    line = json.loads(lines[0])
    assert line["impl"] == "reference" and line["unit"] == "samples/s" and line["higher_is_better"] is True
    assert line["metric"].startswith("diffusion samples/sec") and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1 and line["cpu_baseline"]["value"] == line["value"]
    assert line["e2e"] == {"value": line["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in line["config"] and line["steps"] == 1


def test_per_kernel_roofline_of_a_recorded_bench_line():
    """bench.py's per-launch roofline (host arithmetic only) on the class times of the committed round-2 line: bytes and
    FLOPs follow the layer dims, every class that ran is reported, and the big launches sit near one of their two roofs."""
    import json
    import os
    import bench
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    line = json.loads(open(os.path.join(root, "profiles", "r2_bench.json")).read().strip().splitlines()[-1])
    n_rows, m_rows = 100 * 4096, 428 * 4096
    fp32 = bench.per_kernel_roofline(line["precisions"]["fp32"]["roofline"]["class_ms_per_round"], n_rows, m_rows, "fp32",
                                     1369.7, 6552.3)
    assert set(fp32) == {"query_out", "v1_hidden", "lit_2", "lit_3", "clause_1", "clause_2", "update_3", "output_2",
                         "pairnorm_clause", "pairnorm_var"}
    c1 = fp32["clause_1"]      # 384 -> 208 columns of hi/lo planes: (384 + 208) * 4 bytes per clause row, 3 * 2 * 384 * 204 FLOPs
    assert abs(c1["hbm_frac"] - m_rows * 592 * 4 / (c1["ms"] * 1e-3) / 1e9 / 6552.3) < 1e-12
    assert abs(c1["tensor_pipe_frac"] - 3 * 2 * m_rows * 384 * 204 / (c1["ms"] * 1e-3) / 1e12 / 1369.7) < 1e-12
    assert c1["bound"] == "hbm" and 0.8 < c1["hbm_frac"] < 0.9
    assert fp32["lit_2"]["bound"] == "tensor" and fp32["lit_2"]["tensor_pipe_frac"] > 0.9
    for name in ("lit_2", "lit_3", "clause_1", "clause_2", "update_3", "pairnorm_clause"):
        assert max(fp32[name]["tensor_pipe_frac"], fp32[name]["hbm_frac"]) > 0.65, name
    bf16 = bench.per_kernel_roofline(line["precisions"]["bf16"]["roofline"]["class_ms_per_round"], n_rows, m_rows, "bf16",
                                     1369.7, 6552.3)
    assert set(bf16) == {"query_out", "lit_3", "clause_2", "update_3", "output_2", "pairnorm_clause", "pairnorm_var"}
    assert bench.per_kernel_roofline({}, n_rows, m_rows, "fp32", 1369.7, 6552.3) == {}


def test_dump_outputs_unpacks_the_packed_assignments(tmp_path, monkeypatch):
    """--dump-outputs: packed 64-bit words (x1 = bit 0 of word 0) come out as one 0/1 float32 row per chain; above the size
    cap the same seeded chains are written every time, with their global indices."""
    import numpy as np
    import bench
    rng = np.random.default_rng(3)
    chains, n_vars = 300, 100
    bits = rng.integers(0, 2, (chains, n_vars))
    packed = np.zeros((chains, 2), dtype=np.uint64)
    for v in range(n_vars):
        packed[:, v // 64] |= bits[:, v].astype(np.uint64) << np.uint64(v % 64)
    latch = rng.integers(-1, 32, chains).astype(np.int32)
    outs = (rng.integers(0, 2, chains).astype(np.uint8), latch, (latch >= 0).astype(np.uint8))
    bench.dump_outputs(str(tmp_path / "all"), n_vars, 0, packed, *outs)
    got = {f[:-4]: np.load(str(tmp_path / "all" / f)) for f in os.listdir(str(tmp_path / "all"))}
    assert set(got) == {"assignment", "is_sat", "latch_step", "sat_any_step", "chain"}
    assert got["assignment"].dtype == np.float32 and np.array_equal(got["assignment"], bits)
    assert np.array_equal(got["latch_step"], latch) and np.array_equal(got["chain"], np.arange(chains))
    monkeypatch.setattr(bench, "DUMP_BYTES", 100 * (4 * (n_vars + 3) + 8))
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), n_vars, 1000, packed, *outs)
    chain = np.load(str(tmp_path / "a" / "chain.npy"))
    assert len(chain) == 100 and np.array_equal(chain, np.load(str(tmp_path / "b" / "chain.npy")))
    assert np.array_equal(np.load(str(tmp_path / "a" / "assignment.npy")), bits[chain.astype(np.int64) - 1000])
