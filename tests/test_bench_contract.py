"""bench.py's driver contract on the CPU: the reference arm (`--impl reference`: the restated CPU prover of oracle/) prints ONE
JSON line with the keys the driver reads, and both arms build `config` from the same function (identical dicts)."""
import json, os, subprocess, sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _reference_line(*extra):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1", *extra],
                         capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, out.stdout[-2000:]
    return json.loads(lines[0])


def test_reference_arm_prints_the_contract_line():
    d = _reference_line()
    assert d["impl"] == "reference" and d["metric"] == "proofs_per_sec" and d["unit"] == "proofs/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["steps"] == 1 and d["warmup"] == 1 and d["n_gpus"] == 1 and d["gpu_launches"] == 0
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "restated halo2_proofs 0.2.0" in cb["sample"]
    assert 0.5 < d["cpu_native"]["native_share"] <= 1.0            # the C arithmetic, not the Python driver, is what is timed
    assert d["one_thread"]["value"] > 0 and d["one_thread"]["value"] <= d["value"] * 1.5
    assert d["config"]["workload"].startswith("batched Shot proofs (k=11, IPA/Pasta)")


def test_both_arms_share_the_config_dict():
    sys.path.insert(0, ROOT)
    import bench
    argv, sys.argv = sys.argv, ["bench.py"]
    try:
        args = bench.parse()
    finally:
        sys.argv = argv
    for name in ("shot", "board", "msm", "ntt"):
        args.workload = name
        a, b = bench.WORKLOADS[name](args), bench.WORKLOADS[name](args)
        assert bench.config_for(a) == bench.config_for(b) and "workload" in bench.config_for(a)


def test_dump_outputs_exact_bytes_and_a_seeded_sample_within_the_limit(tmp_path, monkeypatch):
    """--dump-outputs: every item's bytes exactly in float32; over the size limit, the same seeded sample of whole items."""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    small = np.arange(3 * 4, dtype=np.uint64).reshape(3, 4) * 0x0102030405060708
    bench.dump_outputs({"small": small}, str(tmp_path / "a"))
    got = np.load(tmp_path / "a" / "small.npy")
    assert got.dtype == np.float32 and np.array_equal(got, small.view(np.uint8).reshape(3, 32))
    monkeypatch.setattr(bench, "DUMP_LIMIT", 1 << 16)
    big = np.repeat(np.arange(4000, dtype="<u2")[:, None], 8, axis=1)               # item i: 16 bytes that encode i
    other = np.arange(4000 * 2, dtype=np.uint32).reshape(4000, 2)
    for d in ("b", "c"):
        bench.dump_outputs({"big": big, "other": other}, str(tmp_path / d))
    files = sorted((tmp_path / "b").iterdir())
    assert sum(f.stat().st_size for f in files) <= 1 << 16
    rows = np.load(tmp_path / "b" / "big.npy").astype(np.uint8).view("<u2")
    assert 0 < len(rows) < 4000 and (rows == rows[:, :1]).all() and (np.diff(rows[:, 0]) > 0).all()
    for f in files:
        assert np.array_equal(np.load(f), np.load(tmp_path / "c" / f.name))
