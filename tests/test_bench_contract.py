"""bench.py's contract with the driver, as far as it can be checked without a GPU: the reference arm
(`--impl reference`, the CPU path on the host cores) prints exactly ONE line on stdout, a JSON object with the
keys the driver reads, and under torchrun only rank 0 prints (the missing-GPU behaviour of the product path is
covered by tests/test_abi.py)."""
import json
import os
import subprocess
import sys

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")


def run_bench(*args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + list(args), capture_output=True, text=True,
                          cwd=ROOT, env=e, timeout=600)


def test_reference_arm_prints_one_json_line():
    r = run_bench("--impl", "reference", "--steps", "1", "--warmup", "0", "--images", "4", "--no-reference-em")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["n_gpus"] == 1
    assert d["metric"].startswith("images/sec") and d["unit"] == "images/s" and d["value"] > 0
    assert d["steps"] == 1 and d["warmup"] == 0 and d["vs_baseline"] is None
    assert "workload" in d["config"] and "model" not in d["config"]
    assert d["cpu_baseline"]["kind"] in ("port", "reference") and d["cpu_baseline"]["cores"] >= 1
    assert d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_other_ranks_print_nothing():
    r = run_bench("--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0",
                  env={"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"})
    assert r.returncode == 0, r.stderr[-2000:]
    assert r.stdout.strip() == ""


import pytest  # noqa: E402


def test_steps_must_be_positive_and_dump_needs_the_gpu_arm():
    r = run_bench("--impl", "reference", "--steps", "0")
    assert r.returncode != 0 and "--steps" in r.stderr
    r = run_bench("--impl", "reference", "--dump-outputs", "unused")
    assert r.returncode != 0 and "--dump-outputs" in r.stderr


def test_dump_outputs_zeroes_undefined_entries_and_stays_under_the_limit(tmp_path, monkeypatch):
    import numpy as np
    import bench
    n = np.array([30, 0, 75, 12, 51, 9, 64])
    off = np.concatenate([[0], np.cumsum(n)]).astype(np.int32)
    status = np.array([0, 2, 0, 0, 1, 0, 0], np.int32)
    n_vp = np.array([3, 0, 2, 5, 0, 1, 4], np.int32)

    def result(junk):
        """What the library returns, with `junk` wherever it leaves an entry undefined."""
        B, M = len(n), 64
        r = {"status": status, "n_vp": np.where(status == 0, n_vp, junk), "iterations": np.where(status == 0, 7, junk),
             "vp": np.full((B, M, 3), float(junk)), "sigma": np.full((B, M), float(junk)),
             "counts": np.full((B, M), junk, np.int32), "counts_weighted": np.full((B, M), float(junk)),
             "vp_assoc": np.full(off[-1] + 5, junk, np.int32)}
        for b in range(B):
            if status[b] == 0:
                for k in ("vp", "sigma", "counts", "counts_weighted"):
                    r[k][b, :n_vp[b]] = b + 1
                r["vp_assoc"][off[b]:off[b + 1]] = np.arange(n[b]) % (n_vp[b] + 1) - 1
        return r

    a, b, g = tmp_path / "a", tmp_path / "b", tmp_path / "gathered"
    bench.dump_outputs(str(a), result(13), off)
    bench.dump_outputs(str(b), result(-99), off)
    # pipeline.gather_raw's layout: line associations in rank-major order, image i's at assoc_start[i]
    r, order = result(13), [3, 0, 6, 1, 5, 2, 4]
    starts = np.empty(len(n), np.int64)
    starts[order] = np.concatenate([[0], np.cumsum(n[order])])[:-1]
    r["vp_assoc"] = np.concatenate([r["vp_assoc"][off[i]:off[i + 1]] for i in order])
    r["assoc_start"] = starts
    bench.dump_outputs(str(g), r, off)
    names = sorted(os.listdir(a))
    assert names == sorted(k + ".npy" for k in ("image_index", "status", "n_vp", "iterations", "vp", "sigma", "counts",
                                                "counts_weighted", "vp_assoc"))
    for f in names:
        x = np.load(a / f)
        assert x.dtype == np.float64
        np.testing.assert_array_equal(x, np.load(b / f))
        np.testing.assert_array_equal(x, np.load(g / f))
    assert np.load(a / "vp_assoc.npy").shape == (off[-1],)
    # above the limit: a fixed sample of whole images
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 8 * (4 + 6 * 64) * 3 + 8 * 200)
    s = tmp_path / "sample"
    bench.dump_outputs(str(s), result(13), off)
    idx = np.load(s / "image_index.npy").astype(int)
    assert 0 < len(idx) < len(n)
    assert sum(np.load(s / f).nbytes for f in names) <= bench.DUMP_LIMIT_BYTES
    np.testing.assert_array_equal(np.load(s / "vp.npy"), np.load(a / "vp.npy")[idx])


@pytest.mark.gpu
def test_gpu_arm_prints_one_json_line_with_the_contract_keys(tmp_path):
    import numpy as np
    r = run_bench("--steps", "3", "--warmup", "3", "--images", "16", "--cpu-sample", "1", "--no-reference-em",
                  "--dump-outputs", str(tmp_path))
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["n_gpus"] == 1 and d["steps"] == 3 and d["warmup"] == 3 and d["value"] > 0 and d["gpu_launches"] > 0
    assert d["e2e"]["value"] > 0 and d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0
    rf = d["roofline"]
    assert rf["bound"] in ("hbm", "tensor") and rf["peak"] > 0 and abs(rf["frac"] - rf["achieved"] / rf["peak"]) < 1e-9
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["value"] > 0
    assert set(d["clocks"]) >= {"sm_mhz", "sm_max_mhz", "reasons"}
    assert "workload" in d["config"] and d["images_with_vps"] > 0
    # the dumped result of the last step: every image, and as many with VPs as the serial leg found
    status, n_vp, vp = (np.load(tmp_path / (k + ".npy")) for k in ("status", "n_vp", "vp"))
    assert status.shape == (16,) and int(np.sum(status == 0)) == d["images_with_vps"]
    ok = np.flatnonzero(status == 0)
    assert np.all(n_vp[ok] > 0)
    np.testing.assert_allclose(np.linalg.norm(vp[ok[0], :int(n_vp[ok[0]])], axis=1), 1.0, rtol=1e-9)
