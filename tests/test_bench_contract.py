"""bench.py contract: the reference arm prints one JSON line with the agreed keys, the product arm refuses
to run without a GPU (no CPU fallback), and --dump-outputs writes the result of the last timed step."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT


def test_reference_arm_json_line():
    from oracle import build
    if build.ref_bin_dir() is None:
        pytest.skip("GenomeTester4 binaries not installed (oracle/_ref/bin)")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                        "--warmup", "0", "--samples", "12", "--ref-genome-len", "6000"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "k-mers/s" and line["higher_is_better"] is True
    assert line["value"] > 0 and line["cpu_baseline"]["value"] == line["value"]
    assert line["cpu_baseline"]["kind"] in ("reference", "port") and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"] == {"value": line["value"], "unit": "k-mers/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in line["config"] and line["vs_baseline"] is None


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                        "--warmup", "0"], capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_product_arm_needs_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1"], capture_output=True,
                       text=True, timeout=300, cwd=ROOT)
    assert r.returncode != 0 and "no CPU fallback" in (r.stderr + r.stdout)


def test_steps_below_one_are_refused():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True,
                       text=True, timeout=120, cwd=ROOT)
    assert r.returncode == 2 and "--steps" in r.stderr


def _load_dump(d):
    return {fn[:-4]: np.load(os.path.join(d, fn)) for fn in os.listdir(d)}


def test_dump_outputs_float64_and_bounded(tmp_path):
    import bench
    from phenotypeseeker_b200.pipeline import PhenoResult
    rng = np.random.default_rng(3)
    res = []
    for j, n in enumerate((700, 0, 300)):
        res.append(PhenoResult(f"ph{j}", np.sort(rng.choice(1 << 32, n, replace=False)).astype(np.uint64),
                               np.arange(n, dtype=np.uint64), rng.random(n), rng.random(n), rng.random(n), rng.random(n),
                               rng.integers(2, 60, n).astype(np.uint32), presence=rng.integers(0, 2, (n, 70)).astype(np.uint8)))
    names = {"union_kmers", "survivor", "pheno", "kmer", "row", "stat", "p", "mean_x", "mean_y", "n_with", "rowbits"}
    bench.dump_outputs(str(tmp_path / "all"), 12345, res)
    full = _load_dump(tmp_path / "all")
    assert set(full) == names and all(a.dtype == np.float64 for a in full.values())
    assert full["union_kmers"].tolist() == [12345.0] and full["survivor"].tolist() == list(range(1000))
    assert np.array_equal(full["kmer"], np.concatenate([r.kmer for r in res]).astype(np.float64))
    assert np.array_equal(full["rowbits"], np.concatenate([r.rowbits for r in res]).astype(np.float64))
    assert full["pheno"].tolist() == [0.0] * 700 + [2.0] * 300
    # over the limit: the same seeded sample every time, consistent across the files, within the limit
    limit = 64 << 10
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), 12345, res, limit=limit)
    a, b = _load_dump(tmp_path / "a"), _load_dump(tmp_path / "b")
    assert sum(os.path.getsize(tmp_path / "a" / f"{n}.npy") for n in names) <= limit
    idx = a["survivor"].astype(np.int64)
    assert 0 < len(idx) < 1000 and (np.diff(idx) > 0).all()
    for name in names:
        assert np.array_equal(a[name], b[name]), name
        if name not in ("union_kmers", "survivor"):
            assert np.array_equal(a[name], full[name][idx]), name


@pytest.mark.gpu
def test_bench_dumps_the_result_of_its_last_step(tmp_path):
    """Two runs with the same arguments dump identical arrays, and the dump holds what the JSON line reports."""
    runs = []
    for d in ("one", "two"):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--config", "1", "--samples", "12",
                            "--genome-len", "40000", "--steps", "2", "--warmup", "3", "--no-cpu-baseline",
                            "--dump-outputs", str(tmp_path / d)], capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert r.returncode == 0, r.stderr[-2000:]
        runs.append((json.loads(r.stdout.strip().splitlines()[-1]), _load_dump(tmp_path / d)))
    (line, dump), (_, dump2) = runs
    assert line["steps"] == 2
    assert dump["union_kmers"].tolist() == [line["config"]["union_kmers"]]
    assert len(dump["kmer"]) == len(dump["survivor"]) == line["config"]["survivors_read_back"] > 0
    assert (dump["p"] < 0.05).all() and (np.diff(dump["kmer"]) > 0).all()
    for name, a in dump.items():
        assert np.array_equal(a, dump2[name]), name
