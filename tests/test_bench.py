"""bench.py as a tool: --dump-outputs stores what the timed path computed, exactly, --steps is checked, and a run leaves the source tree as it was."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
from conftest import ROOT

import bench


def _load_limbs(path):
    a = np.load(path)
    assert a.dtype == np.float64 and a.shape[-1] == 2
    return a[..., 0].astype(np.uint64) | (a[..., 1].astype(np.uint64) << np.uint64(32))


def _tree_state(root):
    """Every file (and its mtime) under the directories whose code bench.py runs: where bytecode or build caches would land."""
    state = {}
    for sub in ("kogarashi_b200", "oracle", "tools", "tests"):
        for d, _, files in os.walk(os.path.join(root, sub)):
            for f in files:
                p = os.path.join(d, f)
                state[p] = os.stat(p).st_mtime_ns
    return state


def test_dump_outputs_round_trip(tmp_path):
    aff = np.array([0, 1, 2**32 - 1, 2**32, 2**64 - 1, bench.FR_TOP, 2**63, 2**53 + 1, 1], dtype=np.uint64)
    bench.dump_outputs(str(tmp_path / "out"), {"msm_affine": aff})
    assert sorted(os.listdir(tmp_path / "out")) == ["msm_affine.npy"]
    assert (_load_limbs(tmp_path / "out" / "msm_affine.npy") == aff).all()


def test_steps_must_be_positive():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True, timeout=120)
    assert out.returncode == 2 and "--steps" in out.stderr, out.stdout + out.stderr


@pytest.mark.gpu
def test_dumped_result_is_reproducible_matches_the_oracle_and_leaves_the_tree_untouched(tmp_path):
    """Two runs with the same arguments dump the same bytes; the dumped point is the CPU oracle's MSM of the bench's seeded inputs (bases
    generated on the device from BASE_SEED, numpy scalars); the runs write nothing into the source directories."""
    import kogarashi_b200 as k
    from oracle import oracle as A
    logn = 12
    before = _tree_state(ROOT)
    dumps = []
    for run in range(2):
        d = tmp_path / f"run{run}"
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "3", "--quick", "--logn", str(logn),
                              "--dump-outputs", str(d)], capture_output=True, text=True, timeout=900)
        assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
        line = json.loads([s for s in out.stdout.splitlines() if s.startswith("{")][-1])
        assert line["steps"] == 2 and line["checksum_ok"]
        assert sorted(os.listdir(d)) == ["msm_affine.npy"]
        dumps.append((d / "msm_affine.npy").read_bytes())
    assert dumps[0] == dumps[1]
    n = 1 << logn
    k.init()
    bases = k.Bases.generate(A.BN254_G1, n, seed=bench.BASE_SEED)
    pts = bases.download()
    bases.free()
    exp = A.to_affine(A.BN254_G1, A.msm(A.BN254_G1, pts, bench.scalars_range(0, n)))
    assert (_load_limbs(tmp_path / "run0" / "msm_affine.npy") == exp).all()
    assert _tree_state(ROOT) == before


@pytest.mark.gpu
def test_groth16_workload_honours_steps_and_dumps_the_proof(tmp_path):
    """--workload groth16 times the number of proofs asked for, reports it, and dumps the proof it checked against the discrete logs."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "groth16", "--logm", "10", "--steps", "2", "--warmup", "4",
                          "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    line = json.loads([s for s in out.stdout.splitlines() if s.startswith("{")][-1])
    assert (line["steps"], line["warmup"]) == (2, 4) and "best of 2 after 4 warm-up proofs" in line["timing"]
    assert line["proof_checked_against_discrete_logs"]
    assert sorted(os.listdir(tmp_path)) == ["proof_a.npy", "proof_b.npy", "proof_c.npy"]
    shapes = [_load_limbs(tmp_path / f"proof_{c}.npy").shape for c in "abc"]
    assert shapes == [(9,), (17,), (9,)]
