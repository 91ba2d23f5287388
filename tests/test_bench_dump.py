"""bench.py --dump-outputs: the arrays of the last timed step of every leg, checked against the CPU oracle on the same seeded inputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from tools import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BENCH = os.path.join(ROOT, "bench.py")


def kp_columns(kps):
    return np.stack([kps[f].astype(np.float32) for f in kps.dtype.names], axis=-1)


@pytest.mark.parametrize("args", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]])
def test_bench_rejects_arguments_it_cannot_honour(args):
    res = subprocess.run([sys.executable, BENCH] + args, capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert res.returncode == 2 and res.stdout == "", res.stdout + res.stderr


@pytest.mark.gpu
def test_dump_outputs_hold_the_last_timed_step(tmp_path):
    from oracle import pyoracle
    from tests.matcher_cases import GRID
    steps = 3
    res = subprocess.run([sys.executable, BENCH, "--steps", str(steps), "--warmup", "1", "--quick", "--no-c5", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stderr[-3000:]
    assert json.loads(res.stdout)["steps"] == steps
    out = {p.name[:-4]: np.load(p) for p in tmp_path.glob("*.npy")}
    assert set(out) == {"orb_counts", "orb_keypoints", "orb_descriptors", "matcher_matches12", "matcher_prev_matched", "matcher_nmatches",
                        "ba_poses", "ba_points", "ba_chi2"}
    assert all(a.dtype in (np.float32, np.float64) for a in out.values())
    assert sum(a.nbytes for a in out.values()) <= 64 << 20

    # ORB: the last step extracts input batch (steps - 1) mod 8, i.e. the seeded frames rolled right by 7 px per batch index
    assert out["orb_keypoints"].shape == (64, 1000, 7) and out["orb_descriptors"].shape == (64, 1000, 32)
    orb = pyoracle.OrbOracle(1000, 1.2, 8, 20)
    for f in (0, 37):
        img = np.ascontiguousarray(np.roll(synth.orb_frame(1000 + f), 7 * ((steps - 1) % 8), axis=1))
        ko, do_ = orb.extract(img)
        n = len(ko)
        assert out["orb_counts"][f] == n
        np.testing.assert_array_equal(out["orb_keypoints"][f, :n], kp_columns(ko))
        np.testing.assert_array_equal(out["orb_descriptors"][f, :n], do_.astype(np.float32))
        assert not out["orb_keypoints"][f, n:].any() and not out["orb_descriptors"][f, n:].any()

    # matcher: the last timed pair is pair 7 of (frame, shifted frame)
    a = synth.orb_frame(2007)
    k1, d1 = orb.extract(a)
    k2, d2 = orb.extract(np.ascontiguousarray(np.roll(a, (3 + 7 % 3, -5 + 7 % 4), axis=(0, 1))))
    prev = np.stack([k1["x"], k1["y"]], axis=1).astype(np.float32)
    n_o, m_o, prev_o = pyoracle.match_by_window(k1, d1, k2, d2, prev, GRID, 20, 1, 0, 8, 0.9)
    np.testing.assert_array_equal(out["matcher_nmatches"], [n_o])
    np.testing.assert_array_equal(out["matcher_matches12"], m_o.astype(np.float32))
    np.testing.assert_array_equal(out["matcher_prev_matched"], prev_o)

    # local BA: optimize(10) of configs[3]
    ob = pyoracle.BAOracle(synth.ba_config("C4"))
    _, st_o = ob.optimize(10)
    po, lo = ob.get()
    np.testing.assert_allclose(out["ba_chi2"], st_o["chi2_after"], rtol=1e-8)
    np.testing.assert_allclose(out["ba_poses"], po, atol=1e-7)
    np.testing.assert_allclose(out["ba_points"], lo, atol=1e-6)
