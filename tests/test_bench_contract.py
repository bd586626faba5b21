"""CPU tests of bench.py's host-side pieces: the C5a input generator, the HBM-peak lookup, the clock-sample parser and the
reference arm's JSON line (which runs entirely on the CPU)."""
import json
import os
import subprocess
import sys
import time

import numpy as np
import pytest

from conftest import ROOT

sys.path.insert(0, ROOT)
import bench  # noqa: E402


def test_splitmix64_sequence_is_pinned():
    """SURVEY 8(d) C5a: a_k = 0.5 + 3.5 u_k, u_k = k-th output of splitmix64(seed = 20261017) / 2^64."""
    u = bench._splitmix64_unit(20261017, 4)
    assert np.all((u >= 0) & (u < 1)) and len(set(u)) == 4
    assert np.array_equal(u, bench._splitmix64_unit(20261017, 8)[:4])            # a stream, not a function of n
    # first output of the published splitmix64 for seed 0 is 0xE220A8397B1DCDAF
    assert bench._splitmix64_unit(0, 1)[0] == 0xE220A8397B1DCDAF / 2.0 ** 64


def test_hbm_peak_falls_back_to_the_recipe_value(tmp_path, monkeypatch):
    assert bench._hbm_peak() > 1000.0
    monkeypatch.setattr(bench, "ROOT", str(tmp_path))                            # no MEASURED_PEAKS.json there
    assert bench._hbm_peak() == 6459.0


class _Dummy:
    def terminate(self):
        pass


def test_clock_sampler_selects_the_timed_region():
    s = bench.ClockSampler(0)
    s.proc = _Dummy()
    t = time.time()
    mk = lambda sm, *flags: f"0, {sm}, 1965, 700.0, 0x0, " + ", ".join(flags)      # noqa: E731
    idle = mk(345, "Not Active", "Not Active", "Not Active", "Not Active")
    busy = mk(1965, "Not Active", "Not Active", "Not Active", "Not Active")
    capped = mk(1800, "Not Active", "Not Active", "Not Active", "Active")
    s.lines = [(t - 10, idle), (t - 5, busy), (t - 2.0, busy), (t - 1.5, capped), (t - 1.0, busy)]
    c = s.stop(t - 2.2, t - 0.8)
    assert c["samples"] == 3 and c["sm_mhz"] == 1965.0 and c["sm_max_mhz"] == 1965.0
    assert c["reasons"] == ["sw_power_cap"] and c["window"] == "timed region"
    s.lines = [(t - 5, busy), (t - 4, busy)]
    c = s.stop(t - 1.0, t - 0.5)                                                  # nothing inside: warm-up samples are used
    assert c["samples"] == 2 and c["window"] == "warm-up + timed region"


def test_dump_outputs_writes_what_the_caller_received(tmp_path):
    """`bench.py --dump-outputs DIR`: the results of a solve_batch call as float64 .npy files of finite values, atoms in input order, the
    levels of all atoms concatenated with their counts per (atom, spin)."""
    import dftatom_b200 as D
    li = D.Result(D.Options(3, 10, 10.0, 0.01, 0.5, 1), 0, 31, [[(1, 0, 1, 0, -1.8), (2, 0, 1, 1, -0.1)], [(1, 0, 1, 0, -1.7)]],
                  [[(2, 0, 1, 1, -0.1), (1, 0, 1, 0, -1.8)], [(1, 0, 1, 0, -1.7)]], -7.3, 7.2, 4.0, -17.0, -1.5)
    he = D.Result(D.Options(2, 10, 10.0, 0.01, 0.5, 0), 1, 100, [[(1, 0, 2, 0, -0.57)]], [[(1, 0, 2, 0, -0.57)]], -2.8, 2.7, 2.0, -6.6, -0.9)
    bench.dump_outputs([li, he], str(tmp_path))
    out = {p.stem: np.load(p) for p in tmp_path.iterdir()}
    assert sorted(out) == ["eigenvalues", "energies", "levels", "n_levels", "n_steps", "sorted_levels", "status"]
    assert all(x.dtype == np.float64 and np.isfinite(x).all() for x in out.values())
    assert out["energies"].tolist() == [[-7.3, 7.2, 4.0, -17.0, -1.5], [-2.8, 2.7, 2.0, -6.6, -0.9]]
    assert out["n_steps"].tolist() == [31, 100] and out["status"].tolist() == [0, 1]
    assert out["n_levels"].tolist() == [[2, 1], [1, 0]]
    assert out["eigenvalues"].tolist() == [-1.8, -0.1, -1.7, -0.57]
    assert out["levels"].tolist() == [[1, 0, 1, 0], [2, 0, 1, 1], [1, 0, 1, 0], [1, 0, 2, 0]]
    assert out["sorted_levels"][:2].tolist() == [[2, 0, 1, 1, -0.1], [1, 0, 1, 0, -1.8]] and out["sorted_levels"].shape == (4, 5)
    assert sum(x.nbytes for x in out.values()) < 64 << 20
    # a non-finite result is refused, and nothing is written
    broken = D.Result(D.Options(5, 10, 10.0, 0.01, 0.5, 0), 1, 100, [[(1, 0, 2, 0, float("nan"))]], [[(1, 0, 2, 0, float("nan"))]],
                      -24.0, 24.0, 10.0, -60.0, -3.0)
    with pytest.raises(ValueError, match=r"Z = \[5\]"):
        bench.dump_outputs([li, broken], str(tmp_path / "broken"))
    assert not (tmp_path / "broken").exists()


def test_reference_arm_prints_one_json_line():
    """`bench.py --impl reference`: the unmodified reference's CPU solver on the host cores, one JSON line with the arm's keys.
    (One bounded sample; skipped when neither oracle/_ref nor the oracle binary can be run.)"""
    if not (os.path.exists(bench.REF_EXE) or os.path.exists(bench.ORACLE_EXE)):
        pytest.skip("no CPU solver built")
    env = dict(os.environ, RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, env=env, check=True).stdout
    assert out == ""                                                              # ranks other than 0 exit 0 without work
    costs = bench._golden_costs()
    assert len(costs) == 92 and min(costs.values()) > 0
    # rank 0: the pooled sweep (here cut down to two light atoms), value = atoms / wall independent of --steps
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "4", "--warmup", "0", "--ref-atoms", "1,2"],
                         capture_output=True, text=True, env=dict(os.environ, RANK="0"), check=True).stdout
    line = json.loads(out.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "atoms/s" and line["higher_is_better"] is True and line["gpu_launches"] == 0
    cb = line["cpu_baseline"]
    assert cb["complete"] is True and cb["atoms_finished"] == 2 and cb["kind"] in ("reference", "port") and cb["cores"] >= 1
    assert abs(line["value"] - 2.0 / cb["wall_s"]) < 1e-9 and abs(line["ms_per_step"] - cb["wall_s"] * 1e3 / 4) < 1e-6
    assert line["e2e"] == dict(value=line["value"], unit="atoms/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0)
