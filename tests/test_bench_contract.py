"""bench.py's JSON-line contract (CPU side): the reference arm runs here, and the committed round artefact of the
GPU arm carries every key the driver reads."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config"}


def test_reference_arm_prints_one_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--lines", "2000", "--shells", "5",
                          "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert BASE_KEYS <= set(d), BASE_KEYS - set(d)
    assert d["impl"] == "reference" and d["unit"] == "packets/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["cpu_baseline"]["value"] == d["value"] == d["e2e"]["value"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"] and "model" not in d["config"]


def test_committed_gpu_bench_line_has_the_contract_keys():
    path = os.path.join(ROOT, "profiles", "r02_bench_final_default_1e8.json")
    if not os.path.exists(path):
        pytest.skip("the round's final bench line is not committed yet")
    d = json.loads(open(path).read().strip().splitlines()[-1])
    assert BASE_KEYS | {"clocks", "gpu_launches", "e2e", "roofline", "cpu_baseline"} <= set(d)
    assert d["dtype"] == "f64" and d["data"] == "synthetic" and d["scaling"] == "weak" and d["vs_baseline"] is None
    r = d["roofline"]
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(r) and r["bound"] == "hbm" and r["unit"] == "GB/s"
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-12
    e = d["e2e"]
    assert e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0 and 0 < e["value"] < d["value"]
    c = d["cpu_baseline"]
    assert c["kind"] in ("port", "reference") and c["cores"] >= 1 and c["value"] > 0 and c["sample"]
    assert d["gpu_launches"] > 0 and d["warmup"] >= 3
    assert not set(d["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    # a timed step pays for its fresh packets: seed expansion + three ordering kernels + transport + two epilogues
    assert d["gpu_launches"] >= 7 * d["steps"] and e["steps"] == d["steps"]
    # round 2: the BASELINE legs ride in the same line, each with its own e2e / roofline / cpu_baseline / parity
    for k in ("2", "4", "5"):
        leg = d["configs"][k]
        assert leg["value"] > 0 and leg["e2e"]["value"] > 0 and leg["warmup"] >= 3 and leg["scaling"] == "strong"
        assert leg["cpu_baseline"]["value"] > 0 and leg["roofline"]["kernel_ms"] > 0
        p = leg["parity"]
        assert p["counters_equal"] and p["spectrum_l2_vs_oracle"] < 1e-10 and max(p["max_rel_err"].values()) < 1e-10
    assert d["configs"]["4"]["parity"]["virtual_spectrum_l2_vs_oracle"] < 1e-10
    assert d["configs"]["5"]["parity"]["photo_ion_statistics_equal"]
    assert d["parity"]["counters_equal"] and d["parity"]["fused_spectrum_l2_vs_oracle"] < 1e-10
    assert r["traffic"] is not None and r["issue_active_pct"] is not None
    # per-iteration table preparation either side of the path (§8f ranks 3 / 4) rides in the same line
    t = d["tables"]
    assert "error" not in t and t["host_tables"]["ms"] > 0 and t["device_tables"]["ms"] > 0 and t["source_function"]["sweeps"] > 0


def test_formal_integral_work_counter_matches_a_literal_walk():
    """bench.py's count of resonance points / warp sweep steps (the formal integral's roofline numerator) against a literal walk of
    the reference algorithm (populate_intersection_points + the line loop, formal_integral_numba.py:54-118, :472-536)."""
    import numpy as np

    sys.path.insert(0, ROOT)
    import bench
    from tardis_b200 import synthetic as syn

    model = syn.make_model(6, 3000, "downbranch", mu_tau=-3.0, seed=5)
    nu = np.asarray(model.line_list_nu)
    t_exp = float(model.time_explosion)
    freq = np.array([nu[-1] * 0.99, nu[-1] * 1.04, nu[len(nu) // 2], nu[len(nu) // 3] * 1.0001, nu[0] * 0.97, nu[0] * 1.2])
    for points, shells in ((2, -1), (40, 13), (97, 0), (33, -1), (65, 2)):
        got = bench.formal_integral_work(model.r_inner, model.r_outer, t_exp, nu, freq, points, shells)
        n_radii = shells if shells != 0 else max(2 * len(model.r_inner), 80)
        if n_radii > 0:
            radius = np.linspace(model.r_inner[0], model.r_outer[-1], n_radii)
            r_in, r_out = radius[:-1], radius[1:]
        else:
            r_in, r_out = np.asarray(model.r_inner), np.asarray(model.r_outer)
        N, c_inv, inv_t = len(r_in), 3.33564e-11, 1.0 / t_exp
        ip = lambda r, p: np.sqrt(r * r - p * p) * c_inv * inv_t if r > p else 0.0  # noqa: E731
        total, rays, steps = 0, 0, 0
        n_blocks = (points - 1 + 31) // 32
        for f in freq:
            visited = [set() for _ in range(n_blocks)]
            for p_idx in range(1, points):
                p = p_idx * r_out[-1] / (points - 1)
                if p <= r_in[0]:
                    z = [1 - ip(r_out[i], p) for i in range(N)]
                else:
                    off = next((i for i in range(N) if ip(r_out[i], p) != 0), N)
                    z = [0.0] * (2 * (N - off))
                    for i in range(off, N):
                        z[N - i - 1] = 1 + ip(r_out[i], p)
                        z[N + i - 2 * off] = 1 - ip(r_out[i], p)
                if len(z) < 2:
                    continue
                rays += 1
                line = int(np.count_nonzero(nu > f * z[0]))
                for k in range(1, len(z)):
                    while line < len(nu) and nu[line] > f * z[k]:
                        visited[(p_idx - 1) // 32].add(line)
                        total += 1
                        line += 1
            steps += sum(len(v) for v in visited)
        assert got["resonance_points"] == total, (points, shells)
        assert got["rays"] == rays, (points, shells)
        assert got["warp_sweep_steps"] == steps, (points, shells)
        assert got["integrator_shells"] == N


def test_tables_block_plumbing_with_a_stub_engine(monkeypatch):
    """bench.py's `tables` entry (per-iteration table preparation, source function, formal integral with its work count, CPU sample
    and parity) cannot run here -- the product has no CPU path -- so its host-side plumbing runs against a stub engine that answers
    with the ORACLE's numbers: every key the entry promises is there and no side measurement raises."""
    import types

    import numpy as np

    sys.path.insert(0, ROOT)
    import bench
    from oracle import formal_integral_oracle as fio
    from tardis_b200 import engine as engine_mod
    from tardis_b200 import synthetic as syn

    model = syn.make_model(5, 2000, "macroatom", mu_tau=-3.0, seed=3)
    L, S = model.n_lines, model.n_shells
    rng = np.random.default_rng(1)
    tau = np.asarray(model.tau_sobolev)
    att, jblue = rng.random((L, S)) * 1e-6, rng.random((L, S)) * 1e-5
    jred = jblue * np.exp(-tau) + att

    # the stub's source function is the oracle's, on the tables / estimators it hands out (bench.py builds the same atomic data)
    from oracle import opacity_oracle
    from oracle import source_function_oracle as sfo

    atomic = syn.make_atomic_data(model.line_list_nu, 3000, "macroatom", nlte_fraction=0.0)
    plasma = syn.make_plasma_state(atomic, S, model.time_explosion, zero_fraction=0.0, inversion_fraction=0.0, noise=0.0)
    plasma.level_number_density *= 1e-9
    tabs = opacity_oracle.build(atomic, plasma)
    est_jblue, est_edotlu = rng.random((L, S)) * 1e-3, rng.random((L, S)) * 1e-2
    volume = 4.0 / 3.0 * np.pi * (model.r_outer ** 3 - model.r_inner ** 3)
    sf_full = sfo.solve(atomic, tabs["tau_sobolev"], tabs["transition_probabilities"], est_jblue, est_edotlu, float(model.time_explosion), 1.0e5, volume,
                        "macroatom")

    class StubEngine:
        def __init__(self, device):
            self.calls = []

        def download(self, **k):
            return dict(j_blue=est_jblue, edotlu=est_edotlu)

        def __getattr__(self, name):  # everything that only has to be callable
            def call(*a, **k):
                self.calls.append(name)
                return None
            return call

        def solve_source_function(self, want=None, **k):
            return dict(iterations=24, att_S_ul=sf_full["att_S_ul"], Jred_lu=sf_full["Jred_lu"], Jblue_lu=sf_full["Jblue_lu"])

        def download_opacity(self, transition_probabilities=False):
            return dict(tau_sobolev=tabs["tau_sobolev"], beta_sobolev=tabs["beta_sobolev"], transition_probabilities=tabs["transition_probabilities"])

        def formal_integral(self, *, inner_temperature, frequencies, points, interpolate_shells=0, **k):
            o = fio.solve(model.r_inner, model.r_outer, float(model.time_explosion), model.line_list_nu, inner_temperature, frequencies,
                          sf_full["att_S_ul"], sf_full["Jred_lu"], sf_full["Jblue_lu"], tabs["tau_sobolev"], model.electron_density, points, interpolate_shells)
            return dict(luminosity_densities=o["luminosity_densities"], intensities_nu_p=None, interpolation_ms=1.5, integral_ms=20.0)

    monkeypatch.setattr(engine_mod, "Engine", StubEngine)
    # a short frequency grid keeps the oracle's share of this test small
    model.spectrum_frequency_grid = np.linspace(model.line_list_nu[-1] * 1.1, model.line_list_nu[0] * 0.95, 81)
    out = bench.tables_block(types.SimpleNamespace(local_rank=0, peak=6562.6), model, with_cpu=True)
    assert "error" not in out, out.get("error")
    fi = out["formal_integral"]
    assert "error" not in fi, fi.get("error")
    assert fi["n_frequencies"] == 80 and fi["integral_ms"] == 20.0 and fi["frequencies_per_s"] == 80 / 0.02
    assert fi["work"]["resonance_points"] > 0 and fi["work"]["rays"] == 998 * 80
    r = fi["roofline"]
    assert "error" not in r and r["algorithmic_bytes"] == 32 * fi["work"]["resonance_points"] + 8 * fi["work"]["warp_sweep_steps"]
    assert abs(r["x_hbm_peak"] - r["achieved"] / 6562.6) < 1e-12 and 0 < r["lanes_busy_per_sweep_step"] <= 32
    assert fi["cpu_baseline"]["frequencies_per_s"] > 0 and fi["cpu_baseline"]["cores"] == 1
    assert fi["parity"]["max_rel_err_L_nu_vs_oracle"] == 0.0 and fi["parity"]["frequencies_checked"] == 64  # the stub IS the oracle
    dp = out["device_tables"]["parity"]
    assert "error" not in dp and dp["tau_sobolev_bit_identical"] and dp["beta_sobolev_max_rel_err"] == 0.0
    sp = out["source_function"]["parity"]
    assert "error" not in sp, sp.get("error")
    assert sp["shells_checked"] == [0, 2, 4] and all(sp[k]["zero_pattern_equal"] and sp[k]["max_err_over_bar"] <= 1.0 for k in ("att_S_ul", "Jred_lu", "Jblue_lu"))
    assert out["source_function"]["sweeps"] == 24 and out["host_tables"]["ms"] >= 0 and out["device_tables"]["n_levels"] == 3000


def test_dump_outputs_writes_float64_with_a_fixed_sample_of_large_arrays(tmp_path):
    """bench.py --dump-outputs: every array of the result as <name>.npy in float64, counters as one array in sorted-name order, and
    an array above DUMP_SAMPLE entries as the same sorted sample of its flat entries on every call."""
    import numpy as np

    sys.path.insert(0, ROOT)
    import bench

    n = 3 * bench.DUMP_SAMPLE
    res = {"output_nus": np.arange(n, dtype=np.float64), "j": np.linspace(1.0, 2.0, 20), "j_blue": np.arange(n, dtype=np.float64).reshape(-1, 3),
           "photo_ion_estimator_statistics": np.arange(12, dtype=np.int64).reshape(3, 4), "counters": {"n_line_steps": 7, "n_boundary_events": 5}}
    for d in ("a", "b"):
        bench.dump_outputs(res, str(tmp_path / d))
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == ["counters.npy", "j.npy", "j_blue.npy", "output_nus.npy", "photo_ion_estimator_statistics.npy"]
    for name in names:
        a, b = np.load(tmp_path / "a" / name), np.load(tmp_path / "b" / name)
        assert a.dtype == np.float64 and np.array_equal(a, b), name
    assert np.array_equal(np.load(tmp_path / "a" / "counters.npy"), [5.0, 7.0])
    assert np.array_equal(np.load(tmp_path / "a" / "j.npy"), res["j"])
    assert np.array_equal(np.load(tmp_path / "a" / "photo_ion_estimator_statistics.npy"), res["photo_ion_estimator_statistics"])
    s = np.load(tmp_path / "a" / "output_nus.npy")  # the values are their own indices: a sorted sample without repeats
    assert s.shape == (bench.DUMP_SAMPLE,) and np.all(np.diff(s) > 0) and s[-1] < n
    assert np.array_equal(np.load(tmp_path / "a" / "j_blue.npy"), s)  # same size -> same flat positions


def test_dump_outputs_is_refused_on_the_reference_arm(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs", str(tmp_path / "d")],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode != 0 and "--dump-outputs" in out.stderr and not (tmp_path / "d").exists()


@pytest.mark.gpu
def test_bench_dumps_identical_inputs_outputs_on_every_run(tmp_path):
    """A small headline run twice with --dump-outputs: the JSON line reports the requested steps, the dump stays within 64 MB of
    float64 arrays, and the same arguments give the same outputs (integer work exactly, floating-point sums to the last bits)."""
    import numpy as np

    args = ["--gpus", "1", "--steps", "2", "--warmup", "1", "--packets", "200000", "--lines", "20000", "--shells", "10", "--mu-tau", "-4.5",
            "--legs", "none", "--no-cpu-baseline", "--no-tables", "--no-scan-reference", "--no-device-source"]
    for d in ("a", "b"):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args, "--dump-outputs", str(tmp_path / d)],
                             capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-3000:]
        line = json.loads([ln for ln in out.stdout.splitlines() if ln.startswith("{")][-1])
        assert line["steps"] == 2 and line["warmup"] == 1 and line["gpu_launches"] >= 7 * 2
    names = sorted(os.listdir(tmp_path / "a"))
    assert {"output_nus.npy", "output_energies.npy", "j.npy", "nu_bar.npy", "j_blue.npy", "edotlu.npy", "counters.npy"} <= set(names)
    assert sum(os.path.getsize(tmp_path / "a" / n) for n in names) <= 64 << 20
    for name in names:
        a, b = np.load(tmp_path / "a" / name), np.load(tmp_path / "b" / name)
        assert a.dtype == np.float64 and a.shape == b.shape, name
        np.testing.assert_allclose(a, b, rtol=1e-12, atol=0, err_msg=name)
    assert np.array_equal(np.load(tmp_path / "a" / "counters.npy"), np.load(tmp_path / "b" / "counters.npy"))
    assert np.array_equal(np.load(tmp_path / "a" / "output_nus.npy"), np.load(tmp_path / "b" / "output_nus.npy"))
    assert np.load(tmp_path / "a" / "output_nus.npy").shape == (200000,)
