"""Device-side packet source (SURVEY.md §8f rank 1; tardis_b200/csrc/packet_source.cuh).

CPU: (1) the sequential oracle (oracle/packet_source_oracle.c) against golden vectors of the unmodified
`BlackBodySimpleSource.create_packets` and against numpy's `default_rng` itself; (2) the PRODUCT's generator functions --
the very header the CUDA kernel compiles, built for the host by tests/packet_source_shim.cpp and driven chunk by chunk like
the kernel -- against the same, including populations that make the bounded draw reject often.
Bar: seeds, mus, radii, energies bit-identical; nus to 1e-15 (one ulp of `log`).

GPU: the kernel through the C-ABI, in a subprocess (a fault there must not take the parity suite's CUDA context down)."""
import ctypes as C
import glob
import json
import os
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
KB, H = 1.3806488e-16, 6.62606957e-27
NU_RTOL = 1e-15
CASES = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(HERE, "golden", "packet_source_*.npz")))
C_LIGHT = 2.99792458e10


def golden_beta(g):
    """beta of BlackBodySimpleSourceRelativistic (black_body_relativistic.py:122): (radius / time_explosion) / c, or None"""
    return (float(g["radius"]) / float(g["time_explosion"])) / C_LIGHT if "time_explosion" in g.files else None


def relativistic_energy(n, beta):
    """black_body_relativistic.py:168-177 in numpy's own operation order"""
    gamma = 1.0 / np.sqrt(1 - beta**2)
    factor = (2 * beta + 1) / (1 - beta**2)
    return float((np.ones(1) / n * factor / gamma)[0])
EXACT = ("packet_seeds", "initial_mus", "initial_radii", "initial_energies")


def numpy_source(seed, n, pop=2**32 - 1, radius=1.2e15, temperature=1.0e4, l_samples=1000):
    """BlackBodySimpleSource.create_packets restated with numpy's own generator (as tardis_b200.synthetic.make_packets)."""
    rng = np.random.default_rng(seed)
    seeds = rng.choice(pop, n, replace=True).astype(np.int64)
    l_array = np.cumsum(np.arange(1, l_samples, dtype=np.float64) ** -4)
    xis = rng.random((5, n))
    l = l_array.searchsorted(xis[0] * (np.pi**4 / 90.0)) + 1.0
    nus = (-np.log(np.prod(xis[1:], 0)) / l) * (KB * temperature) / H
    return dict(packet_seeds=seeds, initial_nus=nus, initial_mus=np.sqrt(rng.random(n)), initial_radii=np.ones(n) * radius,
                initial_energies=np.ones(n) / n)


def check(got, want):
    for k in EXACT:
        assert np.array_equal(got[k], want[k]), k
    assert got["packet_seeds"].dtype == np.int64
    np.testing.assert_allclose(got["initial_nus"], want["initial_nus"], rtol=NU_RTOL, atol=0)


@pytest.fixture(scope="module")
def shim():
    out = os.path.join(HERE, "_shim", "libpacket_source_shim.so")
    src = os.path.join(HERE, "packet_source_shim.cpp")
    hdr = os.path.join(ROOT, "tardis_b200", "csrc", "packet_source.cuh")
    os.makedirs(os.path.dirname(out), exist_ok=True)
    if not os.path.exists(out) or os.path.getmtime(out) < max(os.path.getmtime(src), os.path.getmtime(hdr)):
        subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-o", out, src], check=True)
    lib = C.CDLL(out)
    lib.shim_create_packets.restype = C.c_int
    lib.shim_create_packets.argtypes = ([C.c_uint64, C.c_uint64, C.c_uint32, C.c_double, C.c_double, C.c_double, C.c_void_p, C.c_int,
                                         C.c_double, C.c_uint64] + [C.c_void_p] * 6 + [C.c_int, C.c_double, C.c_double])

    def run(seed, n, pop=2**32 - 1, chunk=256, radius=1.2e15, temperature=1.0e4, beta=None):
        l_array = np.cumsum(np.arange(1, 1000, dtype=np.float64) ** -4)
        out = {k: np.empty(n, dtype=np.float64) for k in ("initial_radii", "initial_nus", "initial_mus", "initial_energies")}
        out["packet_seeds"] = np.empty(n, dtype=np.int64)
        n_rej = C.c_uint64(0)
        rc = lib.shim_create_packets(seed, n, pop - 1, radius, KB * temperature, H, l_array.ctypes.data, len(l_array), np.pi**4 / 90.0,
                                     chunk, out["initial_radii"].ctypes.data, out["initial_nus"].ctypes.data, out["initial_mus"].ctypes.data,
                                     out["initial_energies"].ctypes.data, out["packet_seeds"].ctypes.data, C.byref(n_rej),
                                     int(beta is not None), 0.0 if beta is None else beta, 0.0 if beta is None else relativistic_energy(n, beta))
        assert rc == 0
        out["n_rejected"] = n_rej.value
        return out

    lib.shim_advance.argtypes = [C.c_uint64, C.c_uint64, C.c_void_p]
    run.lib = lib
    return run


@pytest.mark.parametrize("name", CASES)
def test_oracle_matches_reference_golden(oracle, name):
    g = np.load(os.path.join(HERE, "golden", name + ".npz"))
    got = oracle.create_packets(int(g["n"]), int(g["base_seed"]) + int(g["seed_offset"]), float(g["radius"]), float(g["temperature"]),
                                beta=golden_beta(g))
    check(got, g)


@pytest.mark.parametrize("name", CASES)
def test_product_generator_matches_reference_golden(shim, name):
    g = np.load(os.path.join(HERE, "golden", name + ".npz"))
    got = shim(int(g["base_seed"]) + int(g["seed_offset"]), int(g["n"]), radius=float(g["radius"]), temperature=float(g["temperature"]),
               beta=golden_beta(g))
    check(got, g)
    assert got["n_rejected"] == 0


@pytest.mark.parametrize("seed,n,pop,chunk", [(23111963, 20011, 2**32 - 1, 256), (5, 1, 2**32 - 1, 7), (0, 2, 2**32 - 1, 1),
                                               (77, 5000, 3 * 2**30, 33), (2**40 + 3, 4097, 2**31 + 7, 1000), (9, 3001, 1000, 64),
                                               (123, 777, 2**32 - 1, 100000)])
def test_product_generator_matches_numpy(shim, oracle, seed, n, pop, chunk):
    """Random access into the PCG64 stream (jump-ahead per chunk, 32-bit halves, Lemire redraws, the fixed point on the
    number of rejected draws) against numpy's sequential generator; the oracle is held to the same."""
    want = numpy_source(seed, n, pop)
    got = shim(seed, n, pop, chunk)
    check(got, want)
    if pop in (3 * 2**30, 2**31 + 7):
        assert got["n_rejected"] > n // 4  # these populations reject about every third draw: the redraw path is exercised
    check(oracle.create_packets(n, seed, 1.2e15, 1.0e4, max_seed_val=pop), want)


def test_jump_ahead_equals_stepping(shim):
    """pcg_advance(k) lands on the state that k single steps reach (compared through numpy's own PCG64.advance)."""
    for seed, delta in [(1, 0), (1, 1), (23111963, 12345678901), (7, 2**63 + 5)]:
        out = (C.c_uint64 * 4)()
        shim.lib.shim_advance(seed, delta, out)
        bg = np.random.PCG64(seed)
        bg.advance(delta)
        st = bg.state["state"]
        assert (out[0] << 64) | out[1] == st["state"] and (out[2] << 64) | out[3] == st["inc"]


@pytest.mark.gpu
def test_device_packet_source_matches_oracle_and_feeds_transport():
    code = r"""
import sys, numpy as np
sys.path.insert(0, %r)
from oracle import cpu_oracle
from tardis_b200 import synthetic as syn
from tardis_b200.engine import Engine
model = syn.make_model(10, 4000, "macroatom", mu_tau=-4.0, seed=3)
eng = Engine(0)
eng.set_model_from(model)
for n, seed in ((100003, syn.BASE_SEED + 5), (1, 7), (513, 2**32 + 4)):
    eng.create_packets(n, seed, float(model.r_inner[0]), 1.0e4)
    got = eng.download_packets()
    want = cpu_oracle.create_packets(n, seed, float(model.r_inner[0]), 1.0e4)
    for k in ("packet_seeds", "initial_mus", "initial_radii", "initial_energies"):
        assert np.array_equal(got[k], want[k]), (n, k)
    np.testing.assert_allclose(got["initial_nus"], want["initial_nus"], rtol=1e-15, atol=0)
# BlackBodySimpleSourceRelativistic on the device (what the continuum / full-relativity modes start from)
beta = (float(model.r_inner[0]) / model.time_explosion) / 2.99792458e10
eng.create_packets(20001, 99, float(model.r_inner[0]), 1.0e4, beta=beta)
got = eng.download_packets()
want = cpu_oracle.create_packets(20001, 99, float(model.r_inner[0]), 1.0e4, beta=beta)
for k in ("packet_seeds", "initial_radii"):
    assert np.array_equal(got[k], want[k]), k
for k in ("initial_mus", "initial_energies", "initial_nus"):
    np.testing.assert_allclose(got[k], want[k], rtol=1e-15, atol=0)
# transport straight from the generated packets == transport of the same packets uploaded from the host
eng.create_packets(100003, syn.BASE_SEED + 5, float(model.r_inner[0]), 1.0e4)
pk = eng.download_packets()
eng.transport(True); eng.sync(); a = eng.download()
b = eng.run(pk["initial_radii"], pk["initial_nus"], pk["initial_mus"], pk["initial_energies"], pk["packet_seeds"])
assert a["counters"] == b["counters"]
assert np.array_equal(a["output_nus"], b["output_nus"]) and np.array_equal(a["output_energies"], b["output_energies"])
# tb200_run_resident: the resident packets through the reference-facing pipeline (one range below 4e6 packets ...)
c = eng.run_resident()
assert c["counters"] == a["counters"] and np.array_equal(c["output_nus"], a["output_nus"]) and np.array_equal(c["j_blue"], a["j_blue"])
# ... eight ranges with the outputs streaming back above it)
eng.create_packets(4200000, 11, float(model.r_inner[0]), 1.0e4)
eng.transport(True); eng.sync(); a2 = eng.download()
c2 = eng.run_resident()
assert c2["counters"] == a2["counters"]
assert np.array_equal(c2["output_nus"], a2["output_nus"]) and np.array_equal(c2["output_energies"], a2["output_energies"])
assert np.array_equal(c2["j_blue"], a2["j_blue"]) and np.array_equal(c2["edotlu"], a2["edotlu"])  # integer accumulation: order-free
for k in ("j", "nu_bar", "spectrum_emitted"):
    np.testing.assert_allclose(c2[k], a2[k], rtol=1e-11, atol=0)
c3 = eng.run_resident(per_packet=False)
assert c3["counters"] == a2["counters"] and "output_nus" not in c3
print("PACKET_SOURCE_OK")
""" % ROOT
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert "PACKET_SOURCE_OK" in out.stdout, out.stdout[-2000:] + out.stderr[-4000:]


def test_host_mirror_keeps_the_reference_surface():
    """BlackBodySimpleSourceB200 against the reference class (parsed, not imported) and against its golden luminosity."""
    from tardis_b200.packet_source import BlackBodySimpleSourceB200 as Src

    g = np.load(os.path.join(HERE, "golden", "packet_source_basic.npz"))
    s = Src(radius=float(g["radius"]), temperature=float(g["temperature"]), base_seed=int(g["base_seed"]))
    np.testing.assert_allclose(s.calculate_radfield_luminosity(), float(g["radiation_field_luminosity"]), rtol=1e-14)
    lum = s.calculate_radfield_luminosity()
    s.set_temperature_from_luminosity(lum)
    np.testing.assert_allclose(s.temperature, float(g["temperature"]), rtol=1e-14)
    with pytest.raises(ValueError):
        s.create_packets(10)  # no engine attached
    with pytest.raises(ValueError):
        Src(radius=1.0, temperature=None, base_seed=1).create_packets(10)
    # public methods of BasePacketSource / BlackBodySimpleSource, parsed from the reference by tests/golden/make_golden.py
    with open(os.path.join(HERE, "golden", "reference_interface.json")) as f:
        names = set(json.load(f)["packet_source_public_methods"])
    offered = {"create_packets", "calculate_radfield_luminosity", "set_temperature_from_luminosity", "from_simulation_state"}
    assert offered <= names and all(hasattr(Src, n) for n in offered)
    assert Src.MAX_SEED_VAL == 2**32 - 1 and Src.hdf_properties == ["radius", "temperature", "base_seed"]


def test_product_generator_matches_numpy_at_config_2_s_packet_count(shim):
    """All 1e7 packets of BASELINE config 2 (the 1e8 of the other configs differ only in the number of 256-packet chunks): every chunk
    starts from its own jump-ahead positions in numpy's stream -- 39 063 chunks, positions up to 6.5e7 raw draws -- and every packet is
    compared with numpy's sequential generator."""
    n = 10_000_000
    want = numpy_source(23111963 + 4, n)
    got = shim(23111963 + 4, n, chunk=256)
    check(got, want)
    assert got["n_rejected"] == 0
