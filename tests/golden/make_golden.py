"""Generate golden vectors from the UNMODIFIED reference (TARDIS Numba hot path).

Run in the build container, where /root/reference exists:

    python tests/golden/make_golden.py            # all cases
    python tests/golden/make_golden.py --case scatter_basic
    python tests/golden/make_golden.py --case packet_source   # BlackBodySimpleSource.create_packets (4 cases)

Each case builds a small synthetic model + packet set from seeds
(tardis_b200.synthetic), runs the reference's own
`montecarlo_transport_with_vpackets` (oracle/reference_runner.py) twice -- once
with TrackerFull (per-event trajectories) and once with TrackerLastInteraction
-- and stores the outputs plus a sha256 of the inputs in tests/golden/<case>.npz.
The GPU box has no /root/reference; tests only read the .npz files.

Cases with sigma_thomson != default run in a fresh subprocess because the
reference freezes module constants at first JIT compile
(modes/classic/solver.py:291-300, SURVEY.md Appendix B).
"""
from __future__ import annotations

import argparse
import hashlib
import os
import subprocess
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from tardis_b200 import synthetic as syn  # noqa: E402

N_TRACKED = 300

# name -> (model kwargs, n_packets, run kwargs, sigma_thomson)
CASES = {
    "scatter_basic": (dict(n_shells=10, n_lines=3000, line_interaction_type="scatter", mu_tau=-4.5, seed=101), 1500, {}, None),
    "scatter_fullrel": (dict(n_shells=10, n_lines=3000, line_interaction_type="scatter", mu_tau=-4.5, seed=102), 1500,
                        dict(enable_full_relativity=True), None),
    "scatter_thick": (dict(n_shells=8, n_lines=3000, line_interaction_type="scatter", mu_tau=-3.0, seed=103), 1200, {}, None),
    "scatter_nolines": (dict(n_shells=10, n_lines=3000, line_interaction_type="scatter", mu_tau=-4.5, seed=104), 1200,
                        dict(disable_line_scattering=True), None),
    "downbranch_basic": (dict(n_shells=10, n_lines=3000, line_interaction_type="downbranch", mu_tau=-4.0, seed=105), 1500, {}, None),
    "macroatom_basic": (dict(n_shells=10, n_lines=3000, line_interaction_type="macroatom", mu_tau=-4.0, seed=106), 1500, {}, None),
    "macroatom_fullrel": (dict(n_shells=6, n_lines=2500, line_interaction_type="macroatom", mu_tau=-3.5, seed=107), 1200,
                          dict(enable_full_relativity=True), None),
    "scatter_vpackets": (dict(n_shells=10, n_lines=3000, line_interaction_type="scatter", mu_tau=-4.5, seed=108), 800,
                         dict(number_of_vpackets=3), None),
    "macroatom_vpackets": (dict(n_shells=10, n_lines=3000, line_interaction_type="macroatom", mu_tau=-3.5, seed=109), 800,
                           dict(number_of_vpackets=4, spawn_start=2.5e14, spawn_end=1.5e15), None),
    "vpackets_fullrel": (dict(n_shells=8, n_lines=2500, line_interaction_type="downbranch", mu_tau=-4.0, seed=110), 600,
                         dict(number_of_vpackets=2, enable_full_relativity=True), None),
    # IIP / continuum mode (reference: modes/iip/*).  "continuum" holds the add_continuum kwargs; these run in a fresh
    # subprocess because CONTINUUM_PROCESSES_ENABLED is frozen into the compiled code at first JIT.
    "iip_basic": (dict(n_shells=10, n_lines=3000, line_interaction_type="macroatom", mu_tau=-4.5, seed=121), 1200,
                  dict(continuum=dict(seed=9121)), None),
    "iip_adiabatic": (dict(n_shells=8, n_lines=2500, line_interaction_type="macroatom", mu_tau=-4.0, seed=122), 1000,
                      dict(continuum=dict(seed=9122, adiabatic_fraction=0.4, chi_bf_scale=1e-2)), None),
    "iip_scatter_lines": (dict(n_shells=8, n_lines=2500, line_interaction_type="scatter", mu_tau=-4.0, seed=123), 800,
                          dict(continuum=dict(seed=9123), keep_scatter=True), None),
    "scatter_noescat": (dict(n_shells=10, n_lines=3000, line_interaction_type="scatter", mu_tau=-4.0, seed=111), 1200, {}, 1e-200),
    # Russian roulette with survivors (virtual_packet.py:214-231; the reference's default SURVIVAL_PROBABILITY is 0)
    "vpackets_survival": (dict(n_shells=8, n_lines=3000, line_interaction_type="scatter", mu_tau=-3.0, seed=112), 600,
                          dict(number_of_vpackets=3, survival_probability=0.5), None),
    # The BENCH shapes (bench.py / BASELINE.json configs[2] and configs[4]): the very model the headline runs on --
    # 5e5 lines, 20 shells, macroatom -- and the 50-shell continuum model.  The [L, S] line-estimator tables are stored as
    # checksums (compress_line_table): they would be 80 / 200 MB each.
    "bench_macroatom": (dict(n_shells=20, n_lines=500_000, line_interaction_type="macroatom", mu_tau=-7.5, seed=syn.MODEL_SEED), 2000, {}, None),
    "bench_iip": (dict(n_shells=50, n_lines=500_000, line_interaction_type="macroatom", mu_tau=-7.5, seed=syn.MODEL_SEED), 1000,
                  dict(continuum=dict()), None),
}
# Pinned on the CPU only (oracle against the reference; tests/test_oracle_golden.py): BASELINE.json configs[3] at its own shape -- the
# bench model with 10 virtual packets per packet.  The GPU side of this shape is checked in every bench run (config-4 leg: counters,
# spectrum and virtual spectrum against the oracle).
ORACLE_ONLY_CASES = {
    "bench_vpackets": (dict(n_shells=20, n_lines=500_000, line_interaction_type="macroatom", mu_tau=-7.5, seed=syn.MODEL_SEED), 600,
                       dict(number_of_vpackets=10), None),
}
BIG_TABLE_CELLS = 2_000_000  # above this many (line, shell) cells the goldens carry compress_line_table(...) instead of the table
N_BUCKETS, N_SAMPLE = 97, 40_000


def compress_line_table(a):
    """[L, S] estimator table -> what pins it without storing it: the number of non-zero cells per shell, the sums over the
    lines congruent to r modulo 97 per shell (every cell is in exactly one), and 40 000 of its non-zero cells."""
    a = np.asarray(a, dtype=np.float64)
    L, S = a.shape
    flat = a.ravel()
    nz = np.flatnonzero(flat)
    step = max(1, len(nz) // N_SAMPLE)
    idx = nz[::step][:N_SAMPLE]
    pad = (-L) % N_BUCKETS
    b = np.concatenate([a, np.zeros((pad, S))]).reshape(-1, N_BUCKETS, S).sum(axis=0)
    return dict(nnz_per_shell=(a != 0).sum(axis=0).astype(np.int64), bucket_sums=b, sample_idx=idx.astype(np.int64), sample_val=flat[idx].copy())


IT_NAME2INT = {"NO_INTERACTION": -1, "BOUNDARY": 1, "LINE": 2, "ESCATTERING": 4, "CONTINUUM_PROCESS": 8}
ST_NAME2INT = {"IN_PROCESS": 0, "EMITTED": 1, "REABSORBED": 2, "ADIABATIC_COOLING": 4}


def build_inputs(name):
    mk, n, rk, sig = {**CASES, **ORACLE_ONLY_CASES}[name]
    model = syn.make_model(**mk)
    rk = dict(rk)
    cont = rk.pop("continuum", None)
    keep_scatter = rk.pop("keep_scatter", False)
    if cont is not None:
        syn.add_continuum(model, **cont)
        if keep_scatter:
            model.line_interaction_type = "scatter"  # lines re-emit coherently, continuum still uses the macro atom
    packets = syn.make_packets(n, model.r_inner[0], base_seed=syn.BASE_SEED + mk["seed"])
    return model, packets, rk, sig


def input_digest(model, packets) -> str:
    h = hashlib.sha256()
    arrs = [model.r_inner, model.r_outer, model.electron_density, model.line_list_nu, model.tau_sobolev,
            model.spectrum_frequency_grid, model.macro.transition_probabilities, model.macro.line2macro_level_upper,
            model.macro.macro_block_edge_index, model.macro.transition_type, model.macro.destination_level_id,
            model.macro.transition_line_id, packets.initial_radii, packets.initial_nus, packets.initial_mus,
            packets.initial_energies, packets.packet_seeds]
    c = model.continuum
    if c is not None:
        arrs += [c.bf_threshold_list_nu, c.photo_ion_nu_threshold_mins, c.photo_ion_nu_threshold_maxs,
                 c.photo_ion_block_references, c.chi_bf, c.x_sect, c.phot_nus, c.ff_opacity_factor, c.emissivities,
                 c.photo_ion_activation_idx, np.int64(c.k_packet_idx), c.absorbing_markov_probabilities, model.t_electrons]
    for a in arrs:
        h.update(np.ascontiguousarray(a).tobytes())
    h.update(np.float64(model.time_explosion).tobytes())
    return h.hexdigest()


def generate(name):
    from oracle.reference_runner import run_reference, run_reference_iip, set_sigma_thomson

    model, packets, rk, sig = build_inputs(name)
    if sig is not None:
        set_sigma_thomson(sig)
    if model.continuum is not None:
        full = run_reference_iip(model, packets, track_full=True, **rk)
        last = run_reference_iip(model, packets, track_full=False, **rk)
    else:
        full = run_reference(model, packets, track_full=True, **rk)
        last = run_reference(model, packets, track_full=False, **rk)
    for k in ("output_nus", "output_energies", "j", "nu_bar", "j_blue", "edotlu", "vhist"):
        assert np.array_equal(full[k], last[k]), k
    ev = full["events"]
    pid = ev.index.get_level_values(0).values.astype(np.int64)
    sel = pid < N_TRACKED
    evd = {
        "ev_packet_id": pid[sel],
        "ev_interaction_type": np.array([IT_NAME2INT[str(x)] for x in ev["interaction_type"].values[sel]], dtype=np.int64),
        "ev_status": np.array([ST_NAME2INT[str(x)] for x in ev["status"].values[sel]], dtype=np.int64),
    }
    for col in ("before_shell_id", "after_shell_id", "line_absorb_id", "line_emit_id"):
        evd["ev_" + col] = np.asarray(ev[col].values[sel], dtype=np.int64)
    for col in ("radius", "before_nu", "before_mu", "before_energy", "after_nu", "after_mu", "after_energy"):
        evd["ev_" + col] = np.asarray(ev[col].values[sel], dtype=np.float64)
    counts = np.bincount(pid, minlength=len(packets)).astype(np.int64)
    if full["j_blue"].size > BIG_TABLE_CELLS:
        tables = {}
        for k in ("j_blue", "edotlu"):
            tables.update({f"{k}__{kk}": v for kk, v in compress_line_table(full[k]).items()})
    else:
        tables = dict(j_blue=full["j_blue"], edotlu=full["edotlu"])
    out = dict(
        digest=np.array(input_digest(model, packets)),
        output_nus=full["output_nus"], output_energies=full["output_energies"],
        j=full["j"], nu_bar=full["nu_bar"], vhist=full["vhist"], **tables,
        event_counts=counts,
        **{k: full[k] for k in ("photo_ion_estimator", "stim_recomb_estimator", "bf_heating_estimator",
                                "stim_recomb_cooling_estimator", "ff_heating_estimator", "photo_ion_estimator_statistics")
           if k in full},
        **evd,
        **{k: v for k, v in last.items() if k.startswith("last_")},
    )
    path = os.path.join(HERE, name + ".npz")
    np.savez_compressed(path, **out)
    emitted = (full["output_energies"] > 0).mean()
    nline = (evd["ev_interaction_type"] == 2).sum()
    nesc = (evd["ev_interaction_type"] == 4).sum()
    print(f"{name}: wrote {os.path.getsize(path)/1e3:.0f} kB; emitted {emitted:.2f}; "
          f"tracked events line={nline} escat={nesc}; vhist sum {full['vhist'].sum():.3e}")


# Packet source (SURVEY.md §8f rank 1): name -> (no_of_packets, base_seed, seed_offset, radius [cm], temperature [K])
PACKET_SOURCE_CASES = {
    "packet_source_basic": (4001, 23111963, 0, 1.2355e15, 1.0e4),
    "packet_source_iteration7": (2500, 23111963, 7, 1.2355e15, 9.974969e3),
    "packet_source_big_seed": (1024, 2**32 - 6, 10, 8.0e14, 2.5e4),  # base_seed + seed_offset >= 2**32: two entropy words
    "packet_source_single": (1, 1963, 0, 1.0e15, 1.0e4),
    # BlackBodySimpleSourceRelativistic: sixth entry = time_explosion [s]
    "packet_source_relativistic": (3001, 23111963, 3, 1.2355e15, 1.0e4, 13.0 * 86400.0),
}


def generate_packet_source(name):
    """Golden vectors of the unmodified BlackBodySimpleSource.create_packets (oracle/reference_runner.py)."""
    from oracle.reference_runner import run_reference_packet_source

    n, base_seed, off, radius, temperature, *rest = PACKET_SOURCE_CASES[name]
    t_exp = rest[0] if rest else None
    out = run_reference_packet_source(n, base_seed, off, radius, temperature, time_explosion=t_exp)
    path = os.path.join(HERE, name + ".npz")
    extra = {} if t_exp is None else {"time_explosion": np.float64(t_exp)}
    np.savez_compressed(path, n=np.int64(n), base_seed=np.uint64(base_seed), seed_offset=np.int64(off), radius=np.float64(radius),
                        temperature=np.float64(temperature), **extra, **out)
    print(f"{name}: wrote {os.path.getsize(path)/1e3:.0f} kB; mean nu {out['initial_nus'].mean():.4e}")


# Radiation-field solve (SURVEY.md §8f rank 4): name -> (seed, n_shells, n_lines, zero fraction of the J_blue estimator)
RADFIELD_CASES = {"radfield_basic": (31, 20, 4000, 0.3), "radfield_sparse": (32, 7, 1500, 0.9)}


RADFIELD_BENCH_SHAPE = {"radfield_bench_shape": (33, 20, 500_000, 0.5)}  # the bench's [L, S]


def radfield_inputs(name):
    seed, S, L, zero_frac = {**RADFIELD_CASES, **RADFIELD_BENCH_SHAPE}[name]
    rng = np.random.default_rng(seed)
    j = rng.uniform(0.5, 2.0, S) * 1e-3
    nu_bar = j * rng.uniform(4e14, 1.2e15, S)
    j_blue = rng.uniform(0.0, 1.0, (L, S)) * 1e-18
    j_blue[rng.random((L, S)) < zero_frac] = 0.0
    volume = rng.uniform(1.0, 3.0, S) * 1e45
    nu = np.sort(np.exp(rng.uniform(np.log(1.5e14), np.log(6e15), L)))[::-1].copy()
    return dict(j=j, nu_bar=nu_bar, j_blue=j_blue, volume=volume, line_list_nu=nu, time_explosion=13.0 * 86400.0,
                time_of_simulation=1.0 / 1.07e43, w_epsilon=1e-10)


def generate_radfield(name):
    """Golden vectors of the unmodified MCRadiationFieldPropertiesSolver.solve (oracle/reference_runner.py)."""
    from oracle.reference_runner import run_reference_radfield

    inp = radfield_inputs(name)
    out = run_reference_radfield(inp["j"], inp["nu_bar"], inp["j_blue"], inp["time_explosion"], inp["time_of_simulation"], inp["volume"],
                                 inp["line_list_nu"], inp["w_epsilon"])
    path = os.path.join(HERE, name + ".npz")
    np.savez_compressed(path, **out)
    print(f"{name}: wrote {os.path.getsize(path)/1e3:.0f} kB; T_rad {out['t_radiative'][:3]}, W {out['dilution_factor'][:3]}")


def generate_radfield_bench_shape():
    """Golden of the unmodified MCRadiationFieldPropertiesSolver.solve at the bench's [5e5, 20]; the J_blue table as checksums + samples."""
    from oracle.reference_runner import run_reference_radfield

    name = "radfield_bench_shape"
    inp = radfield_inputs(name)
    out = run_reference_radfield(inp["j"], inp["nu_bar"], inp["j_blue"], inp["time_explosion"], inp["time_of_simulation"], inp["volume"],
                                 inp["line_list_nu"], inp["w_epsilon"])
    keep = dict(t_radiative=out["t_radiative"], dilution_factor=out["dilution_factor"])
    for kk, vv in compress_table(out["j_blues"]).items():
        keep[f"j_blues__{kk}"] = vv
    path = os.path.join(HERE, name + ".npz")
    np.savez_compressed(path, **keep)
    print(f"{name}: wrote {os.path.getsize(path)/1e3:.0f} kB")


# Opacity build (SURVEY.md §8f rank 3): name -> (model seed, n_shells, n_lines, n_levels, mode)
OPACITY_CASES = {"opacity_macroatom": (41, 8, 3000, 400, "macroatom"), "opacity_downbranch": (42, 5, 1200, 150, "downbranch")}


# the bench's size: 5e5 lines, 3000 levels, 1.5e6 macro-atom rows (four shells: every cell depends on its own shell only)
OPACITY_BENCH_SHAPE = {"opacity_bench_shape": (47, 4, 500_000, 3000, "macroatom")}


def opacity_inputs(name):
    seed, S, L, n_levels, mode = {**OPACITY_CASES, **OPACITY_BENCH_SHAPE}[name]
    model = syn.make_model(S, L, "scatter", seed=seed)
    atomic = syn.make_atomic_data(model.line_list_nu, n_levels, mode, seed=seed + 1)
    plasma = syn.make_plasma_state(atomic, S, model.time_explosion, seed=seed + 2)
    return model, atomic, plasma


def generate_opacity(name):
    """Golden vectors of the reference's own tau_sobolev / beta_sobolev / probability functions (oracle/reference_runner.py)."""
    from oracle.reference_runner import run_reference_opacity

    model, atomic, plasma = opacity_inputs(name)
    out = run_reference_opacity(atomic, plasma, nlte=True)
    path = os.path.join(HERE, name + ".npz")
    np.savez_compressed(path, **out)
    print(f"{name}: wrote {os.path.getsize(path)/1e3:.0f} kB; tau in [{out['tau_sobolev'].min():.3e}, {out['tau_sobolev'].max():.3e}]")


def generate_opacity_bench_shape():
    """Golden of the reference's own tau / beta / probability functions at the bench's size; tables as checksums + samples."""
    from oracle.reference_runner import run_reference_opacity

    name = "opacity_bench_shape"
    model, atomic, plasma = opacity_inputs(name)
    out = run_reference_opacity(atomic, plasma, nlte=True)
    keep = {}
    for k, v in out.items():
        for kk, vv in compress_table(v).items():
            keep[f"{k}__{kk}"] = vv
        keep[f"{k}__max_abs"] = np.max(np.abs(v))
    path = os.path.join(HERE, name + ".npz")
    np.savez_compressed(path, **keep)
    print(f"{name}: wrote {os.path.getsize(path)/1e3:.0f} kB; keys {sorted(out)}")


SOURCE_FUNCTION_CASES = {"source_function_macroatom": (51, 6, 2500, 200, "macroatom"), "source_function_downbranch": (55, 4, 1500, 120, "downbranch")}


# the bench's size (5e5 lines, 3000 levels -> 1.5e6 macro-atom rows, 1e6 of them internal), four shells (each shell is its own system)
SOURCE_FUNCTION_BENCH_SHAPE = {"source_function_bench_shape": (57, 4, 500_000, 3000, "macroatom")}
SF_BENCH_SAMPLE = 8000


def source_function_inputs(name):
    """Model, atomic data, opacity tables (oracle port, itself pinned by the opacity goldens), line estimators with the exact
    zeros a Monte Carlo run leaves, volume, times."""
    from oracle import opacity_oracle

    seed, S, L, n_levels, mode = {**SOURCE_FUNCTION_CASES, **SOURCE_FUNCTION_BENCH_SHAPE}[name]
    model = syn.make_model(S, L, "scatter", seed=seed)
    atomic = syn.make_atomic_data(model.line_list_nu, n_levels, mode, seed=seed + 1)
    plasma = syn.make_plasma_state(atomic, S, model.time_explosion, seed=seed + 2, inversion_fraction=0.0)
    plasma.level_number_density *= 1e-9  # optical depths of order one (and a few mildly negative ones)
    tables = opacity_oracle.build(atomic, plasma, nlte=True)
    rng = np.random.default_rng(seed + 3)
    j_blue = rng.random((L, S)) * 1e-3
    j_blue[rng.random((L, S)) < 0.3] = 0.0
    e_dot_lu = rng.random((L, S)) * 1e40
    e_dot_lu[rng.random((L, S)) < 0.3] = 0.0
    volume = 4.0 / 3.0 * np.pi * (model.r_outer**3 - model.r_inner**3)
    return dict(model=model, atomic=atomic, tau_sobolev=tables["tau_sobolev"], transition_probabilities=tables["transition_probabilities"],
                j_blue_estimator=j_blue, e_dot_lu_estimator=e_dot_lu, volume=volume, time_explosion=float(model.time_explosion),
                time_of_simulation=1.3e5, mode=mode)


def generate_source_function(name):
    """Golden vectors of the reference's own SourceFunctionSolver.solve (oracle/reference_runner.py)."""
    from oracle.reference_runner import run_reference_source_function

    i = source_function_inputs(name)
    out = run_reference_source_function(i["atomic"], i["tau_sobolev"], i["transition_probabilities"], i["j_blue_estimator"], i["e_dot_lu_estimator"],
                                        i["time_explosion"], i["time_of_simulation"], i["volume"], i["mode"])
    path = os.path.join(HERE, name + ".npz")
    np.savez_compressed(path, **out)
    print(f"{name}: wrote {os.path.getsize(path)/1e3:.0f} kB; att_S_ul in [{out['att_S_ul'].min():.3e}, {out['att_S_ul'].max():.3e}]")


def compress_table(a, n_sample=SF_BENCH_SAMPLE):
    """[L, S] table -> per-shell sums over the lines congruent to r modulo 97 (every cell is in exactly one) and `n_sample` cells spread
    evenly over the table"""
    a = np.asarray(a, dtype=np.float64)
    L, S = a.shape
    pad = (-L) % N_BUCKETS
    b = np.concatenate([a, np.zeros((pad, S))]).reshape(-1, N_BUCKETS, S).sum(axis=0)
    idx = np.linspace(0, a.size - 1, n_sample).astype(np.int64)
    return dict(bucket_sums=b, sample_idx=idx, sample_val=a.ravel()[idx].copy(), n_zero=np.int64((a == 0).sum()))


def generate_source_function_bench_shape():
    """Golden of the reference's own SourceFunctionSolver.solve at the bench's size; the [L, S] tables are stored as checksums + samples."""
    from oracle.reference_runner import run_reference_source_function

    name = "source_function_bench_shape"
    i = source_function_inputs(name)
    out = run_reference_source_function(i["atomic"], i["tau_sobolev"], i["transition_probabilities"], i["j_blue_estimator"], i["e_dot_lu_estimator"],
                                        i["time_explosion"], i["time_of_simulation"], i["volume"], i["mode"])
    keep = dict(e_dot_u=out["e_dot_u"], e_dot_u_levels=out["e_dot_u_levels"])
    for k in ("att_S_ul", "Jred_lu", "Jblue_lu"):
        for kk, v in compress_table(out[k]).items():
            keep[f"{k}__{kk}"] = v
        keep[f"{k}__max_abs"] = np.max(np.abs(out[k]))
    path = os.path.join(HERE, name + ".npz")
    np.savez_compressed(path, **keep)
    print(f"{name}: wrote {os.path.getsize(path)/1e3:.0f} kB")


# name: (source-function case the tables come from, inner temperature, points, interpolate_shells, number of frequencies)
FORMAL_INTEGRAL_CASES = {"formal_integral_macroatom": ("source_function_macroatom", 1.0e4, 64, 20, 120),
                         "formal_integral_downbranch": ("source_function_downbranch", 1.2e4, 50, -1, 90),
                         "formal_integral_default_shells": ("source_function_macroatom", 0.9e4, 33, 0, 40)}


def formal_integral_inputs(name):
    """The source function's golden tables (the reference's own output) as the integrator's input, the model they belong to, and a
    frequency grid whose rays never leave the line list on the red side (there the reference reads behind its arrays:
    oracle/formal_integral_oracle.c) but do leave it on the blue side."""
    sf_name, t_inner, points, interpolate_shells, n_freq = FORMAL_INTEGRAL_CASES[name]
    i = source_function_inputs(sf_name)
    g = dict(np.load(os.path.join(HERE, sf_name + ".npz")))
    m = i["model"]
    z_max = m.r_outer[-1] / m.time_explosion / 2.99792458e10
    frequencies = np.linspace(m.line_list_nu[-1] / (1 - z_max) * 1.001, m.line_list_nu[0] * 1.02, n_freq)
    return dict(model=m, tau_sobolev=i["tau_sobolev"], att_S_ul=g["att_S_ul"], Jred_lu=g["Jred_lu"], Jblue_lu=g["Jblue_lu"],
                electron_densities=np.asarray(m.electron_density, dtype=np.float64), inner_temperature=t_inner, points=points,
                interpolate_shells=interpolate_shells, frequencies=frequencies, source_function_case=sf_name)


FORMAL_INTEGRAL_BENCH_SHAPE = dict(n_lines=500_000, n_shells=20, points=1000, inner_temperature=1.0e4, n_frequencies=16)


def formal_integral_bench_shape_inputs(n_frequencies=None):
    """The formal integral at the size bench.py runs it (5e5 lines, 20 -> 79 shells, 1000 impact parameters): line list / geometry /
    tau of the bench generator with optical depths around 1e-3 (2 dex scatter), random source-function tables, and `n_frequencies` bins
    of the reference's spectrum grid spread over the whole grid.  Regenerated from seeds; the golden holds only the reference's outputs."""
    from tardis_b200 import synthetic as syn

    c = FORMAL_INTEGRAL_BENCH_SHAPE
    L, S = c["n_lines"], c["n_shells"]
    n_frequencies = c["n_frequencies"] if n_frequencies is None else n_frequencies
    model = syn.make_model(S, L, "downbranch", mu_tau=-3.0, seed=91)
    rng = np.random.default_rng(92)
    att = rng.random((L, S)) * 1e-6
    jblue = rng.random((L, S)) * 1e-5
    jred = jblue * np.exp(-np.asarray(model.tau_sobolev)) + att
    grid = np.asarray(model.spectrum_frequency_grid, dtype=np.float64)[:-1]
    sample = np.linspace(0, len(grid) - 1, n_frequencies + 2).astype(int)[1:-1]
    return dict(model=model, tau_sobolev=np.asarray(model.tau_sobolev), att_S_ul=att, Jred_lu=jred, Jblue_lu=jblue,
                electron_densities=np.asarray(model.electron_density, dtype=np.float64), inner_temperature=c["inner_temperature"],
                points=c["points"], interpolate_shells=0, frequencies=grid[sample].copy())


def generate_formal_integral_bench_shape():
    """Golden of the UNMODIFIED reference at the bench shape (also written by scripts/reference_formal_integral_rate.py --golden)."""
    from oracle.reference_runner import run_reference_formal_integral

    i = formal_integral_bench_shape_inputs()
    out = run_reference_formal_integral(i["model"], i["tau_sobolev"], i["att_S_ul"], i["Jred_lu"], i["Jblue_lu"], i["electron_densities"],
                                        i["inner_temperature"], i["frequencies"], i["points"], i["interpolate_shells"])
    path = os.path.join(HERE, "formal_integral_bench_shape.npz")
    np.savez_compressed(path, frequencies=i["frequencies"], luminosity_densities=out["luminosity_densities"], intensities_nu_p=out["intensities_nu_p"])
    print(f"formal_integral_bench_shape: wrote {os.path.getsize(path)/1e3:.0f} kB")


def generate_formal_integral(name):
    """Golden vectors of the reference's own interpolate_integrator_quantities + numba_formal_integral (oracle/reference_runner.py)."""
    from oracle.reference_runner import run_reference_formal_integral

    i = formal_integral_inputs(name)
    out = run_reference_formal_integral(i["model"], i["tau_sobolev"], i["att_S_ul"], i["Jred_lu"], i["Jblue_lu"], i["electron_densities"],
                                        i["inner_temperature"], i["frequencies"], i["points"], i["interpolate_shells"])
    keep = dict(luminosity_densities=out["luminosity_densities"], intensities_nu_p=out["intensities_nu_p"],
                electron_densities_interpolated=out["electron_densities_interpolated"], r_inner_interpolated=out["r_inner_interpolated"],
                r_outer_interpolated=out["r_outer_interpolated"])
    for k in ("att_S_ul_interpolated", "Jred_lu_interpolated", "Jblue_lu_interpolated", "tau_sobolevs_interpolated"):
        keep[k + "__shell_sums"] = out[k].sum(axis=0)  # pins the glue (shell count, extrapolation, clipping); the values are scipy's
        keep[k + "__line_sums"] = out[k].sum(axis=1)
    path = os.path.join(HERE, name + ".npz")
    np.savez_compressed(path, **keep)
    print(f"{name}: wrote {os.path.getsize(path)/1e3:.0f} kB; L_nu in [{keep['luminosity_densities'].min():.3e}, {keep['luminosity_densities'].max():.3e}]")


# The reference's public surface the host mirrors keep (tests/test_interface_mirror.py, tests/test_packet_source.py): positional
# parameter names of each mirrored function, per source file (paths relative to tardis/transport/montecarlo/modes, as the tests
# name them), parsed with ast and never imported.
INTERFACE_SIGNATURES = {
    "montecarlo_transport.py": ["montecarlo_transport_with_vpackets"],
    "iip/montecarlo_transport.py": ["montecarlo_transport"],
    "classic/solver.py": ["MCTransportSolverClassic.__init__", "MCTransportSolverClassic.from_config",
                          "MCTransportSolverClassic.initialize_transport_state", "MCTransportSolverClassic.run"],
    "iip/solver.py": ["MCTransportSolverIIP.__init__", "MCTransportSolverIIP.from_config", "MCTransportSolverIIP.initialize_transport_state",
                      "MCTransportSolverIIP.run"],
    "../estimators/mc_rad_field_solver.py": ["MCRadiationFieldPropertiesSolver.__init__", "MCRadiationFieldPropertiesSolver.solve"],
    "../../../spectrum/formal_integral/source_function.py": ["SourceFunctionSolver.__init__", "SourceFunctionSolver.solve"],
    "../../../spectrum/formal_integral/formal_integral_solver.py": ["FormalIntegralSolver.__init__", "FormalIntegralSolver.solve"],
    "../../../spectrum/formal_integral/base.py": ["check_formal_integral_requirements"],
    "../../../spectrum/base.py": ["SpectrumSolver.__init__", "SpectrumSolver.setup_optional_spectra", "SpectrumSolver.solve",
                                  "SpectrumSolver.from_config"],
    "../../../spectrum/spectrum.py": ["TARDISSpectrum.__init__"],
}


def generate_reference_interface():
    """tests/golden/reference_interface.json: the mirrored signatures (INTERFACE_SIGNATURES), SpectrumSolver's properties and
    hdf_properties, and the public methods of BasePacketSource / BlackBodySimpleSource."""
    import ast
    import json

    from oracle.reference_loader import REF

    modes = os.path.join(REF, "tardis", "transport", "montecarlo", "modes")

    def parse(rel):
        with open(os.path.normpath(os.path.join(modes, rel))) as f:
            return ast.parse(f.read())

    signatures = {}
    for rel, names in INTERFACE_SIGNATURES.items():
        found = {}
        for node in parse(rel).body:
            if isinstance(node, ast.FunctionDef):
                found[node.name] = [a.arg for a in node.args.args]
            elif isinstance(node, ast.ClassDef):
                for m in node.body:
                    if isinstance(m, ast.FunctionDef):
                        found[f"{node.name}.{m.name}"] = [a.arg for a in m.args.args if a.arg not in ("self", "cls")]
        signatures[rel] = {n: found[n] for n in names}
    cls = next(n for n in parse("../../../spectrum/base.py").body if isinstance(n, ast.ClassDef) and n.name == "SpectrumSolver")
    props = [m.name for m in cls.body if isinstance(m, ast.FunctionDef) and any(getattr(d, "id", None) == "property" for d in m.decorator_list)]
    hdf = next(ast.literal_eval(m.value) for m in cls.body if isinstance(m, ast.Assign) and m.targets[0].id == "hdf_properties")
    packet_source = set()
    for f in ("base.py", "black_body.py"):
        for node in parse(os.path.join("..", "packet_source", f)).body:
            if isinstance(node, ast.ClassDef) and node.name in ("BasePacketSource", "BlackBodySimpleSource"):
                packet_source |= {m.name for m in node.body if isinstance(m, ast.FunctionDef) and not m.name.startswith("_")}
    out = {"signatures": signatures, "spectrum_solver": {"properties": props, "hdf_properties": hdf},
           "packet_source_public_methods": sorted(packet_source)}
    path = os.path.join(HERE, "reference_interface.json")
    with open(path, "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write("\n")
    print(f"reference_interface: wrote {os.path.getsize(path)} bytes")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--case", default=None)
    args = ap.parse_args()
    if args.case == "reference_interface":
        generate_reference_interface()
        return
    if args.case in PACKET_SOURCE_CASES:
        generate_packet_source(args.case)
        return
    if args.case == "packet_source":
        for name in PACKET_SOURCE_CASES:
            generate_packet_source(name)
        return
    if args.case in OPACITY_CASES or args.case == "opacity":
        for name in ([args.case] if args.case in OPACITY_CASES else OPACITY_CASES):
            generate_opacity(name)
        return
    if args.case in SOURCE_FUNCTION_CASES or args.case == "source_function":
        for name in ([args.case] if args.case in SOURCE_FUNCTION_CASES else SOURCE_FUNCTION_CASES):
            generate_source_function(name)
        return
    if args.case == "radfield_bench_shape":
        generate_radfield_bench_shape()
        return
    if args.case == "opacity_bench_shape":
        generate_opacity_bench_shape()
        return
    if args.case == "source_function_bench_shape":
        generate_source_function_bench_shape()
        return
    if args.case == "formal_integral_bench_shape":
        generate_formal_integral_bench_shape()
        return
    if args.case in FORMAL_INTEGRAL_CASES or args.case == "formal_integral":
        for name in ([args.case] if args.case in FORMAL_INTEGRAL_CASES else FORMAL_INTEGRAL_CASES):
            generate_formal_integral(name)
        return
    if args.case in RADFIELD_CASES or args.case == "radfield":
        for name in ([args.case] if args.case in RADFIELD_CASES else RADFIELD_CASES):
            generate_radfield(name)
        return
    if args.case:
        generate(args.case)
        return
    default_sigma = [n for n, c in {**CASES, **ORACLE_ONLY_CASES}.items() if c[3] is None and "continuum" not in c[2]]
    other = [n for n, c in CASES.items() if c[3] is not None or "continuum" in c[2]]
    for n in default_sigma:
        generate(n)
    for n in other:
        subprocess.run([sys.executable, os.path.abspath(__file__), "--case", n], check=True)
    subprocess.run([sys.executable, os.path.abspath(__file__), "--case", "packet_source"], check=True)
    subprocess.run([sys.executable, os.path.abspath(__file__), "--case", "radfield"], check=True)
    subprocess.run([sys.executable, os.path.abspath(__file__), "--case", "opacity"], check=True)
    subprocess.run([sys.executable, os.path.abspath(__file__), "--case", "source_function"], check=True)
    subprocess.run([sys.executable, os.path.abspath(__file__), "--case", "formal_integral"], check=True)
    subprocess.run([sys.executable, os.path.abspath(__file__), "--case", "formal_integral_bench_shape"], check=True)
    subprocess.run([sys.executable, os.path.abspath(__file__), "--case", "source_function_bench_shape"], check=True)
    subprocess.run([sys.executable, os.path.abspath(__file__), "--case", "opacity_bench_shape"], check=True)
    subprocess.run([sys.executable, os.path.abspath(__file__), "--case", "radfield_bench_shape"], check=True)
    generate_reference_interface()


if __name__ == "__main__":
    main()
