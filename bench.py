#!/usr/bin/env python
"""bench.py -- MC packets/sec of the packet-propagation path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's CUDA engine
    python bench.py --impl reference [--gpus N] ...                # CPU arm (oracle port, all host threads)
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N   # one rank per GPU
    python bench.py ... --dump-outputs DIR                          # + what the last timed step computed, DIR/<name>.npy

One "step" = one Monte Carlo iteration of the hot path (`montecarlo_transport_with_vpackets`,
tardis/transport/montecarlo/modes/montecarlo_transport.py:239) over one batch of synthetic packets, INCLUDING what
every iteration pays for its fresh packets (RNG seed expansion, processing order) and the estimator epilogues.

Headline (top-level keys) = BASELINE.json configs[2]: 1e8 packets per GPU, 20 shells, 5e5-line synthetic list,
macroatom (SURVEY.md §8d generator, tardis_b200/synthetic.py); weak scaling (every rank its own 1e8 packets), the only
collective is one all-reduce of the packed estimator buffer.

The same run then measures, as short legs under "configs" (K = --leg-steps, W = 3):
  "2"      BASELINE configs[1]: 1e7 packets TOTAL, line_interaction_type=scatter
  "4"      BASELINE configs[3]: 1e8 packets TOTAL + 10 virtual packets per real packet, macroatom
  "5"      BASELINE configs[4]: 1e8 packets TOTAL, continuum (bound-free + free-free, IIP mode), 50 shells
  "strong" configs[2] with 1e8 packets TOTAL over the N ranks (the strong-scaling point; at N = 1 it is the headline)
each with value / e2e / roofline / cpu_baseline (N = 1) / parity against the oracle (spectrum L2, max relative error of
J, nu_bar, J_blue, Edotlu), and at N > 1 a cross-rank check of the all-reduced estimator buffer.

  value   : packets/s with the packets already resident in HBM (all kernels of an iteration + the all-reduce)
  e2e     : packets/s through the reference-facing call `tb200_run` with pinned HOST buffers:
            H2D of the 5 packet arrays, seed expansion, transport kernel, D2H of output_nus/energies
            and of all estimators ([L,S] layout), every step
  roofline: `achieved` = DRAM bytes of the transport kernel (from the committed ncu capture of the same workload,
            profiles/traffic.json) / its CUDA-event duration measured here; next to it the binding resource the captures
            show (issue-slot utilisation, lanes per instruction, occupancy) and the SURVEY.md §8(d) byte count of the same
            packets -- which the jump algorithm does not move (it is O(log) per trace, not O(lines))
  cpu_baseline: oracle/tardis_oracle.c ("port" of the reference loop) on the host threads, bounded sample
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from tardis_b200 import synthetic as syn  # noqa: E402

METRIC = "MC packets/sec at 1e8 packets, 20 shells, 5e5 lines; spectrum L2 vs ref"


def json_safe(x):
    """NaN / inf -> None, numpy scalars -> Python numbers: the bench line must be strict JSON for every parser."""
    if isinstance(x, dict):
        return {str(k): json_safe(v) for k, v in x.items()}
    if isinstance(x, (list, tuple)):
        return [json_safe(v) for v in x]
    if isinstance(x, np.generic):
        x = x.item()
    if isinstance(x, float) and not np.isfinite(x):
        return None
    if isinstance(x, np.ndarray):
        return json_safe(x.tolist())
    return x


def alg_bytes(c: dict, n_packets: int) -> int:
    """SURVEY.md §8(d): 48 B per line-step, 16 B per virtual-packet line-step, 32 B per event,
    8 B per scanned macro-atom transition, 24 B per macro-atom jump, 56 B per packet."""
    events = c["n_boundary_events"] + c["n_line_events"] + c["n_escat_events"]
    return (48 * c["n_line_steps"] + 16 * c["n_vpacket_line_steps"] + 32 * events
            + 8 * c["n_macro_scanned"] + 24 * c["n_macro_jumps"] + 80 * c.get("n_bf_estimator_updates", 0) + 56 * n_packets)


def make_packets_chunked(n: int, r_inner0: float, seed_base: int, chunk: int = 10_000_000) -> syn.Packets:
    """n packets as a concatenation of BlackBodySimpleSource batches (bounded host memory)."""
    parts = []
    done = 0
    it = 0
    while done < n:
        m = min(chunk, n - done)
        parts.append(syn.make_packets(m, r_inner0, base_seed=seed_base, iteration=it))
        done += m
        it += 1
    if len(parts) == 1:
        p = parts[0]
    else:
        p = syn.Packets(*(np.concatenate([getattr(q, f) for q in parts]) for f in
                          ("initial_radii", "initial_nus", "initial_mus", "initial_energies", "packet_seeds")),
                        parts[0].radiation_field_luminosity)
    p.initial_energies[:] = 1.0 / n
    return p


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""

    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, device_index: int):
        self.device_index = device_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "200",
                 "-i", str(self.device_index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, power, reasons = [], [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        busy = [s for s, p in zip(sm, power) if p > 250.0] or sm
        return {"sm_mhz": float(np.median(busy)), "sm_max_mhz": float(max(smax)), "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": float(max(power))}


def read_peak() -> tuple[float, str]:
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def read_capture(workload_key: str):
    """The committed ncu capture of this workload's transport kernel (profiles/traffic.json): DRAM bytes of one launch, the
    packets of that launch, and the utilisation figures of the same capture."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return json.load(f).get(workload_key)
    except Exception:
        return None


def histogram_spectrum(nus, energies, grid, time_of_simulation, emitted=True):
    """SpectrumSolver.montecarlo_emitted_luminosity / _reabsorbed_luminosity: np.histogram of the packets
    (tardis/spectrum/base.py:139-159)."""
    m = energies >= 0 if emitted else (energies < 0) & (energies != -99.0)
    h, _ = np.histogram(nus[m], weights=np.abs(energies[m]) / time_of_simulation, bins=grid)
    return h


def rel_l2(a, b):
    nb = float(np.linalg.norm(b))
    return float(np.linalg.norm(a - b) / nb) if nb > 0 else (0.0 if not np.any(a) else float("inf"))


def max_rel_err(a, b):
    """max |a - b| / |b| over the entries the reference touched; inf if the zero patterns differ."""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    nz = b != 0
    if np.any((a != 0) != nz):
        return float("inf")
    return float(np.max(np.abs(a[nz] - b[nz]) / np.abs(b[nz]))) if np.any(nz) else 0.0


def cpu_leg(model, n_threads: int, seed_base: int, vp: int, target_seconds: float = 12.0, calibrate: bool = True):
    """Time the CPU oracle (port of the reference loop) on a bounded sample of the workload."""
    from oracle import cpu_oracle

    cpu_oracle.build()
    # Calibrate: thread count x estimator layout (per-thread tables as in the reference, or one shared table with atomic
    # adds).  More threads are not always faster for this memory-latency-bound loop; the timed run uses the fastest.
    cores = n_threads
    key = (cores, vp, model.n_shells, model.continuum is not None, model.line_interaction_type)
    cache = getattr(cpu_leg, "calibrated", {})
    best = cache.get(key)
    if best is None and not calibrate and cache:  # legs reuse the headline's choice of threads / layout
        _, t0_, p0_ = next(iter(cache.values()))
        n0 = max(1_000, 100 * t0_)
        calib = make_packets_chunked(n0, model.r_inner[0], seed_base + 1)
        t0 = time.perf_counter()
        cpu_oracle.run_oracle(model, calib, number_of_vpackets=vp, nthreads=t0_, track_last_interaction=False,
                              private_tables_max_threads=(t0_ if p0_ else 0))
        best = (n0 / max(time.perf_counter() - t0, 1e-3), t0_, p0_)
    if best is None:
        candidates = sorted({(t, private) for t in (cores, cores // 2, cores // 4, 32, 16, 8) if 1 <= t <= cores
                             for private in (True, False) if not (private and t > 32)}, reverse=True)
        for t, private in candidates:
            n0 = max(1_000, 100 * t)
            calib = make_packets_chunked(n0, model.r_inner[0], seed_base + 1)
            t0 = time.perf_counter()
            cpu_oracle.run_oracle(model, calib, number_of_vpackets=vp, nthreads=t, track_last_interaction=False,
                                  private_tables_max_threads=(t if private else 0))
            rate = n0 / max(time.perf_counter() - t0, 1e-3)
            if best is None or rate > best[0]:
                best = (rate, t, private)
    cpu_leg.calibrated = {**cache, key: best}
    rate0, n_threads, private = best
    n = int(min(max(rate0 * target_seconds, 2_000), 4_000_000))
    sample = make_packets_chunked(n, model.r_inner[0], seed_base)
    t0 = time.perf_counter()
    res = cpu_oracle.run_oracle(model, sample, number_of_vpackets=vp, nthreads=n_threads, track_last_interaction=False,
                                private_tables_max_threads=(n_threads if private else 0))
    dt = time.perf_counter() - t0
    cpu_leg.last_choice = {"threads": n_threads, "layout": "per-thread tables" if private else "shared table + atomic adds",
                           "host_cores": cores}
    return n / dt, n, dt, sample, res, n_threads


def workload_text(spec: dict) -> str:
    n = spec["packets_total"] if spec["scaling"] == "strong" else spec["packets_per_gpu"]
    return (f"{n:.0e} packets{' total' if spec['scaling'] == 'strong' else '/GPU'}, {spec['shells']} shells, {spec['lines']} lines, "
            f"{spec['mode']}" + (f", {spec['vpackets']} vpackets" if spec["vpackets"] else "")
            + (", continuum (IIP mode)" if spec["continuum"] else "") + f", tau~10^N({spec['mu_tau']},2)")


def build_model(spec: dict):
    model = syn.make_model(spec["shells"], spec["lines"], spec["mode"], mu_tau=spec["mu_tau"])
    if spec["continuum"]:
        syn.add_continuum(model)
    return model


def kernel_name(spec: dict, algorithm: str) -> str:
    if algorithm == "scan":
        return "tb::transport_scan_kernel"
    return "tb::transport_jump_kernel" if spec["vpackets"] else "tb::transport_pool_kernel"  # (continuum mode: pooled kernel too)


def workload_key(spec: dict, algorithm: str) -> str:
    return (f"{algorithm}_{spec['mode']}_{spec['lines']}_{spec['shells']}" + (f"_vp{spec['vpackets']}" if spec["vpackets"] else "")
            + ("_continuum" if spec["continuum"] else ""))


def roofline_block(spec, algorithm, counters, n, k_ms, peak, peak_src):
    events = counters["n_boundary_events"] + counters["n_line_events"] + counters["n_escat_events"]
    survey_bytes = alg_bytes(counters, n)  # what the reference's loop touches for the same packets (SURVEY.md §8d)
    cap = read_capture(workload_key(spec, algorithm))
    traffic = None if cap is None else cap["bytes"] * n / cap["packets"]
    if algorithm == "scan":
        achieved = survey_bytes / (k_ms * 1e-3) / 1e9
        definition = ("streaming kernel: achieved = SURVEY.md §8(d) bytes (48 B per line-step + 32 B per event + macro-atom terms + "
                      "56 B per packet) / kernel time; the L2 serves part of the stream, so it can exceed the DRAM peak")
    else:
        # the jump algorithm never streams the line list (O(log) probes per trace instead of O(lines) steps): the §8(d)
        # bytes are not moved, so the fraction of the HBM roofline is taken on the DRAM bytes the kernel does move
        achieved = None if traffic is None else traffic / (k_ms * 1e-3) / 1e9
        definition = ("jump kernel: achieved = DRAM bytes per launch (ncu dram__bytes_read.sum + dram__bytes_write.sum of the committed "
                      "capture of this workload, per packet x this launch's packets) / kernel time measured here.  The kernel is bound "
                      "by latency / issue slots, not bandwidth: see issue_active_pct, lanes_per_instruction, occupancy_pct "
                      "(same capture).  survey_8d_* = the SURVEY.md §8(d) byte count of the SAME packets (what the streaming "
                      "formulation would move) / this kernel's time -- not a bandwidth claim")
    own = (40 * counters["n_search_probes"] + 160 * events + 8 * counters["n_macro_scanned"] + 24 * counters["n_macro_jumps"]
           + 16 * counters["n_vpackets"] * 8 + 56 * n)
    block = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": None if achieved is None else achieved / peak,
             "traffic": traffic, "kernel": kernel_name(spec, algorithm), "kernel_ms": k_ms, "peak_source": peak_src,
             "definition": definition, "binding_resource": "hbm/l2 streaming" if algorithm == "scan" else "latency / issue slots",
             "survey_8d_bytes_per_launch": survey_bytes, "survey_8d_GBps": survey_bytes / (k_ms * 1e-3) / 1e9,
             "survey_8d_frac_of_peak": survey_bytes / (k_ms * 1e-3) / 1e9 / peak,
             "own_model_bytes_per_launch": own,
             "per_packet": {"line_steps": counters["n_line_steps"] / max(n, 1), "events": events / max(n, 1),
                            "search_probes": counters["n_search_probes"] / max(n, 1),
                            "vpackets": counters["n_vpackets"] / max(n, 1)}}
    if cap is not None:
        block.update({"traffic_capture": {k: cap.get(k) for k in ("packets", "source", "l2_hit_pct", "dram_bytes_per_packet")},
                      "issue_active_pct": cap.get("issue_active_pct"), "lanes_per_instruction": cap.get("lanes_per_instruction"),
                      "occupancy_pct": cap.get("occupancy_pct"), "registers_per_thread": cap.get("registers_per_thread")})
    return block


class Rig:
    """What all legs share: the engine, the rank's pinned host packets, torch.distributed."""

    def __init__(self, args, rank, world, local_rank):
        import torch

        from tardis_b200.engine import Engine

        self.torch = torch
        self.args, self.rank, self.world, self.local_rank = args, rank, world, local_rank
        self.dist = None
        if world > 1:
            import torch.distributed as dist

            import datetime

            # rank 0 alone runs the CPU legs (oracle samples, table parity) between two collectives: the other ranks wait there
            dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local_rank}"), timeout=datetime.timedelta(minutes=30))
            self.dist = dist
        self.eng = Engine(local_rank)
        self.eng.set_option("algorithm", {"scan": 0, "jump": 1}[args.algorithm])
        self.pins = None
        self.out_pins = {}
        self.peak, self.peak_src = read_peak()

    def ensure_packets(self, n, r_inner0):
        """pinned host packets of this rank (first n used by a leg); generated once for the largest leg"""
        if self.pins is not None and len(self.pins[0][1]) >= n:
            return
        torch = self.torch
        pk = make_packets_chunked(n, r_inner0, syn.BASE_SEED + 1000 * self.rank)
        self.pins = []
        for f in ("initial_radii", "initial_nus", "initial_mus", "initial_energies", "packet_seeds"):
            a = getattr(pk, f)
            t = torch.empty(a.shape, dtype=torch.float64 if a.dtype == np.float64 else torch.int64, pin_memory=True)
            v = t.numpy()
            v[...] = a
            self.pins.append((t, v))
        self.r_inner0 = r_inner0

    def host_in(self, n):
        return [v[:n] for _, v in self.pins]

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.dist is not None:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x: float) -> float:
        if self.dist is None:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device=f"cuda:{self.local_rank}")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def out_buffers(self, n):
        torch = self.torch
        shapes = self.eng.output_shapes(n)
        key = tuple(sorted((k, v) for k, v in shapes.items()))
        if self.out_pins.get("key") != key:
            self.out_pins = {"key": key, "t": {k: torch.empty(shape, dtype=torch.float64, pin_memory=True) for k, shape in shapes.items()}}
        return {k: t.numpy() for k, t in self.out_pins["t"].items()}


DUMP_SAMPLE = 1 << 20  # entries kept per dumped array: four sampled arrays of 8 MB each keep a dump near 32 MB
DUMP_SEED = 20240917


def dump_outputs(res: dict, out_dir: str):
    """What the caller of the timed path receives after its last step (`res`: the engine's download of it), as
    <out_dir>/<name>.npy in float64: the per-packet outputs, the estimators, the fused spectra and luminosity sums, and the work
    counters.  An array larger than DUMP_SAMPLE entries is reduced to the same seeded, sorted sample of its flattened entries on
    every run, so two builds can be compared output for output."""
    os.makedirs(out_dir, exist_ok=True)
    res = dict(res)
    counters = res.pop("counters")
    res["counters"] = np.array([counters[k] for k in sorted(counters)], dtype=np.float64)  # sorted counter names
    for name, a in res.items():
        a = np.asarray(a, dtype=np.float64)
        if a.size > DUMP_SAMPLE:
            idx = np.sort(np.random.default_rng(DUMP_SEED).choice(a.size, DUMP_SAMPLE, replace=False))
            a = a.ravel()[idx]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def measure(rig: Rig, spec: dict, model, steps: int, warmup: int, e2e_steps: int, with_clocks: bool, device_source: bool,
            dump_dir: str | None = None):
    """One workload on this rank's engine: resident steps, end-to-end steps, cross-rank check.  Returns the leg's dict
    (rank 0 adds roofline / cpu_baseline / parity afterwards).  With `dump_dir`, rank 0 writes what the last timed step computed
    there (dump_outputs) before anything else runs on the engine."""
    from tardis_b200 import parallel

    torch, dist, eng, world, args = rig.torch, rig.dist, rig.eng, rig.world, rig.args
    if spec["scaling"] == "strong":
        lo, hi = parallel.shard_bounds(spec["packets_total"], rig.rank, world)
        n = hi - lo
        n_total = spec["packets_total"]
    else:
        n = spec["packets_per_gpu"]
        n_total = n * world
    eng.set_model_from(model, number_of_vpackets=spec["vpackets"])
    est_tensor = parallel.estimator_tensor(eng)  # (re-fetched after every set_model)
    rig.ensure_packets(n, model.r_inner[0])
    host_in = rig.host_in(n)

    def resident_step():
        eng.transport(True)
        eng.sync()
        if dist is not None:
            # the collective of an MC iteration: int64 words of the line estimators (exact) + f64 rest
            parallel.all_reduce_estimators(eng, dist)

    # ---- device-resident measurement ----
    eng.upload_packets(*host_in)
    for _ in range(warmup):
        resident_step()
    sampler = ClockSampler(rig.local_rank) if with_clocks else None
    launches0 = eng.kernel_launches()
    rig.barrier()
    if sampler:
        sampler.start()
    t0 = time.perf_counter()
    kernel_ms = []
    for _ in range(steps):
        resident_step()
        kernel_ms.append(eng.last_kernel_ms())
    rig.barrier()
    elapsed = rig.max_over_ranks(time.perf_counter() - t0)
    clocks = sampler.stop() if sampler else None
    launches = eng.kernel_launches() - launches0
    counters = eng.counters()
    value = n_total * steps / elapsed
    if dump_dir is not None and rig.rank == 0:
        dump_outputs(eng.download(), dump_dir)

    # ---- cross-rank check of the collective (N > 1): sum over ranks of the local buffers == the all-reduced buffer ----
    cross = None
    if dist is not None:
        eng.transport(True)
        eng.sync()
        lay = eng.estimator_layout()
        local = est_tensor.clone()
        dist.all_reduce(est_tensor)
        torch.cuda.synchronize()
        S = lay["n_shells"]
        head = slice(lay["off_j"], lay["off_j"] + 2 * S)  # J and nu_bar rows, gathered and summed on the host in float64
        gathered = [torch.empty_like(local[head]) for _ in range(world)]
        dist.all_gather(gathered, local[head].contiguous())
        host_sum = np.sum([g.cpu().numpy() for g in gathered], axis=0)
        reduced_head = est_tensor[head].cpu().numpy()
        tot_local = local.sum()
        dist.all_reduce(tot_local)
        tot_reduced = float(est_tensor.sum().item())
        # the product's collective (parallel.all_reduce_estimators): line estimators through their integer words -> the
        # finalised J_blue / Edotlu must be bit-identical on every rank
        eng.transport(True)
        exact = parallel.all_reduce_estimators(eng, dist)
        lines = est_tensor[lay["off_j_blue"]:]
        lo_t, hi_t = lines.clone(), lines.clone()
        dist.all_reduce(lo_t, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi_t, op=dist.ReduceOp.MAX)
        lines_identical = bool(torch.equal(lo_t, hi_t))
        del lo_t, hi_t
        cross = {"line_estimators_exact_int64_path": bool(exact), "line_estimators_identical_on_all_ranks": lines_identical,
                 "j_nubar_max_rel_err": max_rel_err(reduced_head, host_sum),
                 "buffer_sum_rel_err": abs(tot_reduced - float(tot_local.item())) / max(abs(tot_reduced), 1e-300),
                 "n_doubles": lay["n_doubles"], "ranks": world}

    # ---- end-to-end through the reference-facing call with host buffers ----
    L, S, G = model.n_lines, model.n_shells, len(model.spectrum_frequency_grid)
    h2d_bytes = int(sum(v.nbytes for v in host_in))
    d2h_bytes = int(2 * n * 8 + (2 * S + 2 * L * S + G + 2 * (G - 1) + 4) * 8)
    if spec["continuum"]:
        d2h_bytes += int((5 * len(model.continuum.bf_threshold_list_nu) * S + S) * 8)
    host_out = rig.out_buffers(n)
    eng.run(*host_in, buffers=host_out)  # warm-up (also sizes the staging buffers)
    rig.barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        eng.run(*host_in, buffers=host_out)
        if dist is not None:
            parallel.all_reduce_estimators(eng, dist)
    rig.barrier()
    e2e_elapsed = rig.max_over_ranks(time.perf_counter() - t0)
    e2e = {"value": n_total * e2e_steps / e2e_elapsed, "unit": "packets/s", "h2d_bytes_per_step": h2d_bytes,
           "d2h_bytes_per_step": d2h_bytes, "steps": e2e_steps, "device_source": None, "fused_spectrum_only": None}

    # same call, but the caller only wants the estimators and the fused spectrum histograms (no per-packet D2H)
    lean_steps = max(1, min(e2e_steps, 3))
    rig.barrier()
    t0 = time.perf_counter()
    for _ in range(lean_steps):
        eng.run(*host_in, per_packet=False, buffers={k: v for k, v in host_out.items() if not k.startswith("output_")})
        if dist is not None:
            parallel.all_reduce_estimators(eng, dist)
    rig.barrier()
    lean_elapsed = rig.max_over_ranks(time.perf_counter() - t0)
    e2e["fused_spectrum_only"] = {"value": n_total * lean_steps / lean_elapsed, "d2h_bytes_per_step": d2h_bytes - 2 * n * 8, "steps": lean_steps,
                                  "note": "same call without the per-packet output arrays: estimators, luminosity sums and the in-kernel "
                                          "emitted/reabsorbed spectrum histograms come back (SURVEY.md §8f rank 2)"}

    # the same step fed by the device-side packet source (SURVEY.md §8f rank 1).  Inputs per step: a seed.  The continuum
    # mode starts from BlackBodySimpleSourceRelativistic, as the reference's IIP workflow does.
    if device_source:
        t_inner = 1.0e4
        beta = (float(model.r_inner[0]) / float(model.time_explosion)) / syn.C_SPEED_OF_LIGHT if spec["continuum"] else None
        ds_steps = max(1, min(e2e_steps, 3))
        lean_buffers = {k: v for k, v in host_out.items() if not k.startswith("output_")}

        def ds_loop(per_packet):
            rig.barrier()
            t0 = time.perf_counter()
            for i in range(ds_steps):
                eng.create_packets(n, syn.BASE_SEED + 1000 * rig.rank + i + 1, float(model.r_inner[0]), t_inner, beta=beta)
                if per_packet:  # tb200_run_resident: the outputs of packet range c-1 go back while range c computes
                    eng.run_resident(buffers=host_out)
                else:
                    eng.run_resident(per_packet=False, buffers=lean_buffers)
                if dist is not None:
                    parallel.all_reduce_estimators(eng, dist)
            rig.barrier()
            return rig.max_over_ranks(time.perf_counter() - t0)

        eng.create_packets(n, syn.BASE_SEED + 1000 * rig.rank, float(model.r_inner[0]), t_inner, beta=beta)  # warm-up
        eng.transport(True); eng.sync()
        ds_elapsed = ds_loop(True)
        ds_lean_elapsed = ds_loop(False)
        e2e["device_source"] = {"value": n_total * ds_steps / ds_elapsed, "unit": "packets/s", "h2d_bytes_per_step": 64,
                                "d2h_bytes_per_step": d2h_bytes, "steps": ds_steps,
                                "fused_spectrum_only": {"value": n_total * ds_steps / ds_lean_elapsed, "d2h_bytes_per_step": d2h_bytes - 2 * n * 8},
                                "note": "packets generated in HBM by tb200_create_packets (BlackBody source on the device, T = 1e4 K"
                                        + (", relativistic variant" if beta is not None else "") + "); generation, transport and the D2H of "
                                        "the results run back to back; fused_spectrum_only = the same without the per-packet output arrays"}

    return {"workload": workload_text(spec), "scaling": spec["scaling"], "packets_per_step": n_total, "packets_this_rank": n,
            "value": value, "unit": "packets/s", "steps": steps, "warmup": warmup, "ms_per_step": elapsed / steps * 1e3,
            "gpu_launches": int(launches), "kernel_ms_mean": float(np.mean(kernel_ms)), "e2e": e2e, "clocks": clocks,
            "cross_rank_check": cross, "counters": counters, "_n": n}


def parity_and_cpu(rig: Rig, spec: dict, model, leg: dict, target_seconds: float, calibrate: bool, seed: int):
    """rank 0: the CPU oracle on a bounded sample (cpu_baseline, N = 1 only as a rate; always as the checker) and the
    engine's results for the same packets: spectrum L2 and max relative error of the estimators (SURVEY.md §8d)."""
    n_threads = os.cpu_count() or 1
    vp = spec["vpackets"]
    rate, ns, dt, sample, ref, used = cpu_leg(model, n_threads, seed, vp, target_seconds=target_seconds, calibrate=calibrate)
    cpu = {"value": rate, "unit": "packets/s", "cores": used, "kind": "port",
           "sample": f"{ns} packets of the same workload in {dt:.1f} s (oracle/tardis_oracle.c restatement of the "
                     f"reference loop; fastest calibrated configuration on {n_threads} host cores: {cpu_leg.last_choice})"}
    g = rig.eng.run_packets(sample)
    grid, tsim = model.spectrum_frequency_grid, sample.time_of_simulation
    spec_ref = histogram_spectrum(ref["output_nus"], ref["output_energies"], grid, tsim)
    spec_gpu = histogram_spectrum(g["output_nus"], g["output_energies"], grid, tsim)
    reab_ref = histogram_spectrum(ref["output_nus"], ref["output_energies"], grid, tsim, emitted=False)
    parity = {"sample_packets": ns,
              "spectrum_l2_vs_oracle": rel_l2(spec_gpu, spec_ref),
              # the kernel epilogue's own histograms and sums against the ORACLE's per-packet outputs
              "fused_spectrum_l2_vs_oracle": rel_l2(g["spectrum_emitted"] / tsim, spec_ref),
              "fused_reabsorbed_spectrum_l2_vs_oracle": rel_l2(g["spectrum_reabsorbed"] / tsim, reab_ref),
              "luminosity_sum_rel_err": abs(g["luminosity_sums"][0] - ref["output_energies"][ref["output_energies"] >= 0].sum())
              / max(ref["output_energies"][ref["output_energies"] >= 0].sum(), 1e-300),
              "max_rel_err": {k: max_rel_err(g[k], ref[k]) for k in ("j", "nu_bar", "j_blue", "edotlu")},
              "counters_equal": all(g["counters"][k] == v for k, v in ref["counters"].items()),
              "packet_outputs_max_rel_err": max_rel_err(g["output_nus"], ref["output_nus"])}
    if vp:
        parity["virtual_spectrum_l2_vs_oracle"] = rel_l2(g["vhist"][:-1], ref["vhist"][:-1])
    if spec["continuum"]:
        parity["max_rel_err"].update({k: max_rel_err(g[k], ref[k]) for k in
                                      ("photo_ion_estimator", "stim_recomb_estimator", "bf_heating_estimator",
                                       "stim_recomb_cooling_estimator", "ff_heating_estimator")})
        parity["photo_ion_statistics_equal"] = bool(np.array_equal(g["photo_ion_estimator_statistics"], ref["photo_ion_estimator_statistics"]))
    return cpu, parity


def formal_integral_work(r_inner, r_outer, time_explosion, line_list_nu, frequencies, points: int, interpolate_shells: int = 0) -> dict:
    """Exact amount of work of one formal integral (analysis for the bench line; nothing here is on the product path): the
    resonance points every ray passes -- the lines with nu z_last < nu_line <= nu z_first, z the Doppler factors of the first and
    the last intersection point of the ray (formal_integral_numba.py:54-118, :472-536) -- and the sweep steps of the kernel's warps
    (32 neighbouring impact parameters of one frequency pass the union of their windows once)."""
    r_inner, r_outer = np.asarray(r_inner, dtype=np.float64), np.asarray(r_outer, dtype=np.float64)
    n_radii = interpolate_shells if interpolate_shells != 0 else max(2 * len(r_inner), 80)  # formal_integral_solver.py:208-214
    if n_radii > 0:
        radius = np.linspace(r_inner[0], r_outer[-1], n_radii)
        r_in, r_out = radius[:-1], radius[1:]
    else:
        r_in, r_out = r_inner, r_outer
    c_inv, inv_t = 3.33564e-11, 1.0 / float(time_explosion)  # spectrum/formal_integral/base.py:12
    p = np.arange(points, dtype=np.float64) * r_out[-1] / (points - 1)  # base.py:101
    ip = lambda r: np.where(r > p, np.sqrt(np.maximum(r * r - p * p, 0.0)) * c_inv * inv_t, 0.0)  # noqa: E731
    z_last = 1.0 - ip(r_out[-1])
    z_first = np.where(p <= r_in[0], 1.0 - ip(r_out[0]), 1.0 + ip(r_out[-1]))
    integrated = (np.arange(points) >= 1) & (p < r_out[-1])  # p = 0 is never integrated; p = r_max has no intersection
    if len(r_out) == 1:
        integrated &= p > r_in[0]  # a photosphere ray through a single shell has one point: no segment
    nu_desc = np.asarray(line_list_nu, dtype=np.float64)
    neg = -nu_desc  # ascending
    freq = np.asarray(frequencies, dtype=np.float64)
    n_points = n_steps = 0
    n_blocks = (points - 1 + 31) // 32
    pad = n_blocks * 32 + 1 - points
    for lo in range(0, len(freq), 256):
        f = freq[lo:lo + 256, None]
        first = np.searchsorted(neg, -(f * z_first[None, :]), side="left")   # entries > nu_start
        last = np.searchsorted(neg, -(f * z_last[None, :]), side="left")     # entries > nu_end of the last segment
        last = np.maximum(last, first)
        cnt = np.where(integrated[None, :], last - first, 0)
        n_points += int(cnt.sum())
        big = len(nu_desc) + 1
        a = np.where(integrated[None, :], first, big)[:, 1:]
        b = np.where(integrated[None, :], last, 0)[:, 1:]
        a = np.pad(a, ((0, 0), (0, pad)), constant_values=big).reshape(len(f), n_blocks, 32)
        b = np.pad(b, ((0, 0), (0, pad)), constant_values=0).reshape(len(f), n_blocks, 32)
        # a warp's lanes have nested windows (both ends are monotone in p on either side of the photosphere), so the union of
        # the windows is one interval except for the one warp that straddles the photosphere's edge: counted as the hull there
        span = np.maximum(b.max(axis=2) - a.min(axis=2), 0)
        n_steps += int(span.sum())
    return {"resonance_points": n_points, "warp_sweep_steps": n_steps, "rays": int(integrated.sum()) * len(freq),
            "integrator_shells": int(len(r_out))}


def tables_block(rig, model, with_cpu: bool):
    """Per-iteration table preparation either side of the MC loop (SURVEY.md §8f ranks 3 and 4), timed on the bench model's
    line list: (a) the reference's way -- the plasma writes [L,S] tau_sobolev and [T,S] transition probabilities on the host
    and `tb200_set_model` uploads and prepares them; (b) this engine's way -- the estimators of the last iteration are turned
    into T_rad / W / J_blue where they lie (`tb200_solve_radiation_field`) and tau / beta / macro-atom probabilities are built
    in HBM from the level populations (`tb200_build_opacity`); only [n_levels,S] populations cross PCIe."""
    from tardis_b200.engine import Engine

    out = {}
    try:
        L, S = model.n_lines, model.n_shells
        eng = Engine(rig.local_rank)
        host_ms = []
        for _ in range(3):
            t0 = time.perf_counter()
            eng.set_model_from(model)
            eng.sync()
            host_ms.append((time.perf_counter() - t0) * 1e3)
        eng.close()
        mac = model.macro
        tp = getattr(mac, "transition_probabilities", None)
        out["host_tables"] = {"call": "tb200_set_model with tau_sobolev [L,S] and transition_probabilities [T,S] in host memory",
                              "ms": float(min(host_ms[1:])), "first_call_ms": float(host_ms[0]),
                              "h2d_bytes": int(model.tau_sobolev.nbytes + (0 if tp is None else np.asarray(tp).nbytes))}

        n_levels = 3000
        atomic = syn.make_atomic_data(model.line_list_nu, n_levels, "macroatom", nlte_fraction=0.0)
        plasma = syn.make_plasma_state(atomic, S, model.time_explosion, zero_fraction=0.0, inversion_fraction=0.0, noise=0.0)
        plasma.level_number_density *= 1e-9  # optical depths of order one
        eng = Engine(rig.local_rank)
        eng.set_option("keep_opacity_tables", 1)  # the normalised probabilities stay next to their running sums (source function)
        eng.set_model(r_inner=model.r_inner, r_outer=model.r_outer, time_explosion=model.time_explosion,
                      electron_density=model.electron_density, line_list_nu=model.line_list_nu, tau_sobolev=None,
                      line_interaction_type="macroatom", transition_probabilities=None,
                      line2macro_level_upper=atomic.line2macro_level_upper, macro_block_edge_index=atomic.macro_block_edge_index,
                      transition_type=atomic.transition_type, destination_level_id=atomic.destination_level_id,
                      transition_line_id=atomic.transition_line_idx, spectrum_frequency_grid=model.spectrum_frequency_grid)
        eng.set_atomic_data(lines_lower_level_index=atomic.lower_level, lines_upper_level_index=atomic.upper_level, g=atomic.g,
                            metastability=atomic.metastable, wavelength_cm=atomic.wavelength_cm, f_lu=atomic.f_lu, f_ul=atomic.f_ul,
                            energy_lower=atomic.energy[atomic.lower_level], energy_upper=atomic.energy[atomic.upper_level],
                            nlte_line=atomic.nlte_line)
        eng.build_opacity(plasma.level_number_density, plasma.time_explosion, plasma.j_blues)  # iteration 0: J_blue from the host
        n_small = 200_000
        pk = syn.make_packets(n_small, model.r_inner[0], base_seed=syn.BASE_SEED + 31)
        eng.upload_packets(pk.initial_radii, pk.initial_nus, pk.initial_mus, pk.initial_energies, pk.packet_seeds)
        volume = 4.0 / 3.0 * np.pi * (model.r_outer ** 3 - model.r_inner ** 3)
        rad_ms, build_ms = [], []
        for _ in range(4):
            eng.transport(True)
            eng.sync()
            t0 = time.perf_counter()
            eng.solve_radiation_field(time_explosion=model.time_explosion, time_of_simulation=1.0e5, volume=volume, want_j_blues=False)
            eng.sync()
            t1 = time.perf_counter()
            eng.build_opacity(plasma.level_number_density, plasma.time_explosion)  # J_blue: the table the solve left in HBM
            eng.sync()
            t2 = time.perf_counter()
            rad_ms.append((t1 - t0) * 1e3)
            build_ms.append((t2 - t1) * 1e3)
        # the step after the LAST iteration: the formal integral's source function from the resident estimators
        sf_ms, sf_all_ms, sf_it = [], [], 0
        sf_args = dict(time_explosion=model.time_explosion, time_of_simulation=1.0e5, volume=volume, wavelength_cm=atomic.wavelength_cm,
                       lines_lower_level_idx=atomic.lower_level, lines_upper_level_idx=atomic.upper_level, n_levels=n_levels)
        for _ in range(3):
            t0 = time.perf_counter()
            sf_it = eng.solve_source_function(want=(), **sf_args)["iterations"]
            t1 = time.perf_counter()
            sf_tables = eng.solve_source_function(**sf_args)
            t2 = time.perf_counter()
            sf_ms.append((t1 - t0) * 1e3)
            sf_all_ms.append((t2 - t1) * 1e3)
        out["source_function"] = {"call": "tb200_solve_source_function on the resident estimators (e_dot_u, the per-shell macro-atom system by "
                                          "fixed-point sweeps, att_S_ul / Jred_lu / Jblue_lu)",
                                  "ms_tables_left_in_hbm": float(min(sf_ms[1:])), "ms_with_three_LS_tables_downloaded": float(min(sf_all_ms[1:])),
                                  "sweeps": int(sf_it), "reference": "SourceFunctionSolver.solve: pandas group-by + one scipy spsolve of an "
                                  "n_levels x n_levels system per shell (1.5 s per shell at this size in the build container)"}
        if with_cpu:  # parity of that solve at THIS size against the oracle (numpy + one scipy spsolve per shell): three of the shells
            try:
                from oracle import source_function_oracle as sfo

                op = eng.download_opacity(transition_probabilities=True)
                est = eng.download(per_packet=False)
                pick = sorted({0, S // 2, S - 1})
                t0 = time.perf_counter()
                want = sfo.solve(atomic, op["tau_sobolev"][:, pick], op["transition_probabilities"][:, pick], est["j_blue"][:, pick], est["edotlu"][:, pick],
                                 float(model.time_explosion), 1.0e5, volume[pick], "macroatom")
                cpu_s = time.perf_counter() - t0
                par = {"shells_checked": [int(x) for x in pick], "bar": "|got - ref| <= 1e-11 |ref| + 1e-14 max|table| (tests/test_source_function.py)",
                       "cpu_oracle_s_per_shell": cpu_s / len(pick)}
                for k in ("att_S_ul", "Jred_lu", "Jblue_lu"):
                    a, b = np.asarray(sf_tables[k])[:, pick], want[k]
                    top = float(np.max(np.abs(b)))
                    par[k] = {"max_err_over_bar": float(np.max(np.abs(a - b) / (1e-11 * np.abs(b) + 1e-14 * top))) if top > 0 else 0.0,
                              "max_abs_err_over_table_max": float(np.max(np.abs(a - b)) / top) if top > 0 else 0.0,
                              "zero_pattern_equal": bool(np.array_equal(a == 0, b == 0))}
                out["source_function"]["parity"] = par
            except Exception as exc:
                out["source_function"]["parity"] = {"error": f"{type(exc).__name__}: {exc}"}
        # ... and the formal integral itself on the tables that solve left in HBM: the reference's spectrum grid (10 000 frequencies),
        # its default 1000 impact parameters, max(2 S, 80) - 1 interpolated shells
        try:
            grid = np.asarray(model.spectrum_frequency_grid, dtype=np.float64)
            fi_freq, fi_points, fi_t_inner = grid[:-1].copy(), 1000, 1.0e4
            # guard the bench's wall time: a 1-in-20 sample of the grid first (it also pays the allocations); if the whole grid would take
            # more than a minute and a half, a uniform subset of it is integrated instead and n_frequencies says so
            probe = fi_freq[:: max(1, len(fi_freq) // 500)]
            fi_probe = eng.formal_integral(inner_temperature=fi_t_inner, frequencies=probe, points=fi_points, interpolate_shells=0)
            est_full_ms = fi_probe["integral_ms"] * len(fi_freq) / max(1, len(probe))
            if est_full_ms > 90_000.0:
                fi_freq = fi_freq[:: int(np.ceil(est_full_ms / 90_000.0))].copy()
            fi_wall, fi_res = [], None
            for _ in range(2 if est_full_ms < 30_000.0 else 1):
                t0 = time.perf_counter()
                fi_res = eng.formal_integral(inner_temperature=fi_t_inner, frequencies=fi_freq, points=fi_points, interpolate_shells=0)
                fi_wall.append((time.perf_counter() - t0) * 1e3)
            n_int_shells = max(2 * S, 80) - 1
            fi = {"call": "tb200_formal_integral on the resident source-function tables (interpolation to the integrator's shells as 32-byte "
                          "cells, one warp per 32 impact parameters of a frequency, trapezoid)",
                  "n_frequencies": int(len(fi_freq)), "n_impact_parameters": fi_points, "integrator_shells": n_int_shells,
                  "interpolation_ms": float(fi_res["interpolation_ms"]), "integral_ms": float(fi_res["integral_ms"]),
                  "wall_ms_incl_d2h": float(min(fi_wall)), "first_call_wall_ms": float(fi_wall[0]),
                  "probe": {"n_frequencies": int(len(probe)), "integral_ms": float(fi_probe["integral_ms"]), "estimate_for_the_grid_ms": float(est_full_ms)},
                  "frequencies_per_s": float(len(fi_freq) / (fi_res["integral_ms"] * 1e-3)) if fi_res["integral_ms"] > 0 else None,
                  "cells_bytes": int(n_int_shells * (L + 2) * 32),
                  "reference": "FormalIntegralSolver.solve: scipy interp1d of four [L,S] tables to [L,79] on the host (1.3 GB), then "
                               "numba_formal_integral (prange over frequencies) or the Numba-CUDA kernel (one thread per ray)"}
            try:  # what the kernel had to do, counted exactly on the host: bytes per resonance point -> the L2-side roofline
                wk = formal_integral_work(model.r_inner, model.r_outer, float(model.time_explosion), model.line_list_nu, fi_freq, fi_points, 0)
                alg = 32 * wk["resonance_points"] + 8 * wk["warp_sweep_steps"]
                sec = fi_res["integral_ms"] * 1e-3
                fi["work"] = wk
                fi["roofline"] = {"bound": "L2 bandwidth / fp64 issue: the cells of one frequency's window (lines x integrator shells x 32 B) stay in "
                                           "L2 and consecutive frequencies share them; HBM sees each cell about once",
                                  "algorithmic_bytes": int(alg), "bytes_per_resonance_point": 32, "bytes_per_warp_step": 8,
                                  "achieved": alg / sec / 1e9 if sec > 0 else None, "unit": "GB/s (L2-served)",
                                  "hbm_peak": rig.peak, "x_hbm_peak": alg / sec / 1e9 / rig.peak if sec > 0 else None,
                                  "distinct_cell_bytes": int(n_int_shells * (L + 2) * 32),
                                  "resonance_points_per_s": wk["resonance_points"] / sec if sec > 0 else None,
                                  "lanes_busy_per_sweep_step": wk["resonance_points"] / max(1, wk["warp_sweep_steps"]), "traffic": None}
            except Exception as exc:
                fi["roofline"] = {"error": f"{type(exc).__name__}: {exc}"}
            if with_cpu:  # the C restatement of numba_formal_integral on a bounded sample of the same frequencies (oracle/: CPU baseline leg only)
                from oracle import formal_integral_oracle as fio

                sample = np.linspace(0, len(fi_freq) - 1, 66).astype(int)[1:-1]  # 64 frequencies inside the grid
                tau_host = eng.download_opacity()["tau_sobolev"]
                r_in_i, r_out_i = fio.interpolated_radii(model.r_inner, model.r_outer, 0)
                t0 = time.perf_counter()
                att_i, jred_i, jblue_i, tau_i, ne_i = fio.interpolate_integrator_quantities(model.r_inner, model.r_outer, r_in_i, r_out_i, sf_tables["att_S_ul"],
                                                                                       sf_tables["Jred_lu"], sf_tables["Jblue_lu"], tau_host, model.electron_density)
                t1 = time.perf_counter()
                lum, _ = fio.integrate(r_in_i, r_out_i, float(model.time_explosion), model.line_list_nu, fi_t_inner, fi_freq[sample], att_i, jred_i, jblue_i, tau_i, ne_i, fi_points)
                t2 = time.perf_counter()
                got = fi_res["luminosity_densities"][sample]
                c_s = getattr(fio.integrate, "last_c_seconds", t2 - t1)
                fi["cpu_baseline"] = {"kind": "port", "cores": 1, "sample": f"{len(sample)} of the {len(fi_freq)} frequencies, all {fi_points} impact parameters",
                                      "interpolation_ms_scipy": (t1 - t0) * 1e3, "table_preparation_ms": (t2 - t1 - c_s) * 1e3,
                                      "frequencies_per_s": float(len(sample) / c_s), "unit": "frequencies/s (integrator alone, oracle/formal_integral_oracle.c)",
                                      "seconds_for_this_grid": (t1 - t0) + (t2 - t1 - c_s) + len(fi_freq) * c_s / len(sample),
                                      "reference_numba": "17.8 / 106 frequencies/s at 1 / 8 threads in the build container (profiles/r02_reference_formal_integral_rate.json)"}
                fi["parity"] = {"max_rel_err_L_nu_vs_oracle": float(np.max(np.abs(got - lum) / np.abs(lum))), "frequencies_checked": int(len(sample))}
            out["formal_integral"] = fi
        except Exception as exc:
            out["formal_integral"] = {"error": f"{type(exc).__name__}: {exc}"}
        op_host = None
        if with_cpu:
            try:
                op_host = eng.download_opacity()
            except Exception:
                op_host = None
        eng.close()
        out["device_tables"] = {"call": "tb200_solve_radiation_field (resident estimators) + tb200_build_opacity (populations [n_levels,S] from the host)",
                                "solve_radiation_field_ms": float(min(rad_ms[1:])), "build_opacity_ms": float(min(build_ms[1:])),
                                "ms": float(min(rad_ms[1:]) + min(build_ms[1:])), "h2d_bytes": int(plasma.level_number_density.nbytes),
                                "n_levels": n_levels, "n_transitions": int(len(atomic.transition_type))}
        out["n_lines"], out["n_shells"] = int(L), int(S)
        if with_cpu:  # the numpy restatement of the reference's per-iteration table build, on this host (oracle/: CPU baseline leg only)
            from oracle import opacity_oracle

            t0 = time.perf_counter()
            ref_tabs = opacity_oracle.build(atomic, plasma)
            out["cpu_numpy_port_ms"] = (time.perf_counter() - t0) * 1e3
            if op_host is not None:  # tau / beta depend on the populations only (the probabilities also on the J_blue of the last solve)
                try:
                    tau_d, tau_r = op_host["tau_sobolev"], ref_tabs["tau_sobolev"]
                    beta_d, beta_r = op_host["beta_sobolev"], ref_tabs["beta_sobolev"]
                    out["device_tables"]["parity"] = {
                        "tau_sobolev_bit_identical": bool(np.array_equal(tau_d, tau_r)),
                        "tau_sobolev_max_rel_err": float(np.max(np.abs(tau_d - tau_r) / np.maximum(np.abs(tau_r), 1e-300))),
                        "beta_sobolev_max_rel_err": float(np.max(np.abs(beta_d - beta_r) / np.maximum(np.abs(beta_r), 1e-300))),
                        "against": "oracle/opacity_oracle.py (pinned on the reference's own tau / beta functions), all L x S cells"}
                except Exception as exc:
                    out["device_tables"]["parity"] = {"error": f"{type(exc).__name__}: {exc}"}
    except Exception as exc:  # a side measurement must never take the bench line down
        out["error"] = f"{type(exc).__name__}: {exc}"
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--packets", type=int, default=100_000_000, help="packets per GPU per step (headline)")
    ap.add_argument("--lines", type=int, default=500_000)
    ap.add_argument("--shells", type=int, default=20)
    ap.add_argument("--mode", default="macroatom", choices=["scatter", "downbranch", "macroatom"])
    ap.add_argument("--vpackets", type=int, default=0)
    ap.add_argument("--continuum", action="store_true", help="IIP mode (BASELINE config 5): bound-free / free-free continuum")
    ap.add_argument("--mu-tau", type=float, default=-7.5)
    ap.add_argument("--algorithm", default="jump", choices=["jump", "scan"],
                    help="jump: prefix-table search + range updates (default, fastest); scan: stream the line list")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-scan-reference", action="store_true", help="skip the short scan-kernel roofline measurement")
    ap.add_argument("--no-device-source", action="store_true", help="skip the e2e.device_source measurement")
    ap.add_argument("--device-source", action="store_true", help="(default now; kept for compatibility)")
    ap.add_argument("--no-tables", action="store_true", help="skip the per-iteration table preparation measurement")
    ap.add_argument("--legs", default=None,
                    help="comma list of the BASELINE legs to measure after the headline: 2,4,5,strong | all | none "
                         "(default: all when the headline is the default workload, none otherwise)")
    ap.add_argument("--leg-steps", type=int, default=3)
    ap.add_argument("--leg-scale", type=float, default=1.0, help="scale the legs' packet counts (quick runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the headline's last timed step computed to DIR/<name>.npy (float64; arrays above "
                         f"{DUMP_SAMPLE} entries as a fixed seeded sample)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs is not None and args.impl == "reference":
        ap.error("--dump-outputs needs --impl b200: the reference arm's sample size is calibrated from its timing")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.gpus != world and world > 1:
        args.gpus = world

    head = {"packets_per_gpu": args.packets, "packets_total": args.packets * world, "shells": args.shells, "lines": args.lines,
            "mode": args.mode, "vpackets": args.vpackets, "continuum": bool(args.continuum), "mu_tau": args.mu_tau, "scaling": "weak"}
    default_head = (args.packets == 100_000_000 and args.lines == 500_000 and args.shells == 20 and args.mode == "macroatom"
                    and args.vpackets == 0 and not args.continuum and args.algorithm == "jump")
    legs_arg = args.legs if args.legs is not None else ("all" if default_head else "none")
    leg_names = [] if legs_arg == "none" else (["2", "4", "5", "strong"] if legs_arg == "all" else [x for x in legs_arg.split(",") if x])

    def leg_spec(name):
        base = {"lines": args.lines, "mu_tau": args.mu_tau, "scaling": "strong", "vpackets": 0, "continuum": False, "shells": 20, "mode": "macroatom"}
        total = {"2": 10_000_000}.get(name, 100_000_000)
        total = max(world * 1000, int(total * args.leg_scale))
        if name == "2":
            base.update(mode="scatter")
        elif name == "4":
            base.update(vpackets=10)
        elif name == "5":
            base.update(continuum=True, shells=50)
        elif name != "strong":
            raise SystemExit(f"unknown leg {name}")
        base.update(packets_total=total, packets_per_gpu=-(-total // world))
        return base

    workload = workload_text(head)
    config = {"workload": workload, "packets_per_gpu": args.packets, "n_shells": args.shells, "n_lines": args.lines,
              "line_interaction_type": args.mode, "number_of_vpackets": args.vpackets, "continuum": bool(args.continuum),
              "algorithm": args.algorithm, "parallelism": f"packet-sharded x{args.gpus}",
              "l2_policy": "inputs larger than L2 (tables 80-400 MB + 56 B/packet of packet arrays per step, 5.6 GB at 1e8)",
              "timed_region": "per step: seed expansion + ordering kernels of the fresh packets, transport kernel, estimator epilogues, all-reduce"}

    # ------------------------------------------------------------------ reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return
        model = build_model(head)
        n_threads = os.cpu_count() or 1
        rates = []
        sample_n = 0
        used = 1
        for i in range(args.warmup + args.steps):
            rate, n, dt, _, _, used = cpu_leg(model, n_threads, syn.BASE_SEED + i, args.vpackets, target_seconds=8.0)
            sample_n = n
            if i >= args.warmup:
                rates.append((rate, dt))
        value = float(np.mean([r for r, _ in rates]))
        line = {"metric": METRIC, "value": value, "unit": "packets/s", "n_gpus": args.gpus, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": float(np.mean([d for _, d in rates]) * 1e3),
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": config, "impl": "reference",
                "cpu_baseline": {"value": value, "unit": "packets/s", "cores": used, "kind": "port",
                                 "sample": f"{sample_n} packets of the same workload per step (oracle/tardis_oracle.c; fastest of "
                                           f"the calibrated thread counts / table layouts on {n_threads} host cores: "
                                           f"{cpu_leg.last_choice}; the reference's Numba loop cannot travel to this box -- its "
                                           "rate measured in the build container is in BASELINE.md §2)"},
                "e2e": {"value": value, "unit": "packets/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(json_safe(line), allow_nan=False))
        return

    # ------------------------------------------------------------------ B200 arm
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    rig = Rig(args, rank, world, local_rank)
    t_start = time.perf_counter()

    model = build_model(head)
    # the rank's host packets are generated once, for the largest leg
    n_max = max([args.packets] + [leg_spec(nm)["packets_per_gpu"] for nm in leg_names])
    rig.ensure_packets(n_max, model.r_inner[0])
    use_ds = not args.no_device_source
    e2e_steps = max(1, args.steps)
    headline = measure(rig, head, model, args.steps, args.warmup, e2e_steps, with_clocks=True, device_source=use_ds,
                       dump_dir=args.dump_outputs)

    if rank == 0:
        n = headline["_n"]
        headline["roofline"] = roofline_block(head, args.algorithm, headline["counters"], n, headline["kernel_ms_mean"], rig.peak, rig.peak_src)
        # ---- the streaming ("scan") kernel on a slice of the same packets: its roofline on the SURVEY.md §8(d) bytes ----
        scan_block = None
        # (skipped with virtual packets: both kernels resolve a volley by prefix search, so the streaming byte count does not apply)
        if args.algorithm == "jump" and not args.no_scan_reference and not args.continuum and args.vpackets == 0:
            eng = rig.eng
            ns = int(min(n, max(2_000_000, n // 20)))
            eng.set_option("algorithm", 0)
            eng.upload_packets(*rig.host_in(ns))
            scan_ms = []
            for i in range(3):
                eng.transport(True)
                eng.sync()
                if i > 0:
                    scan_ms.append(eng.last_kernel_ms())
            sc = eng.counters()
            s_ms = float(np.mean(scan_ms))
            rb = roofline_block(head, "scan", sc, ns, s_ms, rig.peak, rig.peak_src)
            scan_block = {"kernel": "tb::transport_scan_kernel", "packets": ns, "kernel_ms": s_ms, "packets_per_s": ns / s_ms * 1e3, "roofline": rb}
            eng.set_option("algorithm", 1)
        headline["scan_kernel"] = scan_block
        cpu = parity = None
        if not args.no_cpu_baseline:
            cpu, parity = parity_and_cpu(rig, head, model, headline, 12.0, True, syn.BASE_SEED + 777)
        headline["cpu_baseline"], headline["parity"] = cpu, parity
        headline["tables"] = None
        if not args.no_tables and args.mode == "macroatom" and not args.continuum:
            headline["tables"] = tables_block(rig, model, with_cpu=not args.no_cpu_baseline)
    # (the scan reference and the CPU legs run on rank 0 only; the other ranks wait in the next leg's first collective)

    # ------------------------------------------------------------------ the BASELINE legs
    legs = {}
    for name in leg_names:
        spec = leg_spec(name)
        if name == "strong" and world == 1 and args.leg_scale == 1.0 and default_head:
            legs[name] = {"same_as_headline": True, "workload": workload_text(spec), "scaling": "strong",
                          "note": "at N = 1 the strong-scaling point (1e8 packets total) is the headline measurement"}
            continue
        same_model = (spec["shells"] == head["shells"] and spec["mode"] == head["mode"] and spec["continuum"] == head["continuum"]
                      and spec["lines"] == head["lines"])
        m = model if same_model else build_model(spec)
        leg = measure(rig, spec, m, max(1, args.leg_steps), 3, max(1, args.leg_steps), with_clocks=False, device_source=use_ds)
        if rank == 0:
            leg["roofline"] = roofline_block(spec, args.algorithm, leg["counters"], leg["_n"], leg["kernel_ms_mean"], rig.peak, rig.peak_src)
            if not args.no_cpu_baseline:
                cpu, parity = parity_and_cpu(rig, spec, m, leg, 6.0, False, syn.BASE_SEED + 778)
                if world > 1:
                    cpu["note"] = "rate of rank 0's host on the bounded sample; the N = 1 run is the stated CPU baseline"
                leg["cpu_baseline"], leg["parity"] = cpu, parity
        leg.pop("_n", None)
        legs[name] = leg
        del m

    if rank != 0:
        if rig.dist is not None:
            rig.dist.destroy_process_group()
        return

    headline.pop("_n", None)
    parity = headline.get("parity")
    line = {"metric": METRIC, "value": headline["value"], "unit": "packets/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": headline["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config,
            "clocks": headline["clocks"], "gpu_launches": headline["gpu_launches"], "e2e": headline["e2e"],
            "roofline": headline["roofline"], "scan_kernel": headline.get("scan_kernel"), "cpu_baseline": headline.get("cpu_baseline"),
            "spectrum_l2_vs_oracle": None if parity is None else parity["spectrum_l2_vs_oracle"], "parity": parity,
            "cross_rank_check": headline["cross_rank_check"], "counters": headline["counters"], "tables": headline.get("tables"),
            "configs": {k: v for k, v in legs.items() if k != "strong"}, "strong": legs.get("strong"),
            "bench_wall_s": time.perf_counter() - t_start}
    print(json.dumps(json_safe(line), allow_nan=False))
    if rig.dist is not None:
        rig.dist.destroy_process_group()


if __name__ == "__main__":
    main()
