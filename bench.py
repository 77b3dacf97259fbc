#!/usr/bin/env python
"""bench.py — scattering steps/s and s/iteration of the transport loop (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # CUDA arm; N>1 under torchrun, one rank per GPU
    python bench.py --impl reference --steps K --warmup W    # CPU arm: the C restatement of the reference loop

A "step" is one pass of the hot path over one batch: ONE ITERATION of one ion species — every pcut of
`main_loops.jl:179-317` — on the workload BASELINE.json quotes the metric on (configs[1]: unmodified planar
non-relativistic shock, protons, 1e6 particles per pcut, no smoothing).  Weak scaling: every GPU gets 1e6 particles
per pcut, sharded by contiguous index blocks with global RNG counters; the only collectives are one 8-byte
all-gather per pcut and one all-reduce of the packed tallies per ion (NCCL inside the library).

  value        scattering steps/s, population resident in HBM: total steps of all ranks / max-over-ranks device time of
               the pcut loops (CUDA events on the library's stream).
  e2e          the same through the C-ABI with HOST buffers: H2D of the population from pinned memory and D2H of the
               tallies inside the timed region (wall clock between synchronisations, max over ranks).
  roofline     the transport kernel against the FP64 pipe: steps x 185 flop (SURVEY 8d / DESIGN.md) / kernel time,
               over a DFMA peak measured live on this GPU (MEASURED_PEAKS.json has no FP64 entry).
  cpu_baseline the CPU oracle (C restatement; Julia is not available) on a bounded sample, all host threads.

--dump-outputs DIR writes what the last timed step handed back to its caller (per ion: the pcut counts of mcs_run_ion, the
tallies, scalars and counters of mcs_end_ion) as DIR/ion<i>_<name>.npy in float64, so that two builds run with the same
arguments, which see the same inputs, can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

FLOP_PER_STEP = 185.0  # SURVEY.md 8d, Appendix D; restated in DESIGN.md
# roofline.traffic = dram__bytes_read.sum + dram__bytes_write.sum of ONE transport-kernel launch, read from the tracked
# summary of the `ncu --set full` capture of this kernel on this workload (written by tools/ncu_summary.py --json from the
# .ncu-rep; tools/profile.sh).  Reported only when the capture matches the workload and the particle count; else null.
TRAFFIC_FILE = os.path.join(ROOT, "profiles", "r02_traffic.json")
METRIC = "scattering_steps_per_sec"
DUMP_BYTES = 64_000_000
DUMP_TALLIES = ("pxx_flux", "pxz_flux", "energy_flux", "psd", "num_crossings", "esc_psd_feb_upstream", "esc_psd_feb_downstream",
                "esc_energy_eff", "esc_num_eff", "weight_coupled", "spectra_coupled", "energy_transfer_pool", "spectra_sf",
                "spectra_pf")


def measured_traffic(workload, n_per_pcut):
    try:
        rec = json.load(open(TRAFFIC_FILE))
    except (OSError, ValueError):
        return None, None
    for r in rec.get("captures", []):
        if r.get("workload") == workload and int(r.get("n_per_pcut", -1)) == int(n_per_pcut):
            return (float(r["dram_bytes_read"]) + float(r["dram_bytes_write"]),
                    f"profiles/r02_traffic.json: {r.get('source', '?')} (launch {r.get('launch', '?')}, "
                    f"red sectors {r.get('lts_sectors_red')}, atom sectors {r.get('lts_sectors_atom')})")
    return None, None


def build_run(workload: str, n_per_pcut: int, pcuts: str = "bench"):
    from mcs_b200 import problem
    mk = {"planar": problem.planar_test_particle_input, "relativistic": problem.relativistic_input,
          "nonlinear": problem.nonlinear_input, "multi": problem.multi_species_input}[workload]
    kw = {"momentum_cutoffs": list(problem.DEFAULT_PCUTS)} if pcuts == "default" else {}
    inp = mk(n_per_pcut, **kw)
    inp.num_iterations = 1
    run = problem.setup_run(inp)
    prof = problem.synthetic_precursor(run) if workload == "nonlinear" else run.profile
    return run, prof


def workload_config(workload, run, n_per_pcut, extra=None):
    names = {"planar": "configs[1]: planar non-relativistic test-particle shock (u0=1e4 km/s), protons, unmodified profile",
             "relativistic": "configs[3]: gamma0=10 test-particle shock, protons",
             "nonlinear": "configs[2]: smoothed-precursor shock (r_comp=8), protons",
             "multi": "configs[4]: p+He+e-, gamma0=1.5"}
    c = {"workload": names[workload], "particles_per_pcut_per_gpu": n_per_pcut,
         "pcuts_mpc": [float(p) for p in run.inp.momentum_cutoffs], "n_grid": run.n_grid,
         "psd_bins": [run.num_psd_mom_bins + 2, run.num_psd_theta_bins + 2, run.n_grid],
         "xn_per": [run.inp.fine_scattering_Ng, run.inp.coarse_scattering_Ng], "rng": "philox4x32-10 seed 210",
         "step": "one iteration of one ion species (all pcuts)",
         "population_order": "momentum-sorted injection list dealt into 64 strided sub-sequences (balances contiguous rank shards)"}
    if extra:
        c.update(extra)
    return c


def step_outputs(res):
    """name -> array: per ion of one step, what its caller receives from mcs_run_ion and mcs_end_ion."""
    out = {}
    for i, r in res.items():
        t = r["t"]
        arrays = {"n_used": r["n_used"], "n_saved": r["n_saved"], **{nm: getattr(t, nm) for nm in DUMP_TALLIES},
                  **t.scalars, **t.stats}
        out.update({f"ion{i}_{k}": v for k, v in arrays.items()})
    return out


def dump_outputs(path, arrays, limit=DUMP_BYTES):
    """Writes each array as <path>/<name>.npy in float64.  When together they would exceed `limit` bytes, every array of more
    than 1 MB keeps the same fraction of its entries, at flat indices drawn with a fixed seed: two runs of the same shapes
    keep the same entries."""
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in arrays.items()}
    limit -= 1024 * len(arrays)  # .npy headers
    big = sorted(k for k, v in arrays.items() if v.nbytes > 1 << 20)
    small = sum(v.nbytes for k, v in arrays.items() if k not in big)
    total = small + sum(arrays[k].nbytes for k in big)
    if total > limit:
        frac = (limit - small) / (total - small)
        for k in big:
            v = arrays[k].ravel()
            idx = np.random.default_rng(0).choice(v.size, int(v.size * frac), replace=False)
            arrays[k] = v[np.sort(idx)]
    os.makedirs(path, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(path, k + ".npy"), v)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                       "-i", str(gpu_index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            pass

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.p.terminate()
        self.p.wait()
        self.f.flush()
        rows = [r.split(",") for r in open(self.f.name).read().strip().splitlines() if r.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons, pw = [], [], set(), []
        for r in rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); pw.append(float(r[3]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.strip().lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


def cpu_arm(workload, sample_per_pcut, steps, warmup, threads, pcuts="bench", all_species=False, collect=None):
    """The reference's CPU implementation of the path = the C restatement (oracle/), all host threads.
    `collect`: list that receives the ion-1 tallies of every timed step (each step then uses its own seed and injection
    draw, i.e. the steps are independent replicas: bench.py's statistical-parity block)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle_engine
    from mcs_b200 import abi, driver
    lib = oracle_engine.load_oracle_library()
    run, prof = build_run(workload, sample_per_pcut, pcuts)
    run.profile = prof
    e = abi.Engine(lib, driver.make_config(lib, run, threads=threads, na_cr=1000))
    tot_steps, tot_t = 0, 0.0
    for it in range(warmup + steps):
        if collect is not None:  # independent replica: another Philox key and another injection draw
            e.close()
            e = abi.Engine(lib, driver.make_config(lib, run, threads=threads, na_cr=1000, seed=7000 + it))
        t0 = time.perf_counter()
        res = driver.main_loops(run, e, n_iters=1, want_psd=True, want_log=False, shuffle_population=True,
                                only_ions=None if all_species else [1], pop_seed_offset=(1000 * (it + 1) if collect is not None else 0))[0]
        dt = time.perf_counter() - t0
        st = sum(r["tallies"].stats["n_helix_steps"] + r["tallies"].stats["n_retro_steps"] for r in res if r is not None)
        if it >= warmup:
            tot_steps += st
            tot_t += dt
            if collect is not None:
                collect.append(res[0]["tallies"])
    return tot_steps / tot_t, tot_t / max(steps, 1), tot_steps // max(steps, 1)


class _Ranks:
    """rank / world of this process for driver.main_loops (the library does the exchanges itself: device_comm=True)."""
    def __init__(self, rank, world):
        self.rank, self.world = rank, world


def verify_multi_rank(lib, dist, rank, world, local_rank):
    """Driver-visible evidence that the N-rank path computes what one rank computes: a 4000-particle x 4-pcut planar case
    through mcs_run_ion on N ranks (NCCL inside the library, rebalancing split) and, on rank 0, the same global
    population on a second single-rank handle.  Integers must be identical, flux sums agree to summation order."""
    import torch
    from mcs_b200 import abi, driver, problem
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    run = problem.setup_run(problem.planar_test_particle_input(4000, momentum_cutoffs=[0.01, 0.04, 0.06, 0.09]))
    eng = abi.Engine(lib, driver.make_config(lib, run, na_cr=3_000_000, device=local_rank))
    uid = torch.zeros(128, dtype=torch.uint8, device="cuda")
    if rank == 0:
        uid = torch.tensor(list(eng.comm_unique_id()), dtype=torch.uint8, device="cuda")
    dist.broadcast(uid, 0)
    eng.comm_init(rank, world, bytes(uid.cpu().tolist()))
    many = driver.main_loops(run, eng, n_iters=1, comm=_Ranks(rank, world), device_comm=True, want_log=False)[0][0]
    eng.close()
    out = None
    if rank == 0:
        e1 = abi.Engine(lib, driver.make_config(lib, run, na_cr=3_000_000, device=local_rank))
        one = driver.main_loops(run, e1, n_iters=1, want_log=False)[0][0]
        e1.close()
        ta, tb = many["tallies"], one["tallies"]

        def rel(x, y):
            x, y = np.asarray(x, float), np.asarray(y, float)
            sc = np.maximum(np.abs(x), np.abs(y))
            m = sc > 0
            return float((np.abs(x - y)[m] / sc[m]).max()) if m.any() else 0.0

        out = {
            "case": "planar 4000 particles x 4 pcuts, mcs_run_ion on N ranks (NCCL, rebalancing split) vs 1 rank",
            "ranks": world,
            "n_saved_equal": bool(np.array_equal(many["n_saved"], one["n_saved"])),
            "n_used_equal": bool(np.array_equal(many["n_used"], one["n_used"])),
            "n_fate_equal": ta.stats["n_fate"] == tb.stats["n_fate"],
            "n_helix_steps_equal": ta.stats["n_helix_steps"] == tb.stats["n_helix_steps"]
                                   and ta.stats["n_retro_steps"] == tb.stats["n_retro_steps"],
            "num_crossings_equal": bool(np.array_equal(ta.num_crossings, tb.num_crossings)),
            "psd_bitwise_equal": bool(np.array_equal(ta.psd, tb.psd)),
            "fluxes_bitwise_equal": bool(np.array_equal(ta.pxx_flux, tb.pxx_flux) and np.array_equal(ta.pxz_flux, tb.pxz_flux)
                                         and np.array_equal(ta.energy_flux, tb.energy_flux)),
            "max_rel_diff": {"pxx_flux": rel(ta.pxx_flux, tb.pxx_flux), "pxz_flux": rel(ta.pxz_flux, tb.pxz_flux),
                             "energy_flux": rel(ta.energy_flux, tb.energy_flux), "psd": rel(ta.psd, tb.psd),
                             "esc_psd_feb_downstream": rel(ta.esc_psd_feb_downstream, tb.esc_psd_feb_downstream)},
            "n_saved": [int(v) for v in many["n_saved"]],
        }
        d = out["max_rel_diff"]
        out["ok"] = bool(out["n_saved_equal"] and out["n_used_equal"] and out["n_fate_equal"] and out["n_helix_steps_equal"]
                         and out["num_crossings_equal"] and max(d["pxx_flux"], d["pxz_flux"], d["energy_flux"]) < 1e-11
                         and d["psd"] < 1e-10 and d["esc_psd_feb_downstream"] < 1e-10)
    dist.barrier()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="planar", choices=["planar", "relativistic", "nonlinear", "multi"])
    ap.add_argument("--n-per-pcut", type=int, default=1_000_000)
    ap.add_argument("--pcuts", default="bench", choices=["bench", "default"],
                    help="bench: the workload's own ladder; default: the 45 cut-offs of the reference's mc_in.toml:84-130")
    ap.add_argument("--all-species", action="store_true",
                    help="multi workload: one step = all ion species of the iteration (p, He, e-) with the pool hand-over")
    ap.add_argument("--cpu-sample", type=int, default=30000, help="particles per pcut of the CPU sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--stat-parity", type=int, default=0, metavar="R",
                    help="cpu_baseline leg: run the CPU sample as R independent replicas (cpu-sample / R particles per pcut each) and "
                         "report per-spectrum chi-square p-values of the GPU run against them (north_star 'full runs')")
    ap.add_argument("--no-verify", action="store_true", help="skip the N-rank vs 1-rank check that precedes a multi-GPU run")
    ap.add_argument("--generate-in-library", action="store_true",
                    help="SURVEY 8(f2): hand init_pop to the library in run-length form instead of copying host arrays")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the outputs of the last one to DIR/<name>.npy (float64, <= 64 MB)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the CUDA arm (--impl b200)")
    # stdout carries exactly one JSON line: libraries that write to fd 1 (NCCL prints its version there) go to stderr
    sys.stdout.flush()
    out_fd = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        sys.stdout.flush()
        os.write(out_fd, (json.dumps(obj) + "\n").encode())

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    threads = os.cpu_count() or 1
    all_species = a.all_species and a.workload == "multi"

    if a.impl == "reference":
        if rank != 0:
            return 0
        v, s_per_it, st = cpu_arm(a.workload, a.cpu_sample, max(a.steps, 1), min(a.warmup, 1), threads, a.pcuts, all_species)
        run, _ = build_run(a.workload, a.cpu_sample, a.pcuts)
        sample = f"{a.cpu_sample} particles per pcut (of {a.n_per_pcut}), full pcut ladder, {st} steps per iteration"
        emit(({
            "impl": "reference", "metric": METRIC, "value": v, "unit": "steps/s", "n_gpus": a.gpus, "steps": a.steps,
            "warmup": min(a.warmup, 1), "ms_per_step": s_per_it * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(a.workload, run, a.n_per_pcut, {"cpu_sample_per_pcut": a.cpu_sample}),
            "cpu_baseline": {"value": v, "unit": "steps/s", "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": "C restatement of the reference Julia loop (no Julia runtime in this image), OpenMP over particles",
        }))
        return 0

    import torch
    import mcs_b200
    from mcs_b200 import abi, driver, problem

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the transport loop has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def allmax(x):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    lib = mcs_b200.load_cuda_library()
    verify = None
    if world > 1 and not a.no_verify:
        verify = verify_multi_rank(lib, dist, rank, world, local_rank)

    n_global = a.n_per_pcut * world
    run, prof = build_run(a.workload, n_global, a.pcuts)
    run.profile = prof
    cfg = driver.make_config(lib, run, n_pts_cap=n_global + 8, na_cr=1_000_000, device=local_rank)
    eng = abi.Engine(lib, cfg)
    if world > 1:
        uid = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            uid = torch.tensor(list(eng.comm_unique_id()), dtype=torch.uint8, device="cuda")
        dist.broadcast(uid, 0)
        eng.comm_init(rank, world, bytes(uid.cpu().tolist()))

    # host inputs of one step, in pinned memory (the populations main_loops.jl hands to the particle loop)
    ions = [i for i in range(1, run.n_ions + 1) if not (run.species[i - 1].n0 == 0 and run.inp.skip_zero_density_species)]
    if not all_species:
        ions = ions[:1]
    eps = problem.populate_eps_target(run, prof)
    pinned, per_ion, h2d = [], {}, 0
    for i_ion in ions:
        spec = problem.injection_spec(run, prof, i_ion)
        lo, hi = driver.shard_bounds(spec.n, rank, world)
        pop = {}
        if not a.generate_in_library:
            ip = problem.expand_injection(spec, np.random.default_rng(i_ion - 1), shuffle=True)
            for k, v in ip.pop.items():
                t = torch.from_numpy(np.ascontiguousarray(v[lo:hi])).pin_memory()
                pinned.append(t)
                pop[k] = t.numpy()
        per_ion[i_ion] = dict(spec=spec, lo=lo, hi=hi, pop=pop, sp=driver.species_struct(run, i_ion),
                              p_hi=problem.pcut_hi(run.inp.en_pcut_hi, run.species[i_ion - 1].mass))
        h2d += sum(v.nbytes for v in pop.values()) + 11 * (run.n_grid + 2) * 8
        if a.generate_in_library:
            h2d += 6 * 8 * len(spec.bin_ptot) + 8
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")  # > 126 MB L2
    D2H_FIELDS = ("pxx_flux", "pxz_flux", "energy_flux", "psd", "num_crossings", "esc_psd_feb_upstream", "esc_psd_feb_downstream",
                  "esc_energy_eff", "esc_num_eff", "weight_coupled", "spectra_coupled", "energy_transfer_pool")

    def one_step():
        """The call sequence a Julia user makes per iteration: for each ion H2D, the device pcut loop, D2H; the energy pool
        donated by the ions is handed to the next species (main_loops.jl:95-164)."""
        pool = np.zeros(run.n_grid)
        res = {}
        for i_ion in ions:
            d = per_ion[i_ion]
            t0 = eng.timing()
            eng.set_profile(prof, eps, pool.copy())
            if a.generate_in_library:
                eng.begin_ion_generate(1, i_ion, d["sp"], d["spec"], first_global=d["lo"], n_local=d["hi"] - d["lo"], shuffle=True)
            else:
                eng.begin_ion(1, i_ion, d["sp"], d["pop"], first_global=d["lo"])
            n_run, n_used, n_saved = eng.run_ion(run.pcuts, d["p_hi"], run.inp.n_pts_pcut, run.inp.n_pts_pcut_hi)
            t = eng.end_ion(want_psd=True, want_log=False)
            pool = pool + t.energy_transfer_pool
            t1 = eng.timing()
            res[i_ion] = dict(t=t, n_run=n_run, n_used=n_used, n_saved=n_saved,
                              steps=t.stats["n_helix_steps"] + t.stats["n_retro_steps"],
                              loop_ms=t1["ion_loop_ms"] - t0["ion_loop_ms"], kern_ms=t1["transport_ms"] - t0["transport_ms"],
                              d2h=sum(getattr(t, nm).nbytes for nm in D2H_FIELDS) + 8 * 8 + 24 * 8)
        return res

    for _ in range(a.warmup):
        one_step()
    fp64_peak = eng.measure_fp64_peak()
    scatter_peak = eng.measure_scatter_peak()
    atomic_peak = eng.measure_atomic_peak(run.n_grid * (run.num_psd_mom_bins + 2) * (run.num_psd_theta_bins + 2))
    eng.timing(reset=True)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    wall, res = 0.0, {}
    sp_steps = {i: 0.0 for i in ions}
    sp_ms = {i: 0.0 for i in ions}
    try:  # a failing step must not leave the nvidia-smi sampler running
        barrier()
        for _ in range(a.steps):
            flush.fill_(1)  # L2 flush between timed iterations (not timed)
            barrier()
            t0 = time.perf_counter()
            res = one_step()
            torch.cuda.synchronize()
            wall += time.perf_counter() - t0
            for i in ions:
                sp_steps[i] += res[i]["steps"]   # already summed over ranks by the all-reduce of mcs_end_ion
                sp_ms[i] += res[i]["loop_ms"]
        barrier()
    finally:
        clocks = sampler.stop() if sampler else None
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, step_outputs(res))
    tm = eng.timing()
    steps_total = float(sum(sp_steps.values()))      # global, all timed steps
    steps_per_iter = steps_total / a.steps
    d2h = sum(r["d2h"] for r in res.values())
    n_run = max(r["n_run"] for r in res.values())
    dev_s = allmax(tm["ion_loop_ms"]) * 1e-3
    wall_s = allmax(wall)
    kern_s = allmax(tm["transport_ms"]) * 1e-3
    per_rank_kernel_ms = per_rank_steps = per_rank_particles = None
    if dist is not None:
        g = [torch.zeros(1, dtype=torch.float64, device="cuda") for _ in range(world)]
        dist.all_gather(g, torch.tensor([tm["transport_ms"]], dtype=torch.float64, device="cuda"))
        per_rank_kernel_ms = [round(float(x.item()) / a.steps, 1) for x in g]
        dist.all_gather(g, torch.tensor([float(tm["local_steps"])], dtype=torch.float64, device="cuda"))
        per_rank_steps = [float(x.item()) / a.steps for x in g]
        dist.all_gather(g, torch.tensor([float(tm["local_particles"])], dtype=torch.float64, device="cuda"))
        per_rank_particles = [float(x.item()) / a.steps for x in g]
    value = steps_total / dev_s
    e2e = steps_total / wall_s
    # dominant kernel: this rank's steps over this rank's kernel time
    kern_steps_per_s = float(tm["local_steps"]) / (tm["transport_ms"] * 1e-3)
    achieved = kern_steps_per_s * FLOP_PER_STEP / 1e12
    red_gops = float(tm["local_reds"]) / (tm["transport_ms"] * 1e-3) / 1e9
    launches = int(tm["transport_launches"] + tm["other_launches"])
    traffic, traffic_src = measured_traffic(a.workload, a.n_per_pcut) if (a.pcuts == "bench" and not all_species) else (None, None)

    if rank == 0:
        extra = {
            "population": "generated in the library from the run-length injection list" if a.generate_in_library
                          else "host arrays in pinned memory, copied every step",
            "pcuts_run": int(n_run), "steps_per_iteration": int(steps_per_iter), "l2": "flushed between timed iterations",
            "s_per_iteration_device": dev_s / a.steps, "s_per_iteration_e2e": wall_s / a.steps}
        if all_species:
            extra["step"] = "one iteration of ALL ion species (every pcut of each), energy pool handed from ions to electrons"
            extra["species"] = {
                f"ion{i}": {"aa": run.species[i - 1].aa, "n0": run.species[i - 1].n0, "electron": bool(run.species[i - 1].is_electron),
                            "steps_per_iteration": int(sp_steps[i] / a.steps), "ms_per_iteration": sp_ms[i] / a.steps,
                            "steps_per_s": sp_steps[i] / (sp_ms[i] * 1e-3) if sp_ms[i] > 0 else None,
                            "pcuts_run": int(res[i]["n_run"])} for i in ions}
        out = {
            "metric": METRIC, "value": value, "unit": "steps/s", "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": dev_s / a.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": workload_config(a.workload, run, a.n_per_pcut, extra),
            "e2e": {"value": e2e, "unit": "steps/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "ms_per_step": wall_s / a.steps * 1e3},
            "gpu_launches": launches, "per_rank_kernel_ms_per_step": per_rank_kernel_ms,
            "per_rank_steps_per_step": per_rank_steps, "per_rank_particles_per_step": per_rank_particles,
            "clocks": clocks,
            "roofline": {"bound": "fp64", "kernel": "transport_kernel<false>", "achieved": achieved, "peak": fp64_peak,
                         "unit": "TFLOP/s", "frac": achieved / fp64_peak if fp64_peak else None,
                         "traffic": traffic, "traffic_source": traffic_src,
                         "flop_per_step": FLOP_PER_STEP, "kernel_ms_per_launch": kern_s * 1e3 / max(tm["transport_launches"], 1),
                         "kernel_share_of_step": kern_s / dev_s,
                         "peak_source": "measured live: DFMA microbenchmark in libmcs_b200.so (MEASURED_PEAKS.json has no FP64 entry)",
                         "hot_path_ceiling_steps_per_s": scatter_peak,
                         "frac_of_hot_path_ceiling": kern_steps_per_s / scatter_peak if scatter_peak else None,
                         "hot_path_ceiling_source": "measured live: scatter_only_kernel = Philox + kick + phase + move, no control flow",
                         "atomic": {"achieved_gops": red_gops, "peak_gops": atomic_peak,
                                    "frac": red_gops / atomic_peak if atomic_peak else None,
                                    "reds_per_step": float(tm["local_reds"]) / max(float(tm["local_steps"]), 1.0),
                                    "source": "red.global operations into the tallies counted by the kernel (rank 0) over its "
                                              "kernel time; peak = scattered FP64 red microbenchmark over a PSD-sized array, live"}},
        }
        if verify is not None:
            out["verify"] = verify
        if world == 1 and not a.no_cpu_baseline:
            if a.stat_parity >= 4 and not all_species:
                R, n_rep = a.stat_parity, max(a.cpu_sample // a.stat_parity, 500)
                reps = []
                v, s_it, st = cpu_arm(a.workload, n_rep, R, 0, threads, a.pcuts, False, collect=reps)
                sys.path.insert(0, os.path.join(ROOT, "tests"))
                import stat_parity
                cmp_ = stat_parity.compare(stat_parity.observables(res[ions[0]]["t"], run), [stat_parity.observables(t, run) for t in reps],
                                           n_ratio=a.n_per_pcut / n_rep)
                out["cpu_baseline"] = {"value": v, "unit": "steps/s", "cores": threads, "kind": "port",
                                       "sample": f"{R} independent replicas of {n_rep} particles per pcut, full pcut ladder, {st} steps each, {s_it:.1f} s each",
                                       "stat_parity": {"p_min_stated": 1e-3, "replicas": R, "particles_per_pcut_per_replica": n_rep,
                                                       "method": "tests/stat_parity.py: per-bin z of the GPU run against the replica mean, chi-square p",
                                                       "spectra": cmp_}}
            else:
                v, s_it, st = cpu_arm(a.workload, a.cpu_sample, 1, 0, threads, a.pcuts, all_species)
                out["cpu_baseline"] = {"value": v, "unit": "steps/s", "cores": threads, "kind": "port",
                                       "sample": f"{a.cpu_sample} particles per pcut, full pcut ladder, {st} steps, {s_it:.1f} s"}
            # the reference loop itself is serial (the threading directive at main_loops.jl:227 is a comment): one thread too
            n1 = max(a.cpu_sample // 10, 200)
            v1, s1, st1 = cpu_arm(a.workload, n1, 1, 0, 1, a.pcuts, all_species)
            out["cpu_baseline"]["single_thread"] = {"value": v1, "cores": 1,
                                                    "sample": f"{n1} particles per pcut, {st1} steps, {s1:.1f} s"}
        emit(out)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
