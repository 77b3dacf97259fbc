"""The north-star size end to end: 10 000 019 particles per pcut on one device, against exact references.

Every other test builds at most 1e6 particles, below one tile of the split's scan (2^20 particles), and holds the transport
and the generator to the oracle at no more than 30 000.  Here, on the planar config at 1e7 per pcut:
- the generator (shuffle on, n % 64 != 0) equals the host mirror problem.expand_injection bit for bit;
- every pcut's counts agree with its fates and l_save, and mcs_split equals the numpy split of the saved records in
  cuts.jl:69-91 order bit for bit, i_mult = max(n_pts_pcut // ns, 1) (past pcut 1 the library's compaction runs ~10 scan tiles);
- 256-particle windows at 0, 2^20, 2^21 and 2^23 (minus 128) and at the end of each pcut's population run through the
  oracle at the same global indices give identical fates, pass, retro and draw counts, and saved states within the
  tolerances of test_parity_gpu.test_per_particle_parity_at_scale: the static schedule, the Philox counter field
  first_global + ip past 2^23 and the state of particles millions of slots deep are exact;
- the same population started at first_global = 2^32 - n runs pcut 1 with its last window equal to the oracle's at the
  top of the counter range;
- the ion ends with no error and no negative square root, and every particle's weight ends in exactly one fate.
Run with -s to see the wall time.
"""
import os
import time

import numpy as np
import pytest

from helpers import LADDER, compare_saved, make_engine, start_ion
from mcs_b200 import abi, driver, problem

pytestmark = pytest.mark.gpu

N = 10_000_019
SEED = 210
WINDOW = 256
TOL_END_STATE, TOL_PHI = 1e-10, 1e-4  # as test_per_particle_parity_at_scale


def _bits(a):
    return a.view(np.int64) if a.dtype == np.float64 else a


def _windows(n):
    starts = sorted({s for s in (0, 2**20 - 128, 2**21 - 128, 2**23 - 128, max(n - WINDOW, 0)) if s < n})
    return [(s, min(s + WINDOW, n)) for s in starts]


def _slice(pop, s, e):
    return {k: v[s:e] for k, v in pop.items()}


def _check_window(olib, run, pop_in, fates, saved, s, e, k, pcut, prev, first_global):
    """Particles [s, e) of the device's pcut-k input through the oracle at global indices first_global + [s, e)."""
    eo = make_engine(olib, run, seed=SEED, n_pts_cap=WINDOW, na_cr=1000, threads=max(os.cpu_count() or 1, 1))
    start_ion(eo, run, pop=_slice(pop_in, s, e), first_global=first_global + s)
    eo.run_pcut(k, pcut, prev)
    fo = eo.get_fates(e - s)
    for key in ("fate", "helix_count", "retro_steps", "n_draws"):
        d = np.flatnonzero(fo[key] != fates[key][s:e])
        assert d.size == 0, (f"pcut {k}, particle {first_global + s + d[0]}: {key} {fates[key][s + d[0]]} != oracle "
                             f"{fo[key][d[0]]}")
    compare_saved(run, run.species[0], eo.get_population(1, e - s), _slice(saved, s, e), TOL_END_STATE, TOL_PHI)
    eo.close()


def test_north_star_size(olib, clib):
    t0 = time.perf_counter()
    inp = problem.planar_test_particle_input(N, momentum_cutoffs=LADDER[:3])
    run = problem.setup_run(inp)
    spec = problem.injection_spec(run, run.profile, 1)
    n = spec.n
    assert n % 64 != 0 and n > 2**23 + WINDOW  # 10 000 016 injected (whole particles per momentum bin)
    e = make_engine(clib, run, seed=SEED, na_cr=1000)
    e.set_profile(run.profile, problem.populate_eps_target(run, run.profile), np.zeros(run.n_grid))

    # 1. the generator against the host mirror
    assert e.begin_ion_generate(1, 1, driver.species_struct(run, 1), spec, shuffle=True) == n
    gen = e.get_population(0, n)
    ref = problem.expand_injection(spec, problem.PhiloxInjectionRng(SEED, 1, 1), shuffle=True).pop
    for f, v in ref.items():
        assert np.array_equal(_bits(gen[f]), _bits(v)), f"generated {f} differs from the host mirror"
    assert np.all(gen["xn_per"] == inp.fine_scattering_Ng) and np.all(gen["prp_x_cm"] == run.x_grid_stop)
    assert not gen["downstream"].any() and not gen["inj"].any() and np.all(gen["tcut"] == 1) and not gen["acctime_sec"].any()
    del ref
    t_gen = time.perf_counter()

    # 2., 3. every pcut: counts, the split, the oracle windows
    pop_in, w_in, w_out = gen, float(gen["weight"].sum()), 0.0
    for k, pcut in enumerate(run.pcuts, start=1):
        m = e.population_size()
        prev = run.pcuts[k - 2] if k > 1 else 0.0
        ns, steps = e.run_pcut(k, pcut, prev)
        fates, saved = e.get_fates(m), e.get_population(1, m)
        assert ns == int(saved["l_save"].sum()) == int((fates["fate"] == abi.FATE_SAVED).sum()), f"pcut {k}"
        assert steps == int(fates["helix_count"].sum() + fates["retro_steps"].sum()), f"pcut {k}"
        for s, t in _windows(m):
            _check_window(olib, run, pop_in, fates, saved, s, t, k, pcut, prev, 0)
        w_out += float(pop_in["weight"][fates["fate"] != abi.FATE_SAVED].sum())
        pop_in = fates = None
        if ns == 0:
            break
        n_new, n_glob, i_mult = e.split(inp.n_pts_pcut)
        assert i_mult == max(inp.n_pts_pcut // ns, 1) and n_new == n_glob == ns * i_mult
        par = np.repeat(np.flatnonzero(saved["l_save"]), i_mult)
        pop_in = e.get_population(0, n_new)
        for f in abi.POP_F64 + abi.POP_I64 + abi.POP_U8:
            want = saved[f][par] / np.float64(i_mult) if f == "weight" else saved[f][par]
            bad = np.flatnonzero(_bits(pop_in[f]) != _bits(want))
            assert bad.size == 0, f"split after pcut {k} (ns = {ns}, i_mult = {i_mult}): {f} of child {bad[0]} differs"
        print(f"\npcut {k}: {m} particles, {ns} saved, {steps} steps; split into {n_new} (i_mult {i_mult})")
        del saved, par
    t_pcuts = time.perf_counter()

    # 5. end of the ion
    w_last = float(pop_in["weight"].sum()) if ns > 0 else 0.0
    t = e.end_ion()
    assert t.stats["n_errors"] == 0 and t.stats["n_neg_sqrt"] == 0
    assert w_out + w_last == pytest.approx(w_in, rel=1e-10)  # every weight ends in exactly one fate
    e.close()
    pop_in = None

    # 4. the top of the counter range: the same population at global indices [2^32 - n, 2^32), pcut 1
    top = 2**32 - n
    e2 = make_engine(clib, run, seed=SEED, na_cr=1000)
    e2.set_profile(run.profile, problem.populate_eps_target(run, run.profile), np.zeros(run.n_grid))
    e2.begin_ion(1, 1, driver.species_struct(run, 1), gen, first_global=top)
    e2.run_pcut(1, run.pcuts[0], 0.0)
    fates, saved = e2.get_fates(n), e2.get_population(1, n)
    _check_window(olib, run, gen, fates, saved, n - WINDOW, n, 1, run.pcuts[0], 0.0, top)
    assert e2.end_ion().stats["n_errors"] == 0
    e2.close()
    t_end = time.perf_counter()
    print(f"north-star size, {n} particles per pcut: {t_end - t0:.1f} s wall (generator check {t_gen - t0:.1f} s, "
          f"pcuts {t_pcuts - t_gen:.1f} s, top of the counter range {t_end - t_pcuts:.1f} s)")
