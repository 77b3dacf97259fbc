"""Device primitives of the transport kernel against exact references, one primitive at a time.

tests/device_units.cu includes csrc/mcs_device.cuh and is built with the library's flags (sm_100a, -O3, FMA contraction on),
so each kernel here runs the code the library inlines.  References are exact: integer / Fraction arithmetic for the exact
tally accumulators (acc_add + fold_accumulators_kernel), mpmath at 60 digits for the fast loop's math (az_sincos,
rsqrt_nr) and for the device build of the shared sincos_bf / asin_bf (tests/test_device_math.py holds their host build to
libm), numpy index arithmetic and bit patterns for the split of new_pcut (enqueue_compaction, clone_kernel, and the
rebalancing split — split_plan, pack_saved_kernel, clone_gathered_kernel — of up to 64 ranks emulated on one device).
Run with -s to see the worst error measured for each primitive.
"""
import ctypes as C
import math
import os
import subprocess
from fractions import Fraction

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
ACC_D, ACC_ELO = 10, -210  # csrc/mcs_device.cuh: words per cell, weight of the lowest bit
AZ_N = 256
SIN_UPPER_LIMIT = np.nextafter(1.0, 0.0)
P_D = C.POINTER(C.c_double)
P_I64 = C.POINTER(C.c_int64)
P_U32 = C.POINTER(C.c_uint32)
P_U8 = C.POINTER(C.c_uint8)


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("du") / "libdevice_units.so")
    r = subprocess.run([NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xcompiler", "-fPIC",
                        "-shared", "-cudart", "static", "-ccbin", "/usr/bin/g++", "-o", out,
                        os.path.join(HERE, "device_units.cu")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    lib = C.CDLL(out)
    lib.du_acc_add.argtypes = [P_I64, P_D, C.c_long, C.c_long, P_I64, C.POINTER(C.c_uint64)]
    lib.du_fold.argtypes = [P_I64, C.c_long, P_D]
    lib.du_az_table.argtypes = [P_D]
    lib.du_az_sincos.argtypes = [P_U32, P_U32, C.c_long, P_D, P_D]
    lib.du_roots.argtypes = [P_D, C.c_long, P_D, P_D, P_D]
    lib.du_sincos_bf.argtypes = [P_D, C.c_long, P_D, P_D]
    lib.du_asin_bf.argtypes = [P_D, C.c_long, C.c_int, P_D]
    lib.du_compact.argtypes = [P_U8, C.c_long, P_I64, P_I64]
    lib.du_split_local.argtypes = [P_D, P_I64, P_U8, P_U8, C.c_long, C.c_long, C.c_long, P_D, P_I64, P_U8, P_I64]
    lib.du_split_ranks.argtypes = [C.c_int, P_I64, P_U8, P_D, P_I64, P_U8, C.c_longlong, C.c_longlong, C.c_long, P_D, P_I64,
                                   P_U8, P_I64, P_I64]
    lib.du_split_plan.argtypes = [P_I64, C.c_int, C.c_int, C.c_longlong, C.c_longlong, P_I64, P_I64]
    return lib


def _p(a, t=P_D):
    return a.ctypes.data_as(t)


def _ok(rc):
    assert rc == 0, f"CUDA error {rc}"


def test_harness_compiles(harness):
    """Builds on any machine: a change of the header that breaks the harness fails here without a GPU."""
    assert harness.du_fold is not None


def test_azimuth_table_is_the_bin_centres(harness):
    """The library's azimuth table (az_table: host libm at the double nearest each bin centre -pi + 2 pi (k + 1/2) / 256)
    against the exact sine and cosine of the centres.  The centre is rounded to double before libm sees it, which costs up
    to 2.4 ulp of 1 next to +-pi (measured 2.36); az_sincos inherits that error."""
    import mpmath
    mpmath.mp.dps = 60
    tab = np.zeros(2 * AZ_N)
    _ok(harness.du_az_table(_p(tab)))
    worst = 0.0
    for k in range(AZ_N):
        a = -mpmath.pi + 2 * mpmath.pi * (k + mpmath.mpf(0.5)) / AZ_N
        worst = max(worst, float(abs(tab[2 * k] - mpmath.sin(a))), float(abs(tab[2 * k + 1] - mpmath.cos(a))))
    print(f"\nazimuth table: worst {worst * 2**52:.3f} ulp of 1 against the exact bin centres")
    assert worst <= 2.4 * 2.0**-52


# ----------------------------------------------------------------------------------------------------------------------
# Exact accumulators.  acc_add keeps a contribution's multiples of 2^-210 (truncated toward zero below), refuses |v| >= 2^98,
# inf and NaN (CNT_ERR), and fold_accumulators_kernel turns the integer the words hold into the correctly rounded double.

def _units(v):
    """What acc_add adds for v, in units of 2^-210 (0 for a refused value)."""
    if not math.isfinite(v) or abs(v) >= 2.0**98:
        return 0
    n, d = float(v).as_integer_ratio()
    q = (abs(n) << -ACC_ELO) // d
    return q if n >= 0 else -q


def _refused(v):
    return not math.isfinite(v) or abs(v) >= 2.0**98


def _word_value(w):
    return sum(int(x) << (32 * k) for k, x in enumerate(w))


def _rounded(units):
    """The correctly rounded double of units * 2^-210 (Fraction -> float rounds once, to nearest even)."""
    return float(Fraction(units, 1 << -ACC_ELO))


def _acc_add(lib, cells):
    """acc_add every value of cells[i] into cell i; returns (words [n_cells, ACC_D], CNT_ERR)."""
    idx = np.concatenate([np.full(len(c), i, dtype=np.int64) for i, c in enumerate(cells)])
    v = np.concatenate([np.asarray(c, dtype=np.float64) for c in cells])
    words = np.zeros((len(cells), ACC_D), dtype=np.int64)
    n_err = C.c_uint64(0)
    _ok(lib.du_acc_add(_p(idx, P_I64), _p(v), len(v), len(cells), _p(words, P_I64), C.byref(n_err)))
    return words, n_err.value


def _fold(lib, words):
    words = np.ascontiguousarray(words, dtype=np.int64)
    out = np.full(len(words), np.nan)
    _ok(lib.du_fold(_p(words, P_I64), len(words), _p(out)))
    return out


def _assert_bits(got, want, what):
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    bad = np.flatnonzero(got.view(np.int64) != want.view(np.int64))
    assert bad.size == 0, (f"{what}: {bad.size} of {got.size} cells differ from the correctly rounded sum, e.g. "
                           + ", ".join(f"cell {i}: {got[i].hex()} != {want[i].hex()}" for i in bad[:4]))


def _check_cells(lib, cells, what):
    """acc_add + fold on the device against the exact sums: words, folded bits and CNT_ERR."""
    words, n_err = _acc_add(lib, cells)
    sums = [sum(_units(v) for v in c) for c in cells]
    for i, s in enumerate(sums):
        assert _word_value(words[i]) == s, f"{what}: words of cell {i} do not hold the exact sum"
    _assert_bits(_fold(lib, words), [_rounded(s) for s in sums], what)
    assert n_err == sum(_refused(v) for c in cells for v in c), what
    return words


@pytest.mark.gpu
def test_fold_rounds_once(harness):
    """{1, 2^-53, 2^-100}: the exact sum lies just above the midpoint 1 + 2^-53, so its double is 1 + 2^-52; a fold that
    rounds word by word from the top loses the 2^-100 before it meets the tie and returns 1."""
    base = [1.0, 2.0**-53, 2.0**-100]
    cells = [base, base[::-1], [-x for x in base], [1.0, 2.0**-53], [1.0, 2.0**-53, -(2.0**-100)], [3.0, 2.0**-52, 2.0**-200]]
    _check_cells(harness, cells, "double-rounding cases")
    assert _fold(harness, _acc_add(harness, [base])[0])[0] == 1.0 + 2.0**-52


@pytest.mark.gpu
def test_random_cells_of_a_pcut_ladder(harness):
    """Cells of 20 weights spread like a deep pcut ladder (1e-6 at injection, / 3 per pcut down to 3^-40), mixed signs in
    a quarter of them: every folded cell is the correctly rounded exact sum."""
    rng = np.random.default_rng(11)
    cells = []
    for i in range(20_000):
        w = rng.uniform(0, 1, 20) * 1e-6 / 3.0 ** rng.integers(0, 41, 20)
        if i % 4 == 3:
            w *= rng.choice([-1.0, 1.0], 20)
        cells.append(w.tolist())
    _check_cells(harness, cells, "pcut ladder cells")


@pytest.mark.gpu
def test_every_alignment_against_the_word_boundaries(harness):
    """A 53-bit significand at every offset r = 0..31 from a word boundary, in every word the window allows: the pieces
    that straddle two and three words, alone, with signs, and all offsets summed in one cell."""
    rng = np.random.default_rng(12)
    cells = []
    for k0 in range(ACC_D - 2):
        for r in range(32):
            e = 32 * k0 + r + ACC_ELO  # exponent of the significand's lowest bit
            m = [int(x) | (1 << 52) for x in rng.integers(0, 1 << 52, 3)]
            vals = [math.ldexp(x, e) for x in m]
            cells += [[vals[0]], [-vals[0]], [vals[0], vals[1], -vals[2]], [vals[0], -vals[1], vals[2], 2.0 ** (e + 52)]]
        cells.append([math.ldexp(int(rng.integers(1 << 52, 1 << 53)), 32 * k0 + r + ACC_ELO) * float(rng.choice([-1, 1]))
                      for r in range(32)])
    _check_cells(harness, cells, "alignments")


@pytest.mark.gpu
def test_negative_sums_and_exact_cancellation(harness):
    """Negative contributions; sums that cancel to exactly zero fold to +0.0, whatever order the adds came in."""
    rng = np.random.default_rng(13)
    cells = [[1.0, -1.0], [-1.0, 1.0], [0.75, 0.25, -1.0], [-(2.0**97), 2.0**97], [2.0**-150, -(2.0**-150)]]
    for _ in range(500):
        w = (rng.uniform(0, 1, 16) * 2.0 ** rng.integers(-150, 90, 16)).tolist()
        both = w + [-x for x in w]
        rng.shuffle(both)
        cells.append(both)
    n_zero = len(cells)
    for _ in range(500):
        cells.append((-rng.uniform(0, 1, 12) * 2.0 ** rng.integers(-150, 90, 12)).tolist() + [float(rng.uniform(0, 1e-6))])
    _check_cells(harness, cells, "signed cells")
    out = _fold(harness, _acc_add(harness, cells[:n_zero])[0])
    assert np.all(out.view(np.int64) == 0), "a sum that cancels exactly must fold to +0.0"


@pytest.mark.gpu
def test_subnormals_and_the_bottom_of_the_window(harness):
    """Below 2^-210 the window keeps nothing; between 2^-263 and 2^-157 a contribution keeps its multiples of 2^-210
    (truncated toward zero, sign kept).  Subnormals and anything below 2^-210 add nothing and are no error."""
    rng = np.random.default_rng(14)
    cells = [[5e-324], [-5e-324], [2.0**-1022], [np.nextafter(2.0**-1022, 0.0)], [2.0**-210], [-(2.0**-210)],
             [np.nextafter(2.0**-210, 0.0)], [2.0**-211 * 3], [2.0**-157], [np.nextafter(2.0**-157, 0.0)], [2.0**-263],
             [1.0, 2.0**-211], [1.0, -(2.0**-211)]]
    for p in list(range(-160, -154)) + list(range(-213, -207)) + list(range(-266, -260)):
        for _ in range(40):
            cells.append((rng.uniform(1, 2, 8) * 2.0**p * rng.choice([-1.0, 1.0], 8)).tolist())
    cells.append((rng.uniform(0, 1, 64) * 2.0**-1022).tolist())
    _check_cells(harness, cells, "bottom of the window")


@pytest.mark.gpu
def test_top_of_the_window(harness):
    """nextafter(2^98, 0) is the largest contribution taken exactly; 2^98, +-inf and NaN are refused and each is counted in
    CNT_ERR; +-0 adds nothing."""
    top = np.nextafter(2.0**98, 0.0)
    cells = [[top], [-top], [top, top, top, top], [2.0**98], [-(2.0**98)], [math.inf], [-math.inf], [math.nan],
             [0.0], [-0.0], [top, 2.0**98, 1.0, math.nan], [-0.0, 1.0]]
    words = _check_cells(harness, cells, "top of the window")
    assert _fold(harness, words)[0] == top
    _, n_err = _acc_add(harness, [[2.0**98], [math.inf], [-math.inf], [math.nan]])
    assert n_err == 4


@pytest.mark.gpu
def test_carries_from_a_million_adds(harness):
    """10^6 contributions into one cell, so the words run far past 2^32 and the fold has to carry: mixed magnitudes and
    signs in one cell, contributions just below the top of the window in another."""
    rng = np.random.default_rng(15)
    n = 1_000_000
    mixed = rng.uniform(0, 1, n) * 2.0 ** rng.integers(-200, 90, n) * rng.choice([-1.0, 1.0], n, p=[0.3, 0.7])
    big = rng.uniform(0.5, 1.0, n) * 2.0**98
    words = _check_cells(harness, [mixed.tolist(), big.tolist()], "a million adds")
    assert np.abs(words).max() > 2**40


@pytest.mark.gpu
def test_fold_is_a_function_of_the_value(harness):
    """Word vectors built by hand: words near +-2^62, unnormalised carries, and different vectors holding the same integer
    — among them the element-wise sum of two ranks' words, which is what the integer all-reduce hands the fold."""
    rng = np.random.default_rng(16)
    vecs = [rng.integers(-(2**62), 2**62, ACC_D) for _ in range(2000)]
    vecs += [rng.integers(0, 2**62, ACC_D) * np.array([1] * (ACC_D - 1) + [0]) for _ in range(200)]
    vecs += [np.array([2**32] + [-1] + [0] * (ACC_D - 2)), np.array([0] * (ACC_D - 2) + [2**32, -1]),
             np.array([-(2**32), 1] + [0] * (ACC_D - 2)), np.array([0] * (ACC_D - 1) + [-1]),
             np.array([2**32 - 1] * (ACC_D - 1) + [-1]), np.array([2**62] * ACC_D), np.array([-(2**62)] * ACC_D)]
    words = np.array(vecs, dtype=np.int64)
    want = np.array([_rounded(_word_value(w)) for w in words])
    _assert_bits(_fold(harness, words), want, "hand-built words")
    # the same integers, carried between neighbouring words in random amounts
    moved = words.copy()
    for w in moved:
        for k in rng.integers(0, ACC_D - 1, 6):
            t = int(rng.integers(-(2**26), 2**26))
            w[k] += t << 32
            w[k + 1] -= t
    assert all(_word_value(a) == _word_value(b) for a, b in zip(words, moved))
    _assert_bits(_fold(harness, moved), want, "carried words")
    # two ranks' accumulators of the same cells, summed word by word
    cells = [(rng.uniform(0, 1, 40) * 1e-6 / 3.0 ** rng.integers(0, 41, 40) * rng.choice([-1.0, 1.0], 40)).tolist()
             for _ in range(2000)]
    w_all, _ = _acc_add(harness, cells)
    w_a, _ = _acc_add(harness, [c[::2] for c in cells])
    w_b, _ = _acc_add(harness, [c[1::2] for c in cells])
    _assert_bits(_fold(harness, w_a + w_b), _fold(harness, w_all), "two ranks")
    _assert_bits(_fold(harness, w_all), [_rounded(sum(_units(v) for v in c)) for c in cells], "two ranks")


# ----------------------------------------------------------------------------------------------------------------------
# The fast loop's math, and the device build of the shared sincos_bf / asin_bf

def _mp_ref(fn, xs):
    """fn(x) at 60 digits as a double-double (hi, lo): an error against it is exact to ~2^-100 of the value."""
    import mpmath
    mpmath.mp.dps = 60
    hi, lo = np.zeros(len(xs)), np.zeros(len(xs))
    for i, x in enumerate(xs):
        v = fn(mpmath.mpf(float(x)))
        hi[i] = float(v)
        lo[i] = float(v - hi[i])
    return hi, lo


def _ulps(got, ref, unit=None):
    """|got - ref| in ulps of the reference (or in units of `unit`)."""
    hi, lo = ref
    return np.abs((got - hi) - lo) / (np.spacing(np.abs(hi)) if unit is None else unit)


@pytest.mark.gpu
def test_az_sincos_against_the_exact_azimuth(harness):
    """az_sincos(hi, lo) against sin and cos of the exact azimuth 2 pi w / 2^53 - pi, w = (hi:lo) >> 11: every table entry
    k at the offsets f = 0, 1, 2^44, 2^45 - 1 and 4096 random ones (the 11 bits below w set at random).  Bound 2.5 ulp of 1
    (measured 2.45 on B200): up to 2.36 of it is the table's own error (test_azimuth_table_is_the_bin_centres)."""
    import mpmath
    mpmath.mp.dps = 60
    rng = np.random.default_rng(21)
    f = np.concatenate([[0, 1, 2**44, 2**45 - 1], rng.integers(0, 2**45, 4096)]).astype(np.uint64)
    k = np.arange(AZ_N, dtype=np.uint64)
    w = (k[:, None] << np.uint64(45)) | f[None, :]
    u = (w << np.uint64(11)) | rng.integers(0, 2048, w.shape).astype(np.uint64)
    hi, lo = (u >> np.uint64(32)).astype(np.uint32).ravel(), (u & np.uint64(0xFFFFFFFF)).astype(np.uint32).ravel()
    s, c = np.zeros(hi.size), np.zeros(hi.size)
    _ok(harness.du_az_sincos(_p(hi, P_U32), _p(lo, P_U32), hi.size, _p(s), _p(c)))
    # exact reference by angle addition in 200-bit fixed point: azimuth = A_k + t_f, A_k the bin centre
    S = 200
    fix = lambda v: int(mpmath.nint(v * mpmath.mpf(2) ** S))  # noqa: E731
    A = [-mpmath.pi + 2 * mpmath.pi * (kk + mpmath.mpf(0.5)) / AZ_N for kk in range(AZ_N)]
    sA, cA = [fix(mpmath.sin(a)) for a in A], [fix(mpmath.cos(a)) for a in A]
    t = [2 * mpmath.pi * int(ff) / mpmath.mpf(2) ** 53 - mpmath.pi / AZ_N for ff in f]
    st, ct = [fix(mpmath.sin(x)) for x in t], [fix(mpmath.cos(x)) for x in t]
    nf = len(f)
    err_s = [float((int(s[i] * 2.0**S) << S) - (sA[i // nf] * ct[i % nf] + cA[i // nf] * st[i % nf])) for i in range(s.size)]
    err_c = [float((int(c[i] * 2.0**S) << S) - (cA[i // nf] * ct[i % nf] - sA[i // nf] * st[i % nf])) for i in range(c.size)]
    worst = max(np.abs(err_s).max(), np.abs(err_c).max()) * 2.0 ** (52 - 2 * S)
    s2c2 = np.abs(s.astype(np.longdouble) ** 2 + c.astype(np.longdouble) ** 2 - 1).max()
    print(f"\naz_sincos: worst {worst:.3f} ulp of 1 against the exact azimuth, |s^2 + c^2 - 1| <= {float(s2c2):.3g}")
    assert worst <= 2.5
    assert s2c2 <= 4e-16


def _fast_loop_operands(rng, n):
    """Operands the fast loop takes square roots of: sin^2 of the scattering angle 1 - cos_d^2 (u1 down to 2^-53),
    sin^2 of the pitch 1 - cos^2 next to both poles, and sn2 - a^2 next to the clamp of |sin dphi| at prevfloat(1)."""
    u1 = rng.uniform(0, 1, n) * 2.0 ** -rng.integers(0, 54, n)
    omc = 2.0 ** rng.uniform(-30, 1, n)
    cd = 1 - u1 * omc
    pole = (1 - rng.uniform(0, 1, n) * 2.0 ** -rng.integers(1, 53, n)) * rng.choice([-1.0, 1.0], n)
    sn2 = rng.uniform(0, 1, n)
    a = np.sqrt(sn2) * (1 - rng.uniform(0, 1, n) * 2.0 ** -rng.integers(1, 53, n))
    x = np.concatenate([1 - cd * cd, 1 - pole * pole, sn2 - a * a])
    return x[x > 0]


@pytest.mark.gpu
def test_rsqrt_nr(harness):
    """rsqrt_nr(x) against 1/sqrt(x) and the fast loop's square root x * rsqrt_nr(x) against sqrt(x), over [2^-970, 2^64]
    and the loop's own operands; NaN for +-0, negative values and NaN (the loop parks a lane on it)."""
    rng = np.random.default_rng(22)
    x = np.concatenate([2.0 ** rng.uniform(-970, 64, 100_000), _fast_loop_operands(rng, 40_000), [2.0**-970, 1.0, 2.0**64]])
    r, q, sq = np.zeros_like(x), np.zeros_like(x), np.zeros_like(x)
    _ok(harness.du_roots(_p(x), x.size, _p(r), _p(q), _p(sq)))
    import mpmath
    e_r = _ulps(r, _mp_ref(lambda v: 1 / mpmath.sqrt(v), x))
    e_q = _ulps(q, _mp_ref(mpmath.sqrt, x))
    print(f"\nrsqrt_nr: worst {e_r.max():.3f} ulp; x * rsqrt_nr(x): worst {e_q.max():.3f} ulp of sqrt(x)")
    assert e_r.max() <= 1.0
    assert e_q.max() <= 2.0
    assert np.array_equal(sq, np.sqrt(x))  # sqrt_nr: the correctly rounded sqrt() on its range
    special = np.array([0.0, -0.0, -1.0, -(2.0**-1000), -math.inf, math.nan, -math.nan])
    r, q, sq = np.zeros_like(special), np.zeros_like(special), np.zeros_like(special)
    _ok(harness.du_roots(_p(special), special.size, _p(r), _p(q), _p(sq)))
    assert np.all(np.isnan(r)) and np.all(np.isnan(q)), r
    # below the stated range, never an operand of the loop (its operands are >= ~1e-32), measured on B200: subnormals give
    # NaN (the seed flushes them to zero), normal x in [2^-1022, 2^-970) the same <= 1 ulp as above
    tiny = np.array([5e-324, 2.0**-1050, np.nextafter(2.0**-1022, 0.0), 2.0**-1022, 2.0**-1000, 2.0**-980,
                     np.nextafter(2.0**-970, 0.0)])
    r, q, sq = np.zeros_like(tiny), np.zeros_like(tiny), np.zeros_like(tiny)
    _ok(harness.du_roots(_p(tiny), tiny.size, _p(r), _p(q), _p(sq)))
    e_t = _ulps(r, _mp_ref(lambda v: 1 / mpmath.sqrt(v), tiny))
    print("rsqrt_nr below 2^-970:", ", ".join(f"{t.hex()} -> {v!r} ({e:.2f} ulp)" for t, v, e in zip(tiny, r, e_t)))
    assert np.all(np.isnan(r[tiny < 2.0**-1022])) and e_t[tiny >= 2.0**-1022].max() <= 1.0


def _sincos_args(rng):
    x = np.concatenate([rng.uniform(-5 * np.pi, 5 * np.pi, 100_000), rng.uniform(-1e-3, 1e-3, 20_000),
                        np.arange(-10, 11) * (np.pi / 2), np.arange(-10, 11) * (np.pi / 2) + 1e-9, [0.0, 1e-300]])
    return np.concatenate([x, -x])


@pytest.mark.gpu
def test_sincos_bf_device_build(harness):
    """sincos_bf as the library builds it (FMA contraction) against mpmath: <= 2 ulp, absolute 2e-16 next to the zeros
    (2-term Cody-Waite reduction), sin odd and cos even bit for bit away from 0.  (The device build returns sin(-0) = +0.)"""
    import mpmath
    x = _sincos_args(np.random.default_rng(23))
    s, c = np.zeros_like(x), np.zeros_like(x)
    _ok(harness.du_sincos_bf(_p(x), x.size, _p(s), _p(c)))
    worst = []
    for got, fn in ((s, mpmath.sin), (c, mpmath.cos)):
        ref = _mp_ref(fn, x)
        big = np.abs(ref[0]) > 1e-12
        e = _ulps(got[big], (ref[0][big], ref[1][big]))
        a = _ulps(got[~big], (ref[0][~big], ref[1][~big]), unit=1.0)
        worst.append((e.max(), a.max()))
        assert e.max() <= 2.0 and a.max() < 2e-16
    print(f"\nsincos_bf (device): sin worst {worst[0][0]:.3f} ulp / {worst[0][1]:.2g} abs, cos worst {worst[1][0]:.3f} ulp / "
          f"{worst[1][1]:.2g} abs")
    h = x.size // 2
    nz = x[:h] != 0
    assert np.array_equal(s[h:][nz].view(np.int64), (-s[:h][nz]).view(np.int64))
    assert np.array_equal(c[h:].view(np.int64), c[:h].view(np.int64)) and np.all(s[x == 0] == 0)
    assert abs(s * s + c * c - 1).max() < 5e-16


@pytest.mark.parametrize("nr", [0, 1])
@pytest.mark.gpu
def test_asin_bf_device_build(harness, nr):
    """asin_bf<false> and asin_bf<true> (sqrt_nr / div_nr inside, |x| < 1 strictly) as the library builds them, against
    mpmath: odd bit for bit, asin(+-0) = +-0, and <= 2.2 ulp.  tests/test_device_math.py holds the algorithm to 2 ulp of libm;
    against the exact value it is 2.12 ulp just above |x| = 0.5 (pi/2 - 2 asin(sqrt((1 - |x|) / 2)) in plain FP64), the
    same in the host and the device build (measured on B200)."""
    import mpmath
    rng = np.random.default_rng(24)
    x = np.concatenate([rng.uniform(-1, 1, 100_000), rng.uniform(-1e-6, 1e-6, 20_000), 1 - 10.0 ** rng.uniform(-16, -1, 20_000),
                        [0.0, 0.5, SIN_UPPER_LIMIT, np.nextafter(0.5, 1), 1e-300] + ([] if nr else [1.0])])
    x = np.concatenate([x, -x])
    y = np.zeros_like(x)
    _ok(harness.du_asin_bf(_p(x), x.size, nr, _p(y)))
    nz = x != 0
    e = _ulps(y[nz], _mp_ref(mpmath.asin, x[nz]))
    print(f"\nasin_bf<{bool(nr)}> (device): worst {e.max():.3f} ulp")
    assert e.max() <= 2.2
    h = x.size // 2
    assert np.array_equal(y[h:].view(np.int64), (-y[:h]).view(np.int64))
    assert np.array_equal(y[~nz].view(np.int64), x[~nz].view(np.int64))


# ----------------------------------------------------------------------------------------------------------------------
# The split of new_pcut (cuts.jl:69-91): child o of a split is the saved parent flatnonzero(l_save)[o // i_mult] with every
# field copied and its weight w / i_mult (one IEEE division).  compaction_blocks tiles the particles by 1024 and the scan
# carries its running total from one tile of 1024 block counts (2^20 particles) to the next, so the sizes below straddle
# both boundaries.  Populations cross in the harness's field-major layout: f64 [8, n] (weight first), i64 [2, n], u8 [2, n].

SPLIT_PLAN_OK, SPLIT_PLAN_BAD_RANKS, SPLIT_PLAN_NONE_SAVED, SPLIT_PLAN_OVER_CAPACITY, SPLIT_PLAN_OVER_RANGE = range(5)
COMPACTION_SIZES = [1, 31, 32, 33, 1023, 1024, 1025, 2**20 - 1, 2**20, 2**20 + 1, 2**20 + 1024, 10_000_019, 3 * 2**24 + 5]


def _save_patterns(n, rng):
    """name -> l_save of n particles."""
    def one_at(*i):
        return np.bincount(np.concatenate([np.atleast_1d(np.asarray(x, np.int64)) for x in i]), minlength=n).astype(np.uint8)
    edges = np.arange(1024, n, 1024)  # every 2^20 boundary is one of these
    return {"all": np.ones(n, np.uint8), "first": one_at(0), "last": one_at(n - 1),
            "block_edges": one_at(0, edges - 1, edges),
            "every_other": (np.arange(n) % 2 == 0).astype(np.uint8),
            "sparse": (rng.random(n) < 1e-4).astype(np.uint8), "half": (rng.random(n) < 0.5).astype(np.uint8)}


@pytest.mark.gpu
@pytest.mark.parametrize("n", COMPACTION_SIZES)
def test_compaction(harness, n):
    """enqueue_compaction against np.flatnonzero, for every pattern: the saved indices in order, the count, and nothing
    written past it.  3 * 2^24 + 5 particles make 49 scan tiles, the last of them holding a single block count."""
    rng = np.random.default_rng(31 + n % 1000)
    for name, l_save in _save_patterns(n, rng).items():
        idx, total = np.zeros(n, np.int64), np.zeros(1, np.int64)
        _ok(harness.du_compact(_p(l_save, P_U8), n, _p(idx, P_I64), _p(total, P_I64)))
        want = np.flatnonzero(l_save)
        assert total[0] == want.size, f"n = {n}, {name}: total {total[0]} != {want.size}"
        bad = np.flatnonzero(idx[:want.size] != want)
        assert bad.size == 0, f"n = {n}, {name}: {bad.size} saved indices wrong, first at output {bad[0]}"
        assert not idx[want.size:].any(), f"n = {n}, {name}: written past the count"


def _random_pop(rng, n):
    """A population whose 12 fields are random bit patterns: any finite double (subnormals, -0 included), any int64, any
    byte."""
    bits = rng.integers(0, 2**64, (8, n), dtype=np.uint64)
    top = np.uint64(0x7FF) << np.uint64(52)
    bits[(bits & top) == top] ^= np.uint64(1) << np.uint64(62)  # exponent all ones (inf / NaN) -> finite
    return (bits.view(np.float64), rng.integers(-(2**63), 2**63 - 1, (2, n), dtype=np.int64, endpoint=True),
            rng.integers(0, 256, (2, n), dtype=np.uint8, endpoint=False))


def _ref_split(f64, i64, u8, l_save, i_mult):
    """The split in cuts.jl:69-91 order: children of the k-th saved particle at rows [k i_mult, (k + 1) i_mult)."""
    par = np.repeat(np.flatnonzero(l_save), i_mult)
    f = f64[:, par]
    f[0] = f[0] / np.float64(i_mult)
    return f, i64[:, par], u8[:, par]


def _assert_pop_equal(got, want, what):
    for a, b, nm in zip(got, want, ("f64", "i64", "u8")):
        a = a.view(np.int64) if a.dtype == np.float64 else a
        b = b.view(np.int64) if b.dtype == np.float64 else b
        assert a.shape == b.shape, f"{what}: {nm} shape {a.shape} != {b.shape}"
        bad = np.argwhere(a != b)
        assert bad.size == 0, f"{what}: {len(bad)} {nm} values differ, first (field, child) = {tuple(bad[0])}"


def _split_local(lib, pop, l_save, i_mult):
    f64, i64, u8 = (np.ascontiguousarray(a) for a in pop)
    n, cap = len(l_save), int(l_save.sum()) * i_mult
    out = (np.zeros((8, cap)), np.zeros((2, cap), np.int64), np.zeros((2, cap), np.uint8))
    total = np.zeros(1, np.int64)
    _ok(lib.du_split_local(_p(f64), _p(i64, P_I64), _p(u8, P_U8), _p(l_save, P_U8), n, i_mult, cap, _p(out[0]),
                           _p(out[1], P_I64), _p(out[2], P_U8), _p(total, P_I64)))
    assert total[0] == l_save.sum()
    return out


@pytest.mark.gpu
def test_split_local(harness):
    """Compaction + clone_kernel (the single-rank split) bit for bit against the reference split, for i_mult 1, 3, 1000
    and target // ns, on populations of random bit patterns, two of them past one scan tile (2^20 particles)."""
    rng = np.random.default_rng(32)
    cases = [(5000, 0.3, 1), (5000, 0.3, 3), (5000, 0.3, 1000), (4099, 0.05, "target"),
             (2**20 + 4097, 0.5, "target"), (3_000_017, 0.01, "target")]
    for n, density, i_mult in cases:
        pop, l_save = _random_pop(rng, n), (rng.random(n) < density).astype(np.uint8)
        if i_mult == "target":
            i_mult = max(4_000_000 // int(l_save.sum()), 1)
        _assert_pop_equal(_split_local(harness, pop, l_save, i_mult), _ref_split(*pop, l_save, i_mult),
                          f"n = {n}, i_mult = {i_mult}")


def _rank_case(rng, sizes, density, target, n_pts_max=None):
    """Ranks of the given population sizes; density[q] = fraction of rank q's particles saved."""
    l_save = [(rng.random(s) < d).astype(np.uint8) for s, d in zip(sizes, density)]
    return dict(sizes=np.asarray(sizes, np.int64), l_save=l_save, target=target, n_pts_max=n_pts_max or 2**31 - 1)


def _rank_cases():
    rng = np.random.default_rng(33)
    r8 = rng.integers(0, 5000, 8)
    r64 = rng.integers(0, 3000, 64)
    d64 = np.where(np.arange(64) % 7 == 3, 0.0, rng.uniform(0.05, 0.9, 64))
    one_of_64 = np.where(np.arange(64) == 41, 0.3, 0.0)
    r8_one, r64_one = np.where(np.arange(8) == 5, 3001, r8), np.where(np.arange(64) == 41, 2999, r64)
    return {
        "1 rank": _rank_case(rng, [777], [0.4], 10_000),
        "2 ranks, first empty": _rank_case(rng, [1000, 3001], [0.0, 0.3], 50_000),
        "2 ranks, target below S": _rank_case(rng, [2047, 1500], [0.7, 0.6], 1000),
        "3 ranks, middle empty": _rank_case(rng, [513, 0, 2049], [0.5, 0.5, 0.5], 100_000),
        "3 ranks, middle saves none": _rank_case(rng, [1111, 2222, 333], [0.3, 0.0, 0.9], 7),
        "3 ranks past one scan tile": _rank_case(rng, [2**20 + 5, 17, 2**21 - 3], [0.5, 1.0, 0.25], 2_000_000),
        "8 ranks, last empty": _rank_case(rng, r8, [0.4] * 7 + [0.0], 100_003),
        "8 ranks, all but one empty": _rank_case(rng, r8_one, [0.0] * 5 + [0.5] + [0.0] * 2, 12_345),
        "64 ranks": _rank_case(rng, r64, d64, 1_000_003),
        "64 ranks, all but one empty": _rank_case(rng, r64_one, one_of_64, 99_999),
        "64 ranks, target below S": _rank_case(rng, r64, rng.uniform(0, 1, 64), 10),
    }


def _split_ranks(lib, case, pop, l_save):
    sizes, nr = case["sizes"], len(case["sizes"])
    f64, i64, u8 = (np.ascontiguousarray(a) for a in pop)
    S = int(l_save.sum())
    C_ = S * max(case["target"] // S, 1)
    out = (np.zeros((8, C_)), np.zeros((2, C_), np.int64), np.zeros((2, C_), np.uint8))
    n_out, i_mult = np.zeros(nr, np.int64), np.zeros(1, np.int64)
    _ok(lib.du_split_ranks(nr, _p(sizes, P_I64), _p(l_save, P_U8), _p(f64), _p(i64, P_I64), _p(u8, P_U8), case["target"],
                           case["n_pts_max"], C_, _p(out[0]), _p(out[1], P_I64), _p(out[2], P_U8), _p(n_out, P_I64),
                           _p(i_mult, P_I64)))
    return out, n_out, int(i_mult[0])


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(_rank_cases()))
def test_split_emulated_ranks(harness, name):
    """The rebalancing split of N ranks emulated on one device (split_plan, pack_saved_kernel into the exchange buffer as
    the all-gather leaves it, clone_gathered_kernel per rank): rank r's slice is rows [C r / N, C (r + 1) / N) of the
    reference split of the concatenated population, bit for bit, and the slices together are what one rank computes
    (du_split_local on the concatenated population)."""
    case = _rank_cases()[name]
    rng = np.random.default_rng(34)
    sizes, nr = case["sizes"], len(case["sizes"])
    l_save = np.concatenate(case["l_save"])
    pop = _random_pop(rng, int(sizes.sum()))
    ns = np.array([int(x.sum()) for x in case["l_save"]])
    S = int(ns.sum())
    i_mult_ref = max(case["target"] // S, 1)
    C_ = S * i_mult_ref
    out, n_out, i_mult = _split_ranks(harness, case, pop, l_save)
    assert i_mult == i_mult_ref
    ref = _ref_split(*pop, l_save, i_mult_ref)
    for r in range(nr):
        c0, c1 = C_ * r // nr, C_ * (r + 1) // nr
        assert n_out[r] == c1 - c0, f"{name}: rank {r} got {n_out[r]} children, not {c1 - c0}"
        _assert_pop_equal(tuple(a[:, c0:c1] for a in out), tuple(a[:, c0:c1] for a in ref), f"{name}, rank {r}")
    _assert_pop_equal(out, _split_local(harness, pop, l_save, i_mult_ref), f"{name}: N ranks against one")
    print(f"\n{name}: ns {ns.min()}..{ns.max()} over {nr} ranks, S = {S}, i_mult = {i_mult}, C = {C_}, C % N = {C_ % nr}, "
          f"max ns % 16 = {ns.max() % 16}")


def test_emulated_rank_cases_cover_the_edges():
    """The cases above hold every edge of the plan: ranks saving nothing first, last, in the middle and all but one; the
    largest ns not a multiple of 16 (padded stride); a target below S (i_mult clamped to 1); C not divisible by N."""
    seen = set()
    for case in _rank_cases().values():
        ns = np.array([int(x.sum()) for x in case["l_save"]])
        S, nr = int(ns.sum()), len(ns)
        C_ = S * max(case["target"] // S, 1)
        seen |= {k for k, v in {"first empty": ns[0] == 0 and nr > 1, "last empty": ns[-1] == 0 and nr > 1,
                                "middle empty": nr > 2 and (ns[1:-1] == 0).any(), "all but one": nr > 2 and (ns > 0).sum() == 1,
                                "padded stride": ns.max() % 16 != 0, "clamped": case["target"] < S,
                                "ragged slices": C_ % nr != 0}.items() if v}
        for n in (1, 2, 3, 8, 64):
            if nr == n:
                seen.add(n)
    assert seen == {"first empty", "last empty", "middle empty", "all but one", "padded stride", "clamped", "ragged slices",
                    1, 2, 3, 8, 64}, seen


def _plan(lib, ns_all, rank, target, n_pts_max):
    ns_all = np.ascontiguousarray(ns_all, dtype=np.int64)
    out, start = np.full(6, -1, np.int64), np.zeros(65, np.int64)
    rc = lib.du_split_plan(_p(ns_all, P_I64), len(ns_all), rank, target, n_pts_max, _p(out, P_I64), _p(start, P_I64))
    return rc, dict(zip(("S", "i_mult", "C", "c0", "c1", "stride"), (int(v) for v in out))), start[:len(ns_all) + 1]


def test_split_plan_formula(harness):
    """split_plan (host code, no GPU) over a sweep of (S, N, target): i_mult = max(target // S, 1), C = S i_mult, rank r's
    slice [C r // N, C (r + 1) // N), stride = largest ns rounded up to 16, the gather prefix the running sum of ns_all."""
    rng = np.random.default_rng(35)
    n_cases = 0
    for nr in (1, 2, 3, 5, 8, 17, 63, 64):
        for _ in range(40):
            ns_all = rng.integers(0, int(rng.choice([2, 100, 10**5, 10**7])), nr)
            ns_all[rng.random(nr) < 0.3] = 0
            S = int(ns_all.sum())
            if S == 0:
                ns_all[rng.integers(0, nr)] = 1
                S = 1
            target = int(rng.choice([0, 1, S - 1, S, S + 1, 2 * S - 1, int(rng.integers(0, 10**9))]))
            i_mult = max(target // S, 1)
            C_ = S * i_mult
            if C_ > 2**32:
                continue
            for r in range(nr):
                rc, p, start = _plan(harness, ns_all, r, target, 2**62)
                assert rc == SPLIT_PLAN_OK
                assert p == {"S": S, "i_mult": i_mult, "C": C_, "c0": C_ * r // nr, "c1": C_ * (r + 1) // nr,
                             "stride": -(-int(ns_all.max()) // 16) * 16}, (ns_all, r, target)
                assert np.array_equal(start, np.concatenate([[0], np.cumsum(ns_all)]))
            n_cases += 1
    assert n_cases > 250


def test_split_plan_refusals(harness):
    """The refusals at their exact edges: the largest slice at n_pts_max is taken and at n_pts_max + 1 refused; C = 2^32 is
    taken and C = 2^32 + 1 refused (saved counts with no memory behind them); S = 0 and a bad rank layout are refused.
    A refused plan still reports S (the library keeps it as the ion's global saved count)."""
    rng = np.random.default_rng(36)
    for _ in range(300):
        nr = int(rng.choice([1, 2, 3, 7, 64]))
        ns_all = rng.integers(0, 1000, nr)
        ns_all[0] += 1
        S = int(ns_all.sum())
        target = int(rng.integers(0, 10**6))
        C_ = S * max(target // S, 1)
        largest = max(C_ * (r + 1) // nr - C_ * r // nr for r in range(nr))
        for r in {0, nr - 1}:
            assert _plan(harness, ns_all, r, target, largest)[0] == SPLIT_PLAN_OK
            rc, p, _ = _plan(harness, ns_all, r, target, largest - 1)
            assert rc == SPLIT_PLAN_OVER_CAPACITY and p["S"] == S
    big = 2**62
    for ns_all, target, want in (([2**31, 2**31], 0, SPLIT_PLAN_OK), ([2**31, 2**31 + 1], 0, SPLIT_PLAN_OVER_RANGE),
                                 ([2**32], 2**32, SPLIT_PLAN_OK), ([2**32 + 1], 0, SPLIT_PLAN_OVER_RANGE),
                                 ([2**16], 2**32, SPLIT_PLAN_OK), ([2**16], 2**32 + 2**16, SPLIT_PLAN_OVER_RANGE),
                                 ([1, 2**16 - 1], 2**32 + 2**16 - 1, SPLIT_PLAN_OK),
                                 ([3] * 63 + [2**32 + 1 - 189], 0, SPLIT_PLAN_OVER_RANGE),
                                 ([3] * 63 + [2**32 - 189], 5, SPLIT_PLAN_OK)):
        rc, p, _ = _plan(harness, ns_all, len(ns_all) - 1, target, big)
        assert rc == want, (ns_all[-3:], target, rc)
        if want == SPLIT_PLAN_OK:
            assert p["C"] == 2**32 and p["c1"] == 2**32
    # the capacity check comes first: at C = 2^32 + 1 on one rank with n_pts_max = C - 1 it is the capacity that refuses
    assert _plan(harness, [2**32 + 1], 0, 0, 2**32)[0] == SPLIT_PLAN_OVER_CAPACITY
    for nr in (1, 2, 64):
        rc, p, start = _plan(harness, [0] * nr, nr - 1, 10**6, big)
        assert rc == SPLIT_PLAN_NONE_SAVED and p["S"] == 0 and not start.any()
    assert _plan(harness, [1, 1], 2, 10, big)[0] == SPLIT_PLAN_BAD_RANKS
    assert _plan(harness, [1, 1], -1, 10, big)[0] == SPLIT_PLAN_BAD_RANKS
    assert _plan(harness, [1] * 65, 0, 10, big)[0] == SPLIT_PLAN_BAD_RANKS
