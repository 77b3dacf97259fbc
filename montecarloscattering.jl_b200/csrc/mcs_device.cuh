// mcs_device.cuh — device side of the B200 transport loop (sm_100a).
//
// One persistent kernel advances a whole pcut's population (reference src/particle_loop.jl:154-499 +
// src/particle_finish.jl:46-107).  Design, driven by the ncu evidence in profiles/:
//
//  * every lane owns one particle at a time and runs helix-loop passes; idle lanes are refilled from a
//    per-warp interleaved sequence (deterministic) or a global atomic queue (dynamic);
//  * the per-pass HOT path (scatter, move, zone test) is kept compact; everything rare (zone change boost,
//    energy transfer, retro_time, reflection, PRP logic) is out of line so the loop fits the instruction cache;
//  * work that only a few lanes need in a given pass — zone-boundary flux/PSD tallies (all_flux.jl) and the
//    escape tallies (particle_finish.jl) — is NOT done in place: the lane appends a 64-byte event to a
//    per-warp queue in shared memory and the warp processes events 32 at a time, fully converged;
//  * the n_grid-sized flux tallies and the scalars are accumulated per warp in shared memory with plain
//    adds in a fixed order (no FP64 atomics: on sm_100a shared FP64 atomicAdd is a CAS loop), then reduced
//    over warps and blocks in a fixed order -> run-to-run deterministic;
//  * the 22 MB phase-space histogram lives in L2/HBM and takes red.global.add.f64.
//
// FP64 scalar work with data-dependent control flow: no dense contraction, so no tensor cores / TMA.
#pragma once
#include <cstdint>
#include <cstring>
#include <cuda_runtime.h>

#include "../../include/mcs.h"
#include "mcs_math.cuh"

#define MCS_UNLIKELY(x) __builtin_expect(!!(x), 0)
#define MCS_LIKELY(x) __builtin_expect(!!(x), 1)

#ifndef MCS_BLOCK
#define MCS_BLOCK 256
#endif
#ifndef MCS_MIN_BLOCKS
#define MCS_MIN_BLOCKS 2
#endif
#ifndef MCS_PARK_T
#define MCS_PARK_T 24     // lanes that must be waiting (parked or refillable) before the warp leaves the fast loop (capped at 3/4 of the
                          // lanes in use).  A visit to the general section is expensive — cold code, the lane record through local
                          // memory — so waiting pays: 16 -> 24 is +5 % on the gamma0 = 10 ladder, +4 % on p+He+e-, +0.3 % planar
#endif
#ifndef MCS_PSP_DEBT
#define MCS_PSP_DEBT 256  // lane-iterations of waiting after which the pending boosts of a warp are served (fast loop)
#endif
#ifndef MCS_WAIT_DEBT
#define MCS_WAIT_DEBT 4096  // total idle lane-iterations after which the warp leaves the fast loop to serve its waiting lanes
#endif
#ifndef MCS_PSP_NUM
#define MCS_PSP_NUM 2
#endif
#ifndef MCS_FAST_MAX
#define MCS_FAST_MAX 256  // safety bound on consecutive fast passes
#endif

// The event drain and the boost of the fast loop are folded into it: as ABI calls they forced the loop's state through
// local memory around every call site (+6.7 % steps/s inlined, spill traffic 130 B -> 8 B; profiles/r02_*).
// MCS_CALL_COLD restores the out-of-line form (tuning aid).
#ifdef MCS_CALL_COLD
#define MCS_COLD __noinline__
#else
#define MCS_COLD __forceinline__
#endif

namespace mcs {

constexpr double PI = 3.141592653589793;
constexpr double TWO_PI = 6.283185307179586;
constexpr double TWO_PI_LO = 2.4492935982947064e-16;
constexpr double HALF_PI = PI / 2;
constexpr double SIN_UPPER_LIMIT = 0.99999999999999989;  // prevfloat(1.0), scattering.jl:3
constexpr double SPIKE_AWAY = 1000.0;                    // all_flux.jl:4, particle_finish.jl:5
constexpr int E1 = MCS_PSD_MAX + 1;
#ifndef MCS_QCAP
#define MCS_QCAP 64
#endif
constexpr int QCAP = MCS_QCAP;  // per-warp event queue: < 32 left after a drain + up to 32 new events per push point; below 64
                                // the queue is drained early when a push would not fit (push_events)
constexpr unsigned FULL = 0xffffffffu;

enum : uint32_t {
    F_RAD_LOSSES = 1u, F_RETRO = 2u, F_TCUTS = 4u, F_DONT_DSA = 8u, F_DONT_SCATTER = 16u, F_CUSTOM_EPSB = 32u,
    F_KEEP_NEW_PITCH = 64u, F_DYNAMIC_QUEUE = 128u, F_NO_FAST_LOOP = 256u,
};

// event flags
enum : uint32_t {
    EV_VALID = 1u, EV_FINISH = 2u, EV_INJ = 4u, EV_UP = 8u, EV_FEB_UP = 16u, EV_SUMP = 32u,
    EV_REASON_SHIFT = 8, EV_XSPEC_SHIFT = 16,
};

// The particle record (main_loops.jl:212-226), one field per line in storage order: X(element type, PopPtrs member,
// McsPopulation member).  The wider types come first, so in a block of pop_view's layout every field stays aligned.
#define MCS_POP_FIELDS(X)              \
    X(double, weight, weight)          \
    X(double, ptot, ptot_pf)           \
    X(double, pb, pb_pf)               \
    X(double, x, x_cm)                 \
    X(double, xn_per, xn_per)          \
    X(double, prp_x, prp_x_cm)         \
    X(double, acctime, acctime_sec)    \
    X(double, phi, phi_rad)            \
    X(long long, grid, grid)           \
    X(long long, tcut, tcut)           \
    X(uint8_t, down, downstream)       \
    X(uint8_t, inj, inj)

struct PopPtrs {  // SoA particle record: one array per field
#define X(T, name, pub) T* name;
    MCS_POP_FIELDS(X)
#undef X
};

#define X(T, name, pub) +sizeof(T)
constexpr size_t POP_REC_BYTES = 0 MCS_POP_FIELDS(X);  // bytes of one record
#undef X
#define X(T, name, pub) \
    static_assert(sizeof *McsPopulation{}.pub == sizeof(T), "McsPopulation::" #pub " and PopPtrs::" #name " differ in size");
MCS_POP_FIELDS(X)
#undef X

// n records rounded up to a multiple of 16: every f64 and i64 field of a block then starts a multiple of 128 bytes after it
__host__ __device__ constexpr long long pop_cap(long long n) { return (n + 15) / 16 * 16; }

// A population block: each field in turn holds `cap` records, in list order (POP_REC_BYTES * cap bytes).  The view
// starts at record `first`.  The three populations of a handle and each rank's block of the split's exchange buffer
// have this layout.
__host__ __device__ inline PopPtrs pop_view(unsigned char* base, long long cap, long long first) {
    PopPtrs p;
#define X(T, name, pub) p.name = reinterpret_cast<T*>(base) + first; base += (size_t)cap * sizeof(T);
    MCS_POP_FIELDS(X)
#undef X
    return p;
}

enum { SC_ESC_FLUX = 0, SC_PX_ESC_FEB, SC_EN_ESC_FEB, SC_SUMP, SC_SUMKE, SC_PX_ESC_UP, SC_EN_ESC_UP, SC_N = 8 };
enum {
    CNT_HELIX = 0, CNT_RETRO, CNT_W_PPERP, CNT_W_PSDMOM, CNT_NEGSQRT, CNT_RETRO_CAP, CNT_ERR, CNT_FATE0,  // ..FATE5 = 12
    CNT_LOG = 13, CNT_LOG_OVER = 14, CNT_SAVED = 15, CNT_QUEUE = 16, CNT_FAST_LANE = 17, CNT_FAST_ITER = 18, CNT_SLOW_SEC = 19,
    CNT_SLOW_LANE = 20,
    CNT_RED = 21,  // red.global issued into the tallies (FP64 cells + crossing counts): the kernel's atomic work
    CNT_PARK0 = 24, CNT_N = 40  // CNT_PARK0..+15: why lanes left the fast loop (MCS_SCHED_STATS)
};

struct TallyPtrs {
    double* psd;            // [(M+2)(T+2) n_grid]
    double* esc_up;         // [E1*E1]
    double* esc_dn;         // [E1*E1]
    double* esc_en_eff;     // [E1]
    double* esc_num_eff;    // [E1]
    double* w_coupled;      // [NA_C]
    double* s_coupled;      // [E1*NA_C]
    double* pool;           // [n_grid]
    double* spec_sf;        // [E1*MAX_XSPEC]
    double* spec_pf;
    double* therm_sf;       // [(T+2)(M+2) n_grid] or null: thermal crossings binned in the shock frame (SURVEY 8 f1)
    double* therm_pf;       // ... in the local plasma frame
    double* dndp_cr;        // [(M+2) n_grid]
    unsigned long long* counters;  // [CNT_N]
    long long* tg;          // thermal-crossing log
    double *tpx, *tpt, *tw;
    long long na_cr;
    double *pxx, *pxz, *efl, *scal;  // flux arrays [n_grid] and scalars [SC_N] inside the packed tally buffer
    long long* acc;              // exact fixed-point accumulators, ACC_D digits per cell of the packed tally buffer, or null
    const double* tally_base;    // first cell of the packed FP64 tally buffer (cell index = pointer - tally_base)
    unsigned long long* ncross;  // [n_grid] thermal crossings per zone (integer adds: any order gives the same bits)
    double* block_partials; // [gridDim.x][3*n_grid + SC_N]: pxx | pxz | efl | scalars
};

struct DevParams {
    // constants / shock scalars
    double mp, c, qcgs, E_rel_pt, rad_loss_fac, gam0, u0, u2, bmag2, pe_crit, gam_e_crit, eta_mfp;
    double psd_mom_min, psd_cos_fine, delta_cos, psd_theta_min, bpd_mom, bpd_th;
    double energy_transfer_frac, feb_up, feb_dn, x_grid_stop, B_CMBz, xn_fine, xn_coarse, age_max;
    // per-xn_per scattering constants, [0] fine [1] coarse: 1-cos_max (scattering.jl:46-60), 1/xn_per, 2pi/xn_per
    double omc[2], inv_xn[2], dphi[2];
    double cdphi[2], sdphi[2];   // cos / sin of dphi (the fast loop advances the gyro-phase as a rotation)
    const double2* az_tab;       // [AZ_N] {sin, cos} of -pi + 2 pi (k + 1/2) / AZ_N
    double x_spec[MCS_MAX_XSPEC];
    int M, T, n_grid, i_grid_feb, i_shock, n_xspec, n_tcuts, helix_cap;
    int oblique;  // some zone has sin(theta_B) != 0 (the reference refuses those profiles; the move keeps the term)
    long long retro_cap;
    uint32_t flags;
    // species
    double aa, zz, n0, pmax_cutoff, ewf, m, mc, inj_frac;
    // current pcut
    double pcut, pcut_prev;
    uint32_t key0, key1, ctr2, ctr3;
    uint32_t rk[20];  // Philox round keys key + r * Weyl constant: constant-bank operands of the round's XOR
    long long first_global, n_use;
    // grid arrays (n_grid+2) and per-zone tables
    const double *xg, *ux, *uz, *ut, *gsf, *gef, *bt, *sinth, *costh, *tcuts;
    const double *rxt, *rzt, *crt;  // per zone: ux/ut, uz/ut, ux*uz/ut^2 (the direction factors of transform_p_PSP)
    const double *eps_target, *recv_pool;  // [n_grid]
    PopPtrs cur, saved;
    uint8_t* l_save;
    int *fate, *helix;
    long long *retro, *draws;
    TallyPtrs t;
    // debug: replay stream + trajectory trace
    const double* replay_u;
    const long long* replay_off;
    long long replay_n;
    const int* trace_slot;  // [n_use] or null
    McsTraceRec* trace_recs;
    int* trace_cnt;
    int trace_max;
};

// Shared memory of one block: [zone table | warp 0 region | warp 1 region | ...].
//  zone table (fast loop): per grid node i = 0..ng+1 three 16-byte pairs {ux, gsf}, {gef, cos th}, {xg[i], xg[i+1]} and the gyro
//  denominator 1/(zz*btot[i]); a pass reads its zone's constants from here instead of holding them in registers.
//  warp region: flux partials pxx | pxz | efl (ng each) | scalars (SC_N), then the event queue (QCAP x 72 B, SoA).
//  azimuth table (fast loop): 256 x {sin, cos} of the bin centres of the scattering azimuth (see az_sincos).
constexpr int AZ_N = 256;
__host__ __device__ inline size_t zone_tab_bytes(int ng) { return ((((size_t)(ng + 2) * 56) + 15) & ~(size_t)15) + (size_t)AZ_N * 16; }
__host__ __device__ inline size_t warp_smem_bytes(int ng) {
    return (size_t)(3 * ng + SC_N) * 8 + (size_t)QCAP * (6 * 8 + 6 * 4);
}
__host__ __device__ inline size_t block_smem_bytes(int ng, int warps) { return zone_tab_bytes(ng) + (size_t)warps * warp_smem_bytes(ng); }

// per-warp shared-memory view
struct WarpMem {
    double* part;  // [3*ng + SC_N]: pxx | pxz | efl | scalars
    double *q_pb, *q_pperp, *q_gam, *q_cphi, *q_sphi, *q_ptot;  // the gyro-phase travels as (cos, sin)
    int *q_inew, *q_iold, *q_iz, *q_ip;  // q_ip: particle index (its weight is read when the queue is drained)
    uint32_t* q_flags;
};

// The view is rebuilt from the dynamic shared-memory symbol inside every function that needs it, so that the
// accesses stay LDS/STS (a struct of pointers handed to an out-of-line function decays to generic LD/ST).
__device__ __forceinline__ WarpMem warp_mem(int warp, int ng) {
    extern __shared__ __align__(16) unsigned char mcs_smem[];
    WarpMem w;
    unsigned char* p = mcs_smem + zone_tab_bytes(ng) + (size_t)warp * warp_smem_bytes(ng);
    w.part = reinterpret_cast<double*>(p);
    double* q = w.part + 3 * ng + SC_N;
    w.q_pb = q; w.q_pperp = q + QCAP; w.q_gam = q + 2 * QCAP; w.q_cphi = q + 3 * QCAP; w.q_sphi = q + 4 * QCAP;
    w.q_ptot = q + 5 * QCAP;
    int* qi = reinterpret_cast<int*>(q + 6 * QCAP);
    w.q_inew = qi; w.q_iold = qi + QCAP; w.q_iz = qi + 2 * QCAP; w.q_ip = qi + 3 * QCAP;
    w.q_flags = reinterpret_cast<uint32_t*>(qi + 4 * QCAP);  // (+ one spare int column keeps the region a multiple of 8 bytes)
    return w;
}
struct ZoneTab { const double2 *a, *b, *c; const double* gd; const double2* az; };  // {ux, gsf} | {gef, cos th} | {xg[i], xg[i+1]} | 1/(zz*btot) | azimuth
__device__ __forceinline__ ZoneTab zone_tab(int ng) {
    extern __shared__ __align__(16) unsigned char mcs_smem[];
    ZoneTab z;
    z.a = reinterpret_cast<const double2*>(mcs_smem);
    z.b = z.a + (ng + 2); z.c = z.b + (ng + 2);
    z.gd = reinterpret_cast<const double*>(z.c + (ng + 2));
    z.az = reinterpret_cast<const double2*>(mcs_smem + zone_tab_bytes(ng) - (size_t)AZ_N * 16);
    return z;
}

// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void red_add_f64(double* p, double v) {
    asm volatile("red.global.add.f64 [%0], %1;" ::"l"(__cvta_generic_to_global(p)), "d"(v) : "memory");
}
__device__ __forceinline__ void red_add_u64(unsigned long long* p, unsigned long long v) {
    asm volatile("red.global.add.u64 [%0], %1;" ::"l"(__cvta_generic_to_global(p)), "l"(v) : "memory");
}
__device__ __forceinline__ void count(const DevParams& P, int which, unsigned long long v = 1ull) {
    red_add_u64(&P.t.counters[which], v);
}

// ---------------------------------------------------------------------------------------------
// Exact accumulation of the large histograms (McsConfig.det_tallies).  A cell is ACC_D signed 64-bit words, word k holding
// the multiples of 2^(ACC_ELO + 32 k): a contribution m * 2^e (m its 53-bit significand) is cut at the word boundaries into
// at most three pieces of < 2^32 and each piece is ADDED to its word with an integer atomic.  Integer adds commute and the
// words have 31 bits of headroom (2^31 contributions per cell before a carry could be lost), so the words — and the double
// they are folded into at the end of the ion, the correctly rounded value of the integer they hold — do not depend on the
// order of the adds: bitwise identical run to run, for any schedule and any number of GPUs (the per-rank words are summed
// with an integer all-reduce).  The window is fixed:
// values in [2^-157, 2^98) keep all 53 bits, smaller ones lose their low bits below 2^-210, anything else is counted as an
// error.  (Weights here are ~1e-6 at injection and shrink by up to ~1e-20 in a deep pcut ladder; 1/v >= 3e-11.)
constexpr int ACC_D = 10;
constexpr int ACC_ELO = -210;
__device__ __forceinline__ int acc_add(const DevParams& P, size_t cell, double v);
__device__ __noinline__ int acc_add_ool(const DevParams& P, size_t cell, double v);
// one tally update: exact accumulator when configured, else an FP64 red into the cell itself
// OOL: call the one out-of-line copy of the accumulator add / bin evaluation.  Everything outside the fast loop does (the
// general section, the shared copy of the drain): inlined, each copy of the drain was 5000 instructions (80 KB), and the
// instruction caches are what the many-short-pcut ladders wait for (no_instruction 32 % of the stall samples at gamma0 = 10).
// The drain folded into the fast loop keeps them inline (calls there cost the planar config ~1 %).
template <bool OOL = true>
__device__ __forceinline__ int tally_add(const DevParams& P, double* cell, double v) {
    if (P.t.acc != nullptr) return OOL ? acc_add_ool(P, (size_t)(cell - P.t.tally_base), v) : acc_add(P, (size_t)(cell - P.t.tally_base), v);
    red_add_f64(cell, v);
    return 1;
}
__device__ __forceinline__ int acc_add(const DevParams& P, size_t cell, double v) {
    const long long bits = __double_as_longlong(v);
    const int ex = (int)((bits >> 52) & 0x7ff);
    unsigned long long m = (unsigned long long)bits & 0x000fffffffffffffull;
    if (ex == 0 && m == 0) return 0;
    if (ex == 0x7ff) { count(P, CNT_ERR); return 0; }  // NaN / inf: the reference would have thrown long before
    int e = (ex ? ex : 1) - 1075;
    if (ex) m |= 0x0010000000000000ull;
    int s = e - ACC_ELO;
    if (s < 0) {  // below the window: keep what reaches it
        if (s <= -53) return 0;
        m >>= -s;
        s = 0;
    }
    const int k0 = s >> 5, r = s & 31;
    if (k0 + 2 >= ACC_D) { count(P, CNT_ERR); return 0; }  // beyond 2^98
    const unsigned long long lo64 = m << r, hi64 = r ? (m >> (64 - r)) : 0ull;
    unsigned long long d0 = lo64 & 0xffffffffull, d1 = lo64 >> 32, d2 = hi64;
    if (bits < 0) { d0 = 0ull - d0; d1 = 0ull - d1; d2 = 0ull - d2; }
    unsigned long long* c = reinterpret_cast<unsigned long long*>(P.t.acc) + cell * ACC_D + k0;
    int n = 0;
    if (d0) { red_add_u64(c, d0); n++; }
    if (d1) { red_add_u64(c + 1, d1); n++; }
    if (d2) { red_add_u64(c + 2, d2); n++; }
    return n;
}
__device__ __noinline__ int acc_add_ool(const DevParams& P, size_t cell, double v) { return acc_add(P, cell, v); }

// RNG: Philox4x32-10, counter = (block, i_prt, i_pcut | i_ion<<16, i_iter), key = seed. Replaces the
// per-particle Random.Xoshiro(iseed_mod) of particle_loop.jl:34-41.  Integer pipe only.
struct Rng {
    uint32_t n, s2, s3, c1;
    const double* ru;
    long long rn;
    bool exhausted;
};

__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                              uint32_t k1, uint32_t& o0, uint32_t& o1, uint32_t& o2, uint32_t& o3) {
#pragma unroll
    for (int r = 0; r < 10; r++) {
        uint32_t h0 = __umulhi(0xD2511F53u, c0), l0 = 0xD2511F53u * c0;
        uint32_t h1 = __umulhi(0xCD9E8D57u, c2), l1 = 0xCD9E8D57u * c2;
        uint32_t n0 = h1 ^ c1 ^ k0, n2 = h0 ^ c3 ^ k1;
        c0 = n0; c1 = l1; c2 = n2; c3 = l0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    o0 = c0; o1 = c1; o2 = c2; o3 = c3;
}

// the same function with the ten round keys precomputed on the host (DevParams.rk): saves 18 adds per block
__device__ __forceinline__ void philox4x32_10_rk(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, const uint32_t* rk,
                                                 uint32_t& o0, uint32_t& o1, uint32_t& o2, uint32_t& o3) {
#pragma unroll
    for (int r = 0; r < 10; r++) {
        uint32_t h0 = __umulhi(0xD2511F53u, c0), l0 = 0xD2511F53u * c0;
        uint32_t h1 = __umulhi(0xCD9E8D57u, c2), l1 = 0xCD9E8D57u * c2;
        uint32_t n0 = h1 ^ c1 ^ rk[2 * r], n2 = h0 ^ c3 ^ rk[2 * r + 1];
        c0 = n0; c1 = l1; c2 = n2; c3 = l0;
    }
    o0 = c0; o1 = c1; o2 = c2; o3 = c3;
}

__device__ __forceinline__ double u53(uint32_t hi, uint32_t lo) {
    return __ull2double_rn((((unsigned long long)hi << 32) | lo) >> 11) * 0x1.0p-53;
}

template <bool DEBUG>
__device__ __forceinline__ double uniform(Rng& g, const DevParams& P) {
    if (DEBUG && g.ru != nullptr) {
        if ((long long)g.n >= g.rn) { g.exhausted = true; g.n++; return 0.5; }
        return g.ru[g.n++];
    }
    uint32_t k = g.n++;
    if ((k & 1u) == 0u) {
        uint32_t o0, o1, o2, o3;
        philox4x32_10(k >> 1, g.c1, P.ctr2, P.ctr3, P.key0, P.key1, o0, o1, o2, o3);
        g.s2 = o2; g.s3 = o3;
        return u53(o1, o0);
    }
    return u53(g.s3, g.s2);
}

// two consecutive uniforms; one Philox block when the stream is block-aligned (the common case)
template <bool DEBUG>
__device__ __forceinline__ void uniform2(Rng& g, const DevParams& P, double& a, double& b) {
    if ((DEBUG && g.ru != nullptr) || (g.n & 1u)) {
        a = uniform<DEBUG>(g, P);
        b = uniform<DEBUG>(g, P);
        return;
    }
    uint32_t o0, o1, o2, o3;
    philox4x32_10(g.n >> 1, g.c1, P.ctr2, P.ctr3, P.key0, P.key1, o0, o1, o2, o3);
    g.n += 2; g.s2 = o2; g.s3 = o3;
    a = u53(o1, o0);
    b = u53(o3, o2);
}

// ---------------------------------------------------------------------------------------------
__device__ __noinline__ double mod2pi_slow(double x) {
    double k = floor(x / TWO_PI);
    double r = fma(-k, TWO_PI, x);
    r = r - k * TWO_PI_LO;
    if (r < 0.0) r += TWO_PI;
    if (r >= TWO_PI) r -= TWO_PI;
    return r;
}
__device__ __forceinline__ double mod2pi(double x) {  // Base.mod2pi semantics (SURVEY App. E)
    if (x >= 0.0 && x < TWO_PI) return x;
    if (x >= TWO_PI && x < 2 * TWO_PI) {  // k = 1 of the general formula, same roundings
        double r = (x - TWO_PI) - TWO_PI_LO;
        return r < 0.0 ? r + TWO_PI : r;
    }
    if (x < 0.0 && x > -TWO_PI) {  // k = -1 (phase is negative after a boost or a scattering)
        double r = (x + TWO_PI) + TWO_PI_LO;
        return r >= TWO_PI ? r - TWO_PI : r;
    }
    return mod2pi_slow(x);
}

__device__ __forceinline__ double norm3(double x, double y, double z) {
    double s = x * x + y * y + z * z;
    if (s == 0.0 || isinf(s)) {
        double m = fmax(fabs(x), fmax(fabs(y), fabs(z)));
        if (m == 0.0 || isinf(m)) return m;
        double a = x / m, b = y / m, c = z / m;
        return m * sqrt(a * a + b * b + c * c);
    }
    return sqrt(s);
}

__device__ __forceinline__ double sqrt_guard(const DevParams& P, double a) {
    if (MCS_UNLIKELY(a < 0.0)) { count(P, CNT_NEGSQRT); return 0.0; }
    return sqrt(a);
}

// get_psd_bins.jl:16-39
// `uses`: how many call sites of the reference this one evaluation stands for (each would have warned on its own)
__device__ __forceinline__ int psd_bin_momentum(const DevParams& P, double ptot_sk, int uses = 1) {
    int bin;
    if (ptot_sk < P.psd_mom_min) bin = 0;
    else bin = (int)trunc(log10(ptot_sk / P.psd_mom_min) * P.bpd_mom) + 1;
    if (bin > P.M) { count(P, CNT_W_PSDMOM, (unsigned long long)uses); bin = P.M; }
    return bin;
}
// get_psd_bins.jl:73-97
__device__ __forceinline__ int psd_bin_angle(const DevParams& P, double px_sk, double ptot_sk) {
    if (ptot_sk == 0.0) return 0;
    double p_cos = -px_sk / ptot_sk;
    int bin;
    if (p_cos < P.psd_cos_fine) {
        bin = P.T - (int)trunc((p_cos + 1) / P.delta_cos);
    } else {
        double th = acos(p_cos);
        bin = th < P.psd_theta_min ? 0 : (int)trunc(log10(th / P.psd_theta_min) * P.bpd_th) + 1;
    }
    return min(bin, P.T);
}
__device__ __noinline__ int psd_bin_momentum_ool(const DevParams& P, double ptot_sk, int uses) { return psd_bin_momentum(P, ptot_sk, uses); }
__device__ __noinline__ int psd_bin_angle_ool(const DevParams& P, double px_sk, double ptot_sk) { return psd_bin_angle(P, px_sk, ptot_sk); }
template <bool OOL>
__device__ __forceinline__ int bin_mom(const DevParams& P, double ptot_sk, int uses = 1) {
    return OOL ? psd_bin_momentum_ool(P, ptot_sk, uses) : psd_bin_momentum(P, ptot_sk, uses);
}
template <bool OOL>
__device__ __forceinline__ int bin_ang(const DevParams& P, double px_sk, double ptot_sk) {
    return OOL ? psd_bin_angle_ool(P, px_sk, ptot_sk) : psd_bin_angle(P, px_sk, ptot_sk);
}

// transformers.jl:440-476 (uz, utot do not enter the parallel-to-x boost as written)
__device__ __forceinline__ void transform_p_PS(const DevParams& P, double pb, double pperp, double gam_pf, double phi,
                                               double ux, double gsf, double bcos, double bsin, double& ptot_sk,
                                               double& sx, double& sz, double& gam_sk) {
    double sp, cp;
    sincos_bf(phi + HALF_PI, &sp, &cp);
    double p_p_cos = pperp * cp;
    double fx = pb * bcos - p_p_cos * bsin;
    double fy = pperp * sp;
    double fz = pb * bsin + p_p_cos * bcos;
    double dpx = (gsf - 1) * fx + gsf * gam_pf * P.m * ux;
    sx = fx + dpx;
    sz = fz;
    ptot_sk = norm3(sx, fy, sz);
    gam_sk = hypot(ptot_sk / P.mc, 1.0);
}

// the same with the gyro-phase given as (cos phi, sin phi): sin(phi + pi/2) = cos phi, cos(phi + pi/2) = -sin phi
__device__ __forceinline__ void transform_p_PS_cs(const DevParams& P, double pb, double pperp, double gam_pf, double cphi,
                                                  double sphi, double ux, double gsf, double bcos, double bsin, double& ptot_sk,
                                                  double& sx, double& sz, double& gam_sk) {
    const double p_p_cos = pperp * -sphi;
    const double fx = pb * bcos - p_p_cos * bsin;
    const double fy = pperp * cphi;
    const double fz = pb * bsin + p_p_cos * bcos;
    const double dpx = (gsf - 1) * fx + gsf * gam_pf * P.m * ux;
    sx = fx + dpx;
    sz = fz;
    ptot_sk = norm3(sx, fy, sz);
    gam_sk = hypot(ptot_sk / P.mc, 1.0);
}

// pmax test of particle_loop.jl:262-275 (cold: only above pmax_cutoff)
__device__ __noinline__ bool above_pmax_shock_frame(const DevParams& P, double pb, double pperp, double gam_pf, double phi,
                                                    int iz) {
    double ptot_sk, sx, sz, gam_sk;
    transform_p_PS(P, pb, pperp, gam_pf, phi, P.ux[iz], P.gsf[iz], P.costh[iz], P.sinth[iz], ptot_sk, sx, sz, gam_sk);
    return ptot_sk > P.pmax_cutoff;
}

// Scratch records for the out-of-line (cold) functions.  They are passed and returned BY VALUE so that the lane's
// long-lived state is never address-taken: a reference parameter of a noinline function pins the variable in
// local memory for its whole lifetime (seen as LDL/STL in the hot loop of the v4 profile).
struct Mom { double ptot, pb, pperp, gam_pf, phi; };
struct ColdIO {
    double x, prp_x, ptot, pb, pperp, gam_pf, gd, acct, phi;
    long long retro_steps;
    uint32_t rng_n, rng_s2, rng_s3;
    int tcut, i_return, fin;
    bool went_retro, lose_pt, exhausted, err;
};

// transformers.jl:523-607; zone `io` -> shock frame -> zone `in`
__device__ __noinline__ Mom transform_p_PSP(const DevParams& P, int io, int in, Mom mi) {
    double pb = mi.pb, pperp = mi.pperp, gam_pf = mi.gam_pf, phi = mi.phi;
    double ux_o = P.ux[io], uz_o = P.uz[io], gsf_o = P.gsf[io], bcos_o = P.costh[io], bsin_o = P.sinth[io];
    double ux = P.ux[in], uz = P.uz[in], gsf = P.gsf[in], bcos = P.costh[in], bsin = P.sinth[in];
    double sp, cp;
    sincos(phi + HALF_PI, &sp, &cp);
    double p_p_cos = pperp * cp;
    double fx = pb * bcos_o - p_p_cos * bsin_o;
    double fy = pperp * sp;
    double fz = pb * bsin_o + p_p_cos * bcos_o;
    double rxo = P.rxt[io], rzo = P.rzt[io], cro = P.crt[io];  // ux/ut, uz/ut, ux*uz/ut^2 tabulated by mcs_set_profile
    double sx = ((gsf_o - 1) * (rxo * rxo) + 1) * fx + (gsf_o - 1) * cro * fz + gsf_o * gam_pf * P.m * ux_o;
    double sy = fy;
    double sz = (gsf_o - 1) * cro * fx + ((gsf_o - 1) * (rzo * rzo) + 1) * fz + gsf_o * gam_pf * P.m * uz_o;
    double ptot_sk = norm3(sx, sy, sz);
    double pb_sk = sx * bcos + sz * bsin;
    if (ptot_sk < fabs(pb_sk)) count(P, CNT_W_PPERP);
    double gam_sk = hypot(ptot_sk / P.mc, 1.0);
    double rx = P.rxt[in], rz = P.rzt[in], cr = P.crt[in];
    double nx = ((gsf - 1) * (rx * rx) + 1) * sx + (gsf - 1) * cr * sz - gsf * gam_sk * P.m * ux;
    double ny = sy;
    double nz = (gsf - 1) * cr * sx + ((gsf - 1) * (rz * rz) + 1) * sz - gsf * gam_sk * P.m * uz;
    double pt = norm3(nx, ny, nz);
    double b = nx * bcos + nz * bsin, pp;
    if (pt < fabs(b)) {
        pp = 1.0e-6 * pt;
        b = copysign(sqrt(pt * pt - pp * pp), b);
        count(P, CNT_W_PPERP);
    } else {
        pp = sqrt(pt * pt - b * b);
    }
    Mom mo;
    mo.ptot = pt; mo.pb = b; mo.pperp = pp;
    mo.gam_pf = hypot(pt / P.mc, 1.0);
    mo.phi = atan2(ny, -nx * bsin + nz * bcos) - HALF_PI;
    return mo;
}

// The same boost with the gyro-phase carried as (cos phi, sin phi) — the fast loop's representation.  The reference's
// sincos(phi + pi/2) is (cos phi, -sin phi), and its new phase atan(ny, d) - pi/2 has cosine ny / h and sine -d / h with
// h = hypot(ny, d): no trigonometric call at all.
struct MomCS { double ptot, pb, pperp, gam_pf, cphi, sphi; };
__device__ MCS_COLD MomCS transform_p_PSP_cs(const DevParams& P, int io, int in, MomCS mi) {
    const double pb = mi.pb, pperp = mi.pperp, gam_pf = mi.gam_pf;
    const double ux_o = P.ux[io], uz_o = P.uz[io], gsf_o = P.gsf[io], bcos_o = P.costh[io], bsin_o = P.sinth[io];
    const double ux = P.ux[in], uz = P.uz[in], gsf = P.gsf[in], bcos = P.costh[in], bsin = P.sinth[in];
    const double p_p_cos = pperp * -mi.sphi;
    const double fx = pb * bcos_o - p_p_cos * bsin_o;
    const double fy = pperp * mi.cphi;
    const double fz = pb * bsin_o + p_p_cos * bcos_o;
    const double rxo = P.rxt[io], rzo = P.rzt[io], cro = P.crt[io];
    const double sx = ((gsf_o - 1) * (rxo * rxo) + 1) * fx + (gsf_o - 1) * cro * fz + gsf_o * gam_pf * P.m * ux_o;
    const double sy = fy;
    const double sz = (gsf_o - 1) * cro * fx + ((gsf_o - 1) * (rzo * rzo) + 1) * fz + gsf_o * gam_pf * P.m * uz_o;
    const double ptot_sk = norm3(sx, sy, sz);
    const double pb_sk = sx * bcos + sz * bsin;
    if (ptot_sk < fabs(pb_sk)) count(P, CNT_W_PPERP);
    const double gam_sk = hypot(ptot_sk / P.mc, 1.0);
    const double rx = P.rxt[in], rz = P.rzt[in], cr = P.crt[in];
    const double nx = ((gsf - 1) * (rx * rx) + 1) * sx + (gsf - 1) * cr * sz - gsf * gam_sk * P.m * ux;
    const double ny = sy;
    const double nz = (gsf - 1) * cr * sx + ((gsf - 1) * (rz * rz) + 1) * sz - gsf * gam_sk * P.m * uz;
    const double pt = norm3(nx, ny, nz);
    double b = nx * bcos + nz * bsin, pp;
    if (pt < fabs(b)) {
        pp = 1.0e-6 * pt;
        b = copysign(sqrt(pt * pt - pp * pp), b);
        count(P, CNT_W_PPERP);
    } else {
        pp = sqrt(pt * pt - b * b);
    }
    MomCS mo;
    mo.ptot = pt; mo.pb = b; mo.pperp = pp;
    mo.gam_pf = hypot(pt / P.mc, 1.0);
    const double d = -nx * bsin + nz * bcos, h = hypot(ny, d);
    if (h > 0.0) { mo.cphi = ny / h; mo.sphi = -d / h; }
    else { mo.cphi = 0.0; mo.sphi = -1.0; }  // atan(0, 0) = 0
    return mo;
}

__device__ __forceinline__ double perpendicular_momentum(const DevParams& P, double ptot, double pb) {
    if (ptot < fabs(pb)) { count(P, CNT_W_PPERP); return 1.0e-6 * ptot; }
    return sqrt(ptot * ptot - pb * pb);
}

__device__ __forceinline__ double radiation_loss(const DevParams& P, double B2, double p, double dt) {
    double d = P.rad_loss_fac * B2 * p * dt;
    return d > 1.0e-2 ? p / (1 + d) : p * (1 - d);
}

// cuts.jl:149-162
__device__ __noinline__ void tcut_track(const DevParams& P, int tcut_curr, double weight, double ptot) {
    int n = tally_add(P, &P.t.w_coupled[tcut_curr - 1], weight);
    int ip = psd_bin_momentum_ool(P, ptot, 1);
    n += tally_add(P, &P.t.s_coupled[ip + E1 * (tcut_curr - 1)], weight);
    count(P, CNT_RED, (unsigned long long)n);
}

// particle_loop.jl:652-723
__device__ __noinline__ Mom do_energy_transfer(const DevParams& P, int i_grid, int i_grid_old, Mom mi, double weight) {
    double ptot = mi.ptot, pb = mi.pb, pperp = mi.pperp, gam_pf = mi.gam_pf;
    int i_start = i_grid_old, i_stop = min(i_grid, P.i_shock);
    double E0 = P.m * (P.c * P.c), gam_f = 0.0;
    bool scale = false;
    double emax = -1.0, rmax = 0.0;  // F-11: empty range == nothing to do
    for (int i = i_start + 1; i <= i_stop; i++) {
        emax = fmax(emax, P.eps_target[i - 1]);
        rmax = fmax(rmax, P.recv_pool[i - 1]);
    }
    if (P.aa >= 1 && i_start + 1 <= i_stop && emax > 0) {
        double gam_i = hypot(1.0, ptot / P.mc);
        double eps_start = i_start >= 1 ? P.eps_target[i_start - 1] : 0.0;
        gam_f = 1 + (gam_i - 1) * (1 - P.eps_target[i_stop - 1]) / (1 - eps_start);
        int n_split = 0;
        for (int i = i_start + 1; i <= i_stop; i++) n_split += P.eps_target[i - 1] > 0;
        double inc = (gam_i - gam_f) * E0 * weight / n_split;
        int n = 0;
        for (int i = i_start + 1; i <= i_stop; i++)
            if (P.eps_target[i - 1] > 0) n += tally_add(P, &P.t.pool[i - 1], inc);
        count(P, CNT_RED, (unsigned long long)n);
        scale = true;
    } else if (rmax > 0) {
        double sum = 0.0;
        for (int i = i_start + 1; i <= i_stop; i++) sum += P.recv_pool[i - 1];
        double gam_i = hypot(1.0, ptot / P.mc);
        gam_f = gam_i + sum * P.ewf / E0;
        scale = true;
    }
    if (scale) {
        double pf = P.mc * sqrt_guard(P, gam_f * gam_f - 1);
        double s = pf / ptot;
        pb *= s; pperp *= s; ptot = pf; gam_pf = gam_f;
    }
    Mom mo;
    mo.ptot = ptot; mo.pb = pb; mo.pperp = pperp; mo.gam_pf = gam_pf; mo.phi = mi.phi;
    return mo;
}

// prob_return.jl:217-344.  Nested loop on the lane: retro passes are ~1e-3 of all passes.
template <bool DEBUG, bool ELECTRON>
__device__ __forceinline__ bool retro_time(const DevParams& P, Rng& rng, double& gd, double prp_x, double& ptot,
                                        double& pb, double& pperp, double& gam_pf, double& acct, double weight,
                                        int& tcut_curr, double& phi_out, long long& n_steps) {
    const int ng = P.n_grid;
    const bool custom = P.flags & F_CUSTOM_EPSB;
    const double xn_per = 10.0, phi_step = TWO_PI / xn_per;
    const double t_step_fac = TWO_PI * P.aa * P.mp * P.c * gd / xn_per;
    const double ux = -P.ux[ng], gsf = P.gsf[ng], gef = P.gef[ng];
    double B = P.bt[ng];
    if (custom) B *= sqrt(P.x_grid_stop / prp_x);
    const double bcos = P.costh[ng], bsin = P.sinth[ng];
    const double Bcmb = P.B_CMBz * gef;
    double B2 = B * B + Bcmb * Bcmb;
    bool lose = false;
    double x = prp_x;
    double phi = uniform<DEBUG>(rng, P) * TWO_PI;
    long long steps = 0;
    for (;;) {
        steps++;
        double x_old = x, phi_old = phi, ptot_old = ptot;
        double cos_old = pb / ptot, sin_old = pperp / ptot;
        if (custom) {
            B = P.bt[ng] * sqrt(P.x_grid_stop / x);
            B2 = B * B + Bcmb * Bcmb;
            gd = 1 / (P.zz * B);
        }
        double gyro_rad = pperp * P.c * gd;
        phi = mod2pi(phi_old + phi_step);
        double t_step = t_step_fac * gam_pf;
        double x_move = pb * t_step_fac / (P.aa * P.mp);
        double gyr = bsin != 0.0 ? gyro_rad * bsin * (cos(phi) - cos(phi_old)) : 0.0;
        x = x_old + gsf * (x_move * bcos - gyr + ux * t_step);
        acct += t_step * gef;
        if ((P.flags & F_TCUTS) && tcut_curr <= P.n_tcuts && acct >= P.tcuts[tcut_curr - 1]) {
            tcut_track(P, tcut_curr, weight, ptot);
            tcut_curr++;
        }
        phi = TWO_PI * uniform<DEBUG>(rng, P);
        pb = (2 * uniform<DEBUG>(rng, P) - 1) * ptot;
        pperp = sqrt_guard(P, ptot * ptot - pb * pb);
        if (ELECTRON && (P.flags & F_RAD_LOSSES)) ptot = radiation_loss(P, B2, ptot, t_step);
        if (ptot <= 0) {
            ptot = 1.0e-99; gam_pf = 1.0; lose = true;
            break;
        }
        if (P.flags & F_KEEP_NEW_PITCH) {
            double r = ptot / ptot_old;
            pb *= r; pperp *= r;
        } else {
            pb = ptot * cos_old; pperp = ptot * sin_old;
        }
        if (ELECTRON) gam_pf = hypot(1.0, ptot / P.mc);  // ions: ptot is unchanged, hypot returns the same bits
        if (x < prp_x) break;
        if (steps >= P.retro_cap) { count(P, CNT_RETRO_CAP); break; }
    }
    phi_out = phi;
    n_steps += steps;
    return lose;
}

// SURVEY 8(f1): what get_dNdp_2D (particle_counter.jl:426-445) and thermo_calcs (thermo_calcs.jl:133-164) build from the
// crossing log, accumulated on the fly so the log can stay small.  Out of line: only runs with cfg.bin_thermal.
__device__ __noinline__ int bin_thermal_crossing(const DevParams& P, int lo, int hi, double sx, double ptot_sk, double gam_sk,
                                                 double ux, double weight) {
    int n_at = 0;
    const double w = weight * (ptot_sk > fabs(sx * SPIKE_AWAY) ? fabs(SPIKE_AWAY / ux) : fabs(gam_sk * P.aa * P.mp / sx));
    const size_t sT = (size_t)(P.T + 2), sM = (size_t)(P.M + 2);
    const int k = psd_bin_momentum_ool(P, ptot_sk, 1), jt = psd_bin_angle_ool(P, sx, ptot_sk);
    const double E0 = P.m * (P.c * P.c), etot = hypot(ptot_sk * P.c, E0);
    for (int i = lo; i <= hi; i++) {
        n_at += tally_add(P, &P.t.therm_sf[(size_t)jt + sT * ((size_t)k + sM * (size_t)(i - 1))], w);
        const double g = P.gsf[i], b = P.ux[i] / P.c;
        double pxX = g * (sx - b * etot / P.c);
        const double ptX = sqrt((ptot_sk * ptot_sk - sx * sx) + pxX * pxX);
        if (fabs(pxX) > ptX) pxX = copysign(ptX, pxX);
        const int kX = psd_bin_momentum_ool(P, ptX, 1), jX = psd_bin_angle_ool(P, pxX, ptX);
        n_at += tally_add(P, &P.t.therm_pf[(size_t)jX + sT * ((size_t)kX + sM * (size_t)(i - 1))], w);
    }
    return n_at;
}

// ---------------------------------------------------------------------------------------------
// Process up to 32 queued events, one per lane, fully converged:
//   crossing event -> all_flux.jl:86-158 (transform to the shock frame, flux / PSD / thermal-log tallies, x_spec spectra,
//                     upstream-FEB scalars);
//   finish event   -> particle_finish.jl:46-107 and the downstream sums of particle_loop.jl:478-495.
// The n_grid-sized tallies and the scalars go to this warp's shared partials with plain adds in event order.
// Converged: butterfly sums (fixed order) of the escape / downstream scalars of one batch of events into the warp's partials.
__device__ __noinline__ void reduce_scalars(double s0, double s1, double s2, double s3, double s4, double s5, double s6, int ng) {
    static_assert(SC_N - 1 == 7, "reduce_scalars takes the first SC_N - 1 scalars");
    const WarpMem wm = warp_mem(threadIdx.x >> 5, ng);
    const int lane = threadIdx.x & 31;
    double v[7] = {s0, s1, s2, s3, s4, s5, s6};
#pragma unroll
    for (int k = 0; k < 7; k++) {
        double t = v[k];
        for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(FULL, t, o);
        if (lane == 0) wm.part[3 * ng + k] += t;
    }
}

template <bool OOL>
__device__ MCS_COLD void process_events(const DevParams& P, int base, int n_ev) {
    const int lane = threadIdx.x & 31, ng = P.n_grid;
    const WarpMem wm = warp_mem(threadIdx.x >> 5, ng);
    const bool act = lane < n_ev;
    const int q = base + (act ? lane : 0);
    const uint32_t fl = act ? wm.q_flags[q] : 0u;
    const double weight = act ? P.cur.weight[wm.q_ip[q]] : 0.0;
    const double pb = wm.q_pb[q], pperp = wm.q_pperp[q], gam_pf = wm.q_gam[q], cphi = wm.q_cphi[q], sphi = wm.q_sphi[q],
                 ptot = wm.q_ptot[q];
    const int i_new = wm.q_inew[q], i_old = wm.q_iold[q], iz = wm.q_iz[q];
    const double ux = P.ux[iz], gsf = P.gsf[iz], bcos = P.costh[iz], bsin = P.sinth[iz];
    double ptot_sk, sx, sz, gam_sk;
    transform_p_PS_cs(P, pb, pperp, gam_pf, cphi, sphi, ux, gsf, bcos, bsin, ptot_sk, sx, sz, gam_sk);
    const bool is_cross = (fl & EV_VALID) && !(fl & EV_FINISH), is_fin = (fl & EV_VALID) && (fl & EV_FINISH);
    const bool inj = fl & EV_INJ, up = fl & EV_UP;
    const double g0u0w = weight * P.gam0 * P.u0;  // reference order: value * weight * gam0 * u0 (kept below)
    (void)g0u0w;
    double sc[SC_N];
#pragma unroll
    for (int k = 0; k < SC_N; k++) sc[k] = 0.0;
    int lo = 1, hi = 0;
    double f_pxx = 0, f_pxz = 0, f_en = 0;
    bool thermal = false;
    int n_red = 0;  // atomics this lane issues into the tallies (reported as the achieved atomic rate)

    if (is_cross) {
        double pt_o_px_sk, abs_inv_vx;
        if (ptot_sk > fabs(sx * SPIKE_AWAY)) {
            pt_o_px_sk = SPIKE_AWAY;
            abs_inv_vx = fabs(SPIKE_AWAY / ux);
        } else {
            pt_o_px_sk = ptot_sk / sx;
            abs_inv_vx = fabs(gam_sk * P.aa * P.mp / sx);
        }
        double en_add;
        if ((gam_sk - 1) > P.E_rel_pt) en_add = (gam_sk - 1) * P.m * (P.c * P.c) * weight;
        else en_add = ptot_sk * ptot_sk / (2 * P.m) * weight;
        const uint32_t xmask = fl >> EV_XSPEC_SHIFT;
        if (xmask) {  // calculate_x_spec_spectra! :164-190
            double pt_o_px_pf = fmin(fabs(ptot / pb), SPIKE_AWAY);
            int ipt = bin_mom<OOL>(P, ptot_sk), ipf = bin_mom<OOL>(P, ptot);
            for (int i = 0; i < P.n_xspec; i++)
                if (xmask & (1u << i)) {
                    n_red += tally_add<OOL>(P, &P.t.spec_sf[ipt + E1 * i], weight * pt_o_px_sk);
                    double F = fabs(pb / sx) * (gam_sk / gam_pf);
                    n_red += tally_add<OOL>(P, &P.t.spec_pf[ipf + E1 * i], weight * pt_o_px_pf * F);
                }
        }
        const double sign_fac = up ? -1.0 : 1.0;
        if (!up) { lo = i_old + 1; hi = i_new; }
        else { lo = i_new + 1; hi = i_old; if (inj) lo = max(lo, P.i_grid_feb + 1); }  // :223-225
        f_pxx = sign_fac * sx * weight * P.gam0 * P.u0;
        f_pxz = fabs(sz) * weight * P.gam0 * P.u0;
        f_en = sign_fac * en_add * P.gam0 * P.u0;
        if (lo <= hi) {
            const double w = weight * abs_inv_vx;
            if (inj) {
                int ipt = bin_mom<OOL>(P, ptot_sk), jth = bin_ang<OOL>(P, sx, ptot_sk);
                const size_t stride = (size_t)(P.M + 2) * (size_t)(P.T + 2);
                double* cell = P.t.psd + (size_t)ipt + (size_t)(P.M + 2) * (size_t)jth + stride * (size_t)(lo - 1);
                for (int i = lo; i <= hi; i++, cell += stride) n_red += tally_add<OOL>(P, cell, w);
            } else {
                thermal = true;
                n_red += hi - lo + 1;  // crossing counts
            }
        }
        if (fl & EV_FEB_UP) {  // :155-158
            sc[SC_EN_ESC_UP] = en_add * P.gam0 * P.u0;
            sc[SC_PX_ESC_UP] = -(sx * weight * P.gam0 * P.u0);
        }
    }
    // thermal-crossing log (all_flux.jl:242-254): slots for the whole warp claimed with one atomic
    {
        const int nrec = thermal ? hi - lo + 1 : 0;
        int incl = nrec;
        for (int o = 1; o < 32; o <<= 1) {
            int t = __shfl_up_sync(FULL, incl, o);
            if (lane >= o) incl += t;
        }
        const int total = __shfl_sync(FULL, incl, 31);
        if (total > 0) {
            unsigned long long b0 = 0;
            if (lane == 0) b0 = atomicAdd(&P.t.counters[CNT_LOG], (unsigned long long)total);
            b0 = __shfl_sync(FULL, b0, 0);
            if (nrec > 0) {
                long long slot = (long long)b0 + (incl - nrec);
                const double w = weight * (ptot_sk > fabs(sx * SPIKE_AWAY) ? fabs(SPIKE_AWAY / ux) : fabs(gam_sk * P.aa * P.mp / sx));
                long long over = 0;
                for (int k = 0; k < nrec; k++, slot++) {
                    int i = up ? hi - k : lo + k;  // reference order: downstream ascending, upstream descending
                    if (slot < P.t.na_cr) { P.t.tg[slot] = i; P.t.tpx[slot] = sx; P.t.tpt[slot] = ptot_sk; P.t.tw[slot] = w; }
                    else over++;
                }
                if (over) count(P, CNT_LOG_OVER, (unsigned long long)over);
            }
        }
        if (P.t.therm_sf != nullptr && nrec > 0) n_red += bin_thermal_crossing(P, lo, hi, sx, ptot_sk, gam_sk, ux, weight);
    }
    if (is_fin) {
        const int reason = (fl >> EV_REASON_SHIFT) & 7;
        const double E0 = P.m * (P.c * P.c);
        if (reason == 1 || reason == 2) {
            int ip = min(bin_mom<OOL>(P, ptot_sk), MCS_PSD_MAX), jt = min(bin_ang<OOL>(P, sx, ptot_sk), MCS_PSD_MAX);
            double wf;
            if (ptot_sk > fabs(SPIKE_AWAY * sx)) wf = gam_sk * P.m * SPIKE_AWAY / ptot_sk;
            else wf = gam_sk * (P.m / fabs(sx));
            if (reason == 1) {
                n_red += tally_add<OOL>(P, &P.t.esc_dn[ip + E1 * jt], weight * wf);
            } else {
                sc[SC_ESC_FLUX] = weight;
                n_red += tally_add<OOL>(P, &P.t.esc_up[ip + E1 * jt], weight * wf);
                bool rel = (gam_sk - 1) >= P.E_rel_pt;  // F-8
                double Ek = rel ? (gam_sk - 1) * E0 : ptot_sk * ptot_sk / (2 * P.m);
                double en_add = Ek * weight;
                sc[SC_PX_ESC_FEB] = fabs(sx) * weight;
                sc[SC_EN_ESC_FEB] = en_add;
                n_red += tally_add<OOL>(P, &P.t.esc_en_eff[ip], en_add);
                n_red += tally_add<OOL>(P, &P.t.esc_num_eff[ip], weight);
            }
        }
        if (fl & EV_SUMP) {  // particle_loop.jl:478-486
            double vel = ptot / P.m;
            if ((gam_pf - 1) >= P.E_rel_pt) vel /= gam_pf;
            sc[SC_SUMP] = ptot / 3 * vel * weight * P.n0;
            sc[SC_SUMKE] = (gam_pf - 1) * P.m * (P.c * P.c) * weight * P.n0;
        }
    }
    // ---- ordered accumulation into the warp's partials --------------------------------------------------------------
    // Nearly every crossing covers ONE zone.  Those are added by their own lanes, all zones in parallel: lanes that hit the
    // same zone take turns in lane (= queue) order, so the order of the adds into any cell is fixed.  The few events that
    // span several zones follow, one after the other, with the lanes spread over the zones.
    {
        const bool single = is_cross && lo == hi;
        const unsigned peers = __match_any_sync(FULL, single ? lo : -1 - lane);
        const int turn = __popc(peers & ((1u << lane) - 1u));
        int n_turns = single ? __popc(peers) : 0;
        for (int o = 16; o > 0; o >>= 1) n_turns = max(n_turns, __shfl_xor_sync(FULL, n_turns, o));
        for (int r = 0; r < n_turns; r++) {
            if (single && turn == r) {
                wm.part[lo - 1] += f_pxx;
                wm.part[ng + lo - 1] += f_pxz;
                wm.part[2 * ng + lo - 1] += f_en;
            }
            __syncwarp();
        }
        if (single && thermal) red_add_u64(&P.t.ncross[lo - 1], 1ull);  // integer adds: any order
    }
    unsigned todo = __ballot_sync(FULL, is_cross && lo < hi);
    while (todo) {
        const int e = __ffs(todo) - 1;
        todo &= todo - 1;
        const int lo_e = __shfl_sync(FULL, lo, e), hi_e = __shfl_sync(FULL, hi, e);
        const double a = __shfl_sync(FULL, f_pxx, e), b = __shfl_sync(FULL, f_pxz, e), c = __shfl_sync(FULL, f_en, e);
        const int th = __shfl_sync(FULL, (int)thermal, e);
        for (int j = lo_e + lane; j <= hi_e; j += 32) {
            wm.part[j - 1] += a;
            wm.part[ng + j - 1] += b;
            wm.part[2 * ng + j - 1] += c;
            if (th) red_add_u64(&P.t.ncross[j - 1], 1ull);
        }
        __syncwarp();  // the next event's lanes may touch the same cells: order the read-modify-write chain
    }
    bool any_sc = false;
#pragma unroll
    for (int k = 0; k < SC_N; k++) any_sc |= sc[k] != 0.0;
    if (__any_sync(FULL, any_sc)) {
        reduce_scalars(sc[0], sc[1], sc[2], sc[3], sc[4], sc[5], sc[6], ng);  // rare (finish / FEB events): one shared copy
    }
    for (int o = 16; o > 0; o >>= 1) n_red += __shfl_xor_sync(FULL, n_red, o);
    if (lane == 0 && n_red > 0) count(P, CNT_RED, (unsigned long long)n_red);
    __syncwarp();
}

// Everything of the downstream end of Code Block 2 that is not the common case: downstream_test (particle_loop.jl:595-637)
// and prob_return (prob_return.jl:36-173) with retro_time.  State goes in and out by value (ColdIO).
template <bool DEBUG, bool ELECTRON>
__device__ __noinline__ ColdIO downstream_block(const DevParams& P, ColdIO io, double x_old, double grt, double weight,
                                                int helix, uint32_t rng_c1, const double* ru, long long rn) {
    const bool custom = P.flags & F_CUSTOM_EPSB;
    Rng rng;
    rng.n = io.rng_n; rng.s2 = io.rng_s2; rng.s3 = io.rng_s3; rng.c1 = rng_c1; rng.ru = ru; rng.rn = rn;
    rng.exhausted = io.exhausted;
    double x = io.x, prp_x = io.prp_x, ptot = io.ptot, pb = io.pb, pperp = io.pperp, gam_pf = io.gam_pf, gd = io.gd,
           acct = io.acct, phi = io.phi;
    int tcut = io.tcut, i_return = io.i_return, fin = -1;
    long long retro_steps = io.retro_steps;
    bool went_retro = false, lose_pt = false;
    bool do_prob_ret = true;
    if (P.feb_dn > 0 && x > P.feb_dn) {
        i_return = 0; do_prob_ret = false;
    } else if (x > 1.1 * prp_x) {
        double v_fac;
        if (ELECTRON && ptot < P.pe_crit) {
            double gyro_fac = P.pe_crit * P.c * gd;
            v_fac = gyro_fac * P.pe_crit / (P.m * P.gam_e_crit * P.u2);
        } else {
            v_fac = grt * ptot / (P.m * gam_pf * P.u2);
        }
        double L = P.eta_mfp / 3 * v_fac;
        if (x > 6.91 * L) { i_return = 0; do_prob_ret = false; }
    }
    if (do_prob_ret) {
        i_return = 2;
        if (x < P.x_grid_stop) {
        } else if (x_old < P.x_grid_stop && P.x_grid_stop <= x) {
            double gyro_tmp = (custom && x > P.x_grid_stop) ? sqrt(P.x_grid_stop / x) : 1.0;
            double g2 = ptot * P.c * gyro_tmp / (P.qcgs * P.bmag2);  // K-5
            double L = P.eta_mfp / 3 * g2 * ptot / (P.aa * P.mp * gam_pf * P.u2);
            prp_x = x + 3 * L;
        } else if (x_old < prp_x && x >= prp_x) {
            double vt = ptot / (gam_pf * P.aa * P.mp);
            double r = (vt - P.u2) / (vt + P.u2);
            if (vt < P.u2 || uniform<DEBUG>(rng, P) > r * r) {
                i_return = 0;
            } else {
                i_return = 1;
                if (!(P.flags & F_RETRO)) {
                    fin = MCS_FATE_ERROR;  // reference: error() prob_return.jl:134
                } else {
                    went_retro = true;
                    lose_pt = retro_time<DEBUG, ELECTRON>(P, rng, gd, prp_x, ptot, pb, pperp, gam_pf, acct, weight, tcut,
                                                         phi, retro_steps);
                    if (lose_pt) i_return = 0;
                    x = prp_x;
                }
            }
        } else if (ELECTRON && ptot < P.pcut_prev && helix % 1000 == 0) {
            double g2 = ptot * P.c * gd;
            double L = P.eta_mfp / 3 * g2 * ptot / (P.aa * P.mp * gam_pf * P.u2);
            if (x > 2.0e3 * L) prp_x = 0.8 * x;
            else prp_x = fmin(prp_x, P.x_grid_stop + L * pow(P.pcut_prev / ptot, 5.0));
        }
    }
    ColdIO o;
    o.x = x; o.prp_x = prp_x; o.ptot = ptot; o.pb = pb; o.pperp = pperp; o.gam_pf = gam_pf; o.gd = gd; o.acct = acct;
    o.phi = phi; o.retro_steps = retro_steps; o.rng_n = rng.n; o.rng_s2 = rng.s2; o.rng_s3 = rng.s3; o.tcut = tcut;
    o.i_return = i_return; o.fin = fin; o.went_retro = went_retro; o.lose_pt = lose_pt; o.exhausted = rng.exhausted;
    o.err = false;
    return o;
}

// no_DSA_loop reflection branch (particle_loop.jl:551-568): only when a not-yet-injected particle steps back upstream.
// Uses io.{x, pb, phi, rng_*}; sets io.err if the loop does not terminate.
template <bool DEBUG>
__device__ __noinline__ ColdIO reflect_loop(const DevParams& P, ColdIO io, double x_old, double phi_old, double dphi,
                                            double t_step, double inv_gm, double gsf, double bcos, double bsin, double gr,
                                            double ux, uint32_t rng_c1, const double* ru, long long rn) {
    Rng rng;
    rng.n = io.rng_n; rng.s2 = io.rng_s2; rng.s3 = io.rng_s3; rng.c1 = rng_c1; rng.ru = ru; rng.rn = rn;
    rng.exhausted = io.exhausted;
    double pb = io.pb, phi = io.phi, x = io.x;
    bool err = false;
    for (int pass = 0;; pass++) {
        if ((P.flags & F_DONT_DSA) || uniform<DEBUG>(rng, P) > P.inj_frac) {
            if (pb < 0) pb = -pb; else phi = uniform<DEBUG>(rng, P) * TWO_PI;
        } else break;
        phi = mod2pi(phi + dphi);
        double x_move = pb * t_step * inv_gm;
        double gyr = bsin != 0.0 ? gr * bsin * (cos(phi) - cos(phi_old)) : 0.0;
        x = x_old + gsf * (x_move * bcos - gyr + ux * t_step);
        if (!(x <= 0 && x_old > 0)) break;
        if (pass > 1000) { err = true; break; }
    }
    io.pb = pb; io.phi = phi; io.x = x; io.err = err;
    io.rng_n = rng.n; io.rng_s2 = rng.s2; io.rng_s3 = rng.s3; io.exhausted = rng.exhausted;
    return io;
}

// ---------------------------------------------------------------------------------------------
// Lane state.  The full record lives in local memory: the general section (out of line) works on a copy of it, the
// fast loop keeps only what a plain pass needs in registers.  Splitting the kernel this way is what lets the fast loop
// run at 64-80 registers (24-32 warps per SM): with the general pass inlined next to it the allocation was 128
// registers with spills inside the loop (profiles/r01_v13_*).
struct Lane {
    double mu, sn, cph, sph;  // the fast loop's pitch and phase registers, kept across sections while cs_valid (see below)
    double ptot, pb, pperp, x, prp_x, acct, phi;
    double gam_pf, gd, grt, gr, gper, t_step, inv_ptot, inv_gm;
    double ux, gsf, gef, bsin, bcos;
    const double* rng_ru;
    long long rng_rn;
    int ip, next_j, iz, i_grid, i_grid_old, helix, tcut, i_return, xsel, slot, qn;
    uint32_t rng_n, rng_s2, rng_s3, rng_c1;
    bool rng_exhausted, queue_empty, down, inj, x_old_le0, parked;
    // A lane that leaves the fast loop WITHOUT needing the general pass (the warp left because of other lanes) must come
    // back with bit-identical registers: pb = ptot * mu -> mu = pb / ptot is not the identity, and how often a warp leaves
    // depends on which particles share it.  With the registers kept here a particle's arithmetic depends on nothing but
    // itself, so per-particle results are the same for any schedule and any number of GPUs.
    bool cs_valid;
    uint32_t cs_flags;  // ST_RAN | ST_MUSN | ST_PHI carried along
};

// One shared out-of-line copy of the drain for everything outside the fast loop (the general section's two push sites and
// the end of the kernel): three fewer inlined copies of ~16 KB each for the instruction caches to hold.
__device__ __noinline__ void process_events_ool(const DevParams& P, int base, int n_ev) { process_events<true>(P, base, n_ev); }

// Converged: append the lanes' events (ev != 0) to the warp's queue, drain a full batch.  Returns the new queue length.
// INLINE_DRAIN: the fast loop folds the drain in (an ABI call there forces the loop's registers through local memory).
// OOL_HELPERS: that folded-in drain calls the out-of-line bin evaluation / accumulator add (the SLIM kernel: 5181 instead of
// 6743 instructions; +5 % on ladders of many short pcuts, -0.5 % on long ones — chosen per launch by the host, see launch_pcut).
template <bool INLINE_DRAIN, bool OOL_HELPERS = true>
__device__ __forceinline__ int push_events(const DevParams& P, const WarpMem& wm, int qn, uint32_t ev, int ip, double pb,
                                           double pperp, double gam_pf, double cphi, double sphi, double ptot, int i_new,
                                           int i_old, int iz) {
    const unsigned m = __ballot_sync(FULL, ev != 0u);
    if (m) {
        const int cnt = __popc(m);
        if (QCAP < 64 && qn + cnt > QCAP) {  // would not fit: drain what is queued as a partial batch first
            __syncwarp();
            if (INLINE_DRAIN) process_events<OOL_HELPERS>(P, 0, qn); else process_events_ool(P, 0, qn);
            qn = 0;
        }
        if (ev) {
            const int q = qn + __popc(m & ((1u << (threadIdx.x & 31)) - 1u));
            wm.q_pb[q] = pb; wm.q_pperp[q] = pperp; wm.q_gam[q] = gam_pf; wm.q_cphi[q] = cphi; wm.q_sphi[q] = sphi;
            wm.q_ip[q] = ip;  // the weight is fetched when the queue is drained (32 lanes at once)
            wm.q_ptot[q] = ptot; wm.q_inew[q] = i_new; wm.q_iold[q] = i_old; wm.q_iz[q] = iz; wm.q_flags[q] = ev;
        }
        qn += cnt;
        if (qn >= 32) {  // sums commute; the order is fixed by the lock-step schedule
            __syncwarp();
            if (INLINE_DRAIN) process_events<OOL_HELPERS>(P, qn - 32, 32); else process_events_ool(P, qn - 32, 32);
            qn -= 32;
        }
    }
    return qn;
}

// Converged: give every lane of `need` (idle, queue not yet found empty) the next particle of this warp's sequence —
// chunks of 32 consecutive particles dealt round-robin to the warps (deterministic), or one atomic per warp on a global
// queue head (dynamic) — and set up its record (particle_loop.jl:44-96, 131-153).
template <bool DEBUG>
__device__ __forceinline__ void refill_lanes(const DevParams& P, Lane& l, const unsigned need, const bool fast_ok) {
    const int ng = P.n_grid;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
    const bool custom = P.flags & F_CUSTOM_EPSB, dynamic = P.flags & F_DYNAMIC_QUEUE;
    const long long total_warps = (long long)gridDim.x * n_warps, gwarp = (long long)blockIdx.x * n_warps + warp;
    const int rank = __popc(need & ((1u << lane) - 1u));
    long long base;
    if (dynamic) {
        base = 0;
        const int leader = __ffs(need) - 1;
        if (lane == leader) base = (long long)atomicAdd(&P.t.counters[CNT_QUEUE], (unsigned long long)__popc(need));
        base = __shfl_sync(FULL, base, leader);
    } else {
        base = l.next_j;
        l.next_j += __popc(need);
    }
    if (!((need >> lane) & 1u)) return;
    const long long j = base + rank;
    const long long mine = dynamic ? j : ((j >> 5) * total_warps + gwarp) * 32 + (j & 31);
    if (mine >= P.n_use) { l.queue_empty = true; return; }
    const int ip = (int)mine;
    l.ip = ip;
    l.ptot = P.cur.ptot[ip]; l.pb = P.cur.pb[ip]; l.x = P.cur.x[ip];
    const double xn_per = P.cur.xn_per[ip];
    l.prp_x = P.cur.prp_x[ip]; l.acct = P.cur.acctime[ip]; l.phi = P.cur.phi[ip];
    l.i_grid = (int)P.cur.grid[ip]; l.i_grid_old = l.i_grid; l.tcut = (int)P.cur.tcut[ip];
    l.down = P.cur.down[ip]; l.inj = P.cur.inj[ip];
    l.helix = 0; l.i_return = -1; l.t_step = 0.0; l.x_old_le0 = true; P.retro[ip] = 0;
    l.xsel = xn_per == P.xn_fine ? 0 : (xn_per == P.xn_coarse ? 1 : 2);
    // A fresh particle needs nothing the fast loop cannot do, unless its record is outside what the loop itself
    // produces (hand-made populations): those take the general pass first.
    l.parked = !fast_ok || l.xsel > 1 || l.prp_x < P.x_grid_stop || (l.inj && l.x < P.feb_up) || (l.down && !l.inj && l.x < 0) ||
               l.i_grid > ng;
    l.gam_pf = hypot(1.0, l.ptot / P.mc);
    l.gd = 1 / (P.zz * P.bt[l.i_grid]);
    if (custom && l.x > P.x_grid_stop) l.gd *= sqrt(l.x / P.x_grid_stop);
    l.grt = l.ptot * P.c * l.gd;
    l.gper = TWO_PI * l.gam_pf * P.m * P.c * l.gd;
    l.iz = l.i_grid;
    const int iz = l.iz;
    l.ux = P.ux[iz]; l.gsf = P.gsf[iz]; l.gef = P.gef[iz]; l.bsin = P.sinth[iz]; l.bcos = P.costh[iz];
    l.pperp = perpendicular_momentum(P, l.ptot, l.pb);
    l.gr = l.pperp * P.c * l.gd;
    l.inv_ptot = 1 / l.ptot; l.inv_gm = 1 / (l.gam_pf * P.m);
    l.rng_n = 0; l.rng_c1 = (uint32_t)(P.first_global + ip); l.rng_exhausted = false;
    l.cs_valid = false; l.cs_flags = 0u;
    if (DEBUG) {
        l.rng_ru = nullptr; l.rng_rn = 0;
        if (P.replay_u != nullptr && ip < P.replay_n) {
            l.rng_ru = P.replay_u + P.replay_off[ip];
            l.rng_rn = P.replay_off[ip + 1] - P.replay_off[ip];
        }
        l.slot = P.trace_slot ? P.trace_slot[ip] : -1;
    }
}

// ---------------------------------------------------------------------------------------------
// General section: refill idle lanes, then run ONE full helix-loop pass (particle_loop.jl:154-499) for every lane that
// asked for it (`parked`), including everything rare: escapes, pcut save, tcuts, energy transfer, reflection, probability
// of return with retro_time, radiative losses, custom eps_B, replay/trace.  Repeats while lanes still need it (a particle
// that finished is replaced at once; a particle back from retro_time gets its follow-up pass).  Returns true when the
// warp has no particles left.  Configurations the fast loop cannot do (fast_ok false) never leave this function.
template <bool DEBUG, bool ELECTRON>
__device__ __noinline__ bool general_section(const DevParams& P, Lane& Lref, const bool fast_ok) {
    Lane l = Lref;
    const int ng = P.n_grid;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
    const WarpMem wm = warp_mem(warp, ng);
    const uint32_t flags = P.flags;
    const bool custom = flags & F_CUSTOM_EPSB, dont_scatter = flags & F_DONT_SCATTER, dynamic = flags & F_DYNAMIC_QUEUE;
    const bool rad = ELECTRON && (flags & F_RAD_LOSSES);
    const long long total_warps = (long long)gridDim.x * n_warps, gwarp = (long long)blockIdx.x * n_warps + warp;
    int &ip = l.ip, &next_j = l.next_j, &iz = l.iz, &i_grid = l.i_grid, &i_grid_old = l.i_grid_old, &helix = l.helix,
        &tcut = l.tcut, &i_return = l.i_return, &xsel = l.xsel, &slot = l.slot, &qn = l.qn;
    double &ptot = l.ptot, &pb = l.pb, &pperp = l.pperp, &x = l.x, &prp_x = l.prp_x, &acct = l.acct, &phi = l.phi;
    double &gam_pf = l.gam_pf, &gd = l.gd, &grt = l.grt, &gr = l.gr, &gper = l.gper, &t_step = l.t_step,
           &inv_ptot = l.inv_ptot, &inv_gm = l.inv_gm;
    double &ux = l.ux, &gsf = l.gsf, &gef = l.gef, &bsin = l.bsin, &bcos = l.bcos;
    bool &queue_empty = l.queue_empty, &down = l.down, &inj = l.inj, &x_old_le0 = l.x_old_le0, &parked = l.parked;
    Rng rng;
    rng.n = l.rng_n; rng.s2 = l.rng_s2; rng.s3 = l.rng_s3; rng.c1 = l.rng_c1; rng.ru = l.rng_ru; rng.rn = l.rng_rn;
    rng.exhausted = l.rng_exhausted;
    bool all_done = false;

    for (;;) {
        // ---- refill idle lanes ---------------------------------------------------------------------
        {
            const unsigned need = __ballot_sync(FULL, ip < 0 && !queue_empty);
            if (need != 0u) {
                l.rng_n = rng.n; l.rng_c1 = rng.c1; l.rng_exhausted = rng.exhausted; l.rng_ru = rng.ru; l.rng_rn = rng.rn;
                refill_lanes<DEBUG>(P, l, need, fast_ok);
                rng.n = l.rng_n; rng.c1 = l.rng_c1; rng.exhausted = l.rng_exhausted; rng.ru = l.rng_ru; rng.rn = l.rng_rn;
            }
        }
        if (__all_sync(FULL, ip < 0)) { all_done = true; break; }
        if (!__any_sync(FULL, ip >= 0 && parked)) break;  // nobody asks for the general pass: back to the fast loop

        // ---- one pass of the helix loop (particle_loop.jl:154-499) ------------------------------------
        int fin = -1;          // -1 running; 0 saved; 1..4 i_reason; 5 error
        uint32_t ev = 0;       // crossing event to queue at point A
        bool moved = false;
        double x_old = 0.0;    // position before this pass's move
        const bool served = ip >= 0 && parked;
        if (served) {
            l.cs_valid = false;
            helix++;
            if (MCS_UNLIKELY(helix > P.helix_cap)) {
                fin = 1;  // K-1
            } else if (MCS_UNLIKELY(i_return == 1)) {
                pperp = perpendicular_momentum(P, ptot, pb);
                gr = pperp * P.c * gd;
            } else {
                // Code Block 3
                const int iz_old = iz;
                const bool zc = i_grid != iz;
                if (MCS_UNLIKELY(zc)) {
                    iz = i_grid;
                    ux = P.ux[iz]; gsf = P.gsf[iz]; gef = P.gef[iz]; bsin = P.sinth[iz]; bcos = P.costh[iz];
                    gd = 1 / (P.zz * P.bt[iz]);
                }
                double bmag = 0.0;
                if (custom || rad) {
                    bmag = (custom && x > P.x_grid_stop) ? P.bt[ng] * sqrt(P.x_grid_stop / x) : P.bt[iz];
                    gd = 1 / (P.zz * bmag);
                }
                if (MCS_UNLIKELY(zc && ux != P.ux[iz_old])) {
                    Mom mi;
                    mi.ptot = ptot; mi.pb = pb; mi.pperp = pperp; mi.gam_pf = gam_pf; mi.phi = phi;
                    const Mom mo = transform_p_PSP(P, iz_old, iz, mi);
                    ptot = mo.ptot; pb = mo.pb; pperp = mo.pperp; gam_pf = mo.gam_pf; phi = mo.phi;
                    gr = pperp * P.c * gd;
                    grt = ptot * P.c * gd;
                    inv_ptot = 1 / ptot; inv_gm = 1 / (gam_pf * P.m);
                }
                if (MCS_UNLIKELY(P.energy_transfer_frac > 0 && !inj && x_old_le0 && i_grid_old != i_grid)) {
                    Mom mi;
                    mi.ptot = ptot; mi.pb = pb; mi.pperp = pperp; mi.gam_pf = gam_pf; mi.phi = phi;
                    const Mom mo = do_energy_transfer(P, i_grid, i_grid_old, mi, P.cur.weight[ip]);
                    ptot = mo.ptot; pb = mo.pb; pperp = mo.pperp; gam_pf = mo.gam_pf;
                    inv_ptot = 1 / ptot; inv_gm = 1 / (gam_pf * P.m);
                }
                if (dont_scatter && x > 10 * gr) {
                    i_return = 0; fin = 1;
                } else if (MCS_UNLIKELY(ptot > P.pmax_cutoff) && above_pmax_shock_frame(P, pb, pperp, gam_pf, phi, iz)) {
                    fin = 2;
                }
                if (MCS_UNLIKELY(fin < 0 && inj && x < P.feb_up)) fin = 2;
                if (MCS_UNLIKELY(fin < 0 && P.age_max > 0 && acct > P.age_max)) fin = 3;
                if (rad && fin < 0) {
                    double p_old = ptot, Bcmb = P.B_CMBz * gef;
                    ptot = radiation_loss(P, bmag * bmag + Bcmb * Bcmb, ptot, t_step);
                    if (ptot <= 0) {
                        ptot = 1.0e-99; pb = 1.0e-99; pperp = 1.0e-99; gam_pf = 1;
                        fin = 4;
                    } else {
                        gam_pf = hypot(ptot / P.mc, 1.0);
                        pb *= ptot / p_old;
                        pperp *= ptot / p_old;
                        grt = ptot * P.c * gd;
                        gr = pperp * P.c * gd;
                        inv_ptot = 1 / ptot; inv_gm = 1 / (gam_pf * P.m);
                    }
                }
                if (MCS_LIKELY(fin < 0)) {
                    if (MCS_LIKELY(!dont_scatter)) {
                        // scattering.jl:29-101; cos_max depends on xn_per only and is precomputed
                        if (ELECTRON && ptot < P.pe_crit) gper = TWO_PI * P.gam_e_crit * P.mc * gd;
                        else gper = TWO_PI * gam_pf * P.mc * gd;
                        double omc;
                        if (xsel < 2) omc = P.omc[xsel];
                        else omc = 1 - cos(sqrt(6 * TWO_PI / (P.cur.xn_per[ip] * P.eta_mfp)));
                        double u1, u2;
                        uniform2<DEBUG>(rng, P, u1, u2);
                        const double cos_old = pb * inv_ptot, sin_old = pperp * inv_ptot;
                        const double cos_d = 1 - u1 * omc;
                        const double sin_d = sqrt_guard(P, 1 - cos_d * cos_d);
                        const double phi_s = u2 * TWO_PI - PI;
                        double sps, cps;
                        sincos_bf(phi_s, &sps, &cps);
                        const double cos_new = cos_old * cos_d + sin_old * sin_d * cps;
                        const double sin_new = sqrt_guard(P, 1 - cos_new * cos_new);
                        pb = ptot * cos_new;
                        pperp = ptot * sin_new;
                        double phi_p = phi + HALF_PI;
                        if (MCS_LIKELY(sin_new != 0)) {
                            double s = sps * sin_d / sin_new;
                            if (fabs(s) > SIN_UPPER_LIMIT) s = copysign(SIN_UPPER_LIMIT, s);
                            phi_p += asin_bf(s);
                        }
                        phi = phi_p - HALF_PI;
                    }
                    if (down) {
                        acct += t_step * gef;
                        if (MCS_UNLIKELY((flags & F_TCUTS) && tcut <= P.n_tcuts && acct >= P.tcuts[tcut - 1])) {
                            tcut_track(P, tcut, P.cur.weight[ip], ptot);
                            tcut++;
                        }
                        if (MCS_UNLIKELY(ptot > P.pcut)) fin = 0;  // saved below
                    }
                    if (fin < 0) xsel = x > grt ? 1 : 0;  // xn_per = coarse : fine (particle_loop.jl:385)
                }
            }
            if (MCS_LIKELY(fin < 0)) {
                // Code Block 2: move (no_DSA_loop :510-571), shock crossing, zone search (all_flux.jl:65-82)
                moved = true;
                x_old = x;
                const double phi_old = phi;
                double dphi;
                if (MCS_LIKELY(xsel < 2)) { t_step = gper * P.inv_xn[xsel]; dphi = P.dphi[xsel]; }
                else { const double xn_per = P.cur.xn_per[ip]; t_step = gper / xn_per; dphi = TWO_PI / xn_per; }
                phi = mod2pi(phi + dphi);
                const double x_move = pb * t_step * inv_gm;
                const double gyr = MCS_UNLIKELY(bsin != 0.0) ? gr * bsin * (cos_bf(phi) - cos_bf(phi_old)) : 0.0;
                x = x_old + gsf * (x_move * bcos - gyr + ux * t_step);
                bool err = false;
                if (MCS_UNLIKELY(x <= 0 && x_old > 0 && !inj && ((flags & F_DONT_DSA) || P.inj_frac < 1))) {
                    ColdIO io;
                    io.x = x; io.pb = pb; io.phi = phi; io.rng_n = rng.n; io.rng_s2 = rng.s2; io.rng_s3 = rng.s3;
                    io.exhausted = rng.exhausted;
                    const ColdIO o = reflect_loop<DEBUG>(P, io, x_old, phi_old, dphi, t_step, inv_gm, gsf, bcos, bsin, gr, ux,
                                                         rng.c1, rng.ru, rng.rn);
                    x = o.x; pb = o.pb; phi = o.phi; err = o.err;
                    rng.n = o.rng_n; rng.s2 = o.rng_s2; rng.s3 = o.rng_s3; rng.exhausted = o.exhausted;
                }
                if (MCS_UNLIKELY(x_old < 0 && x >= 0)) {
                    down = true;
                    double Ld = P.eta_mfp / 3 * grt * ptot / (P.m * gam_pf * P.u2);
                    prp_x = fmax(prp_x, Ld);
                }
                if (down && x < 0) inj = true;
                i_grid_old = i_grid;
                {   // all_flux.jl:65-82. Common case first: one load decides "same zone" for either direction
                    const bool dn = x > x_old;
                    const double edge = P.xg[i_grid + (dn ? 1 : 0)];
                    const bool same = dn ? (edge > x) : (edge <= x);
                    if (MCS_UNLIKELY(!same)) {  // linear scans from the current zone (K-3)
                        if (dn) {
                            int k = i_grid + 1;
                            while (k <= ng + 1 && !(P.xg[k] > x)) k++;
                            if (k > ng + 1) err = true;
                            i_grid = k - 1;
                        } else {
                            int k = i_grid;
                            while (k >= 0 && !(P.xg[k] <= x)) k--;
                            if (k < 0) err = true;
                            i_grid = k;
                        }
                    }
                }
                if (MCS_UNLIKELY(err)) {
                    fin = MCS_FATE_ERROR;
                    i_grid = i_grid_old;
                }
            }
        }
        // crossing event? (all_flux.jl:80-82 early-out inverted), evaluated by every lane in converged code
        if (moved && fin < 0 && !(i_grid == i_grid_old && i_grid > P.i_grid_feb && P.n_xspec == 0)) {
            ev = (inj ? EV_INJ : 0u) | (x > x_old ? 0u : EV_UP) | ((inj && x < P.feb_up && x_old >= P.feb_up) ? EV_FEB_UP : 0u);
            for (int i = 0; i < P.n_xspec; i++) {
                const double xs = P.x_spec[i];
                if ((x_old < xs && x >= xs) || (x <= xs && x_old > xs)) ev |= 1u << (EV_XSPEC_SHIFT + i);
            }
            // with the zone unchanged F_stream's range is empty: only the FEB scalars / x_spec spectra can be touched
            if (i_grid != i_grid_old || (ev & (EV_FEB_UP | (0xffffu << EV_XSPEC_SHIFT)))) ev |= EV_VALID;
            else ev = 0;
        }
        // ---- point A (converged): queue the crossing events with the state as it is right after the move ----
        {
            double ec = 1.0, es = 0.0;
            if (ev) sincos_bf(phi, &es, &ec);
            qn = push_events<false>(P, wm, qn, ev, ip, pb, pperp, gam_pf, ec, es, ptot, i_grid, i_grid_old, iz);
        }
        // ---- rest of Code Block 2: downstream escape / return ------------------------------------------------
        bool sum_p = false;
        if (moved && fin < 0) {
            bool went_retro = false, lose_pt = false;
            // downstream_test / prob_return do something only if the particle is beyond a downstream FEB, far beyond
            // the PRP, has just crossed the end of the grid or the PRP, or is a cooling electron (prob_return.jl:155)
            const bool special = (P.feb_dn > 0 && x > P.feb_dn) || (x > 1.1 * prp_x) ||
                                 (x >= P.x_grid_stop && (x_old < P.x_grid_stop || (x_old < prp_x && x >= prp_x) || ELECTRON));
            if (MCS_LIKELY(!special)) {
                i_return = 2;
            } else {
                ColdIO io;
                io.x = x; io.prp_x = prp_x; io.ptot = ptot; io.pb = pb; io.pperp = pperp; io.gam_pf = gam_pf; io.gd = gd;
                io.acct = acct; io.phi = phi; io.retro_steps = 0; io.rng_n = rng.n; io.rng_s2 = rng.s2;
                io.rng_s3 = rng.s3; io.tcut = tcut; io.i_return = i_return; io.exhausted = rng.exhausted;
                const ColdIO o = downstream_block<DEBUG, ELECTRON>(P, io, x_old, grt, P.cur.weight[ip], helix, rng.c1, rng.ru,
                                                                   rng.rn);
                x = o.x; prp_x = o.prp_x; ptot = o.ptot; pb = o.pb; pperp = o.pperp; gam_pf = o.gam_pf; gd = o.gd;
                acct = o.acct; phi = o.phi; if (o.retro_steps) P.retro[ip] += o.retro_steps; rng.n = o.rng_n; rng.s2 = o.rng_s2;
                rng.s3 = o.rng_s3; tcut = o.tcut; i_return = o.i_return; fin = o.fin; went_retro = o.went_retro;
                lose_pt = o.lose_pt; rng.exhausted = o.exhausted;
                if (went_retro && ELECTRON) { inv_ptot = 1 / ptot; inv_gm = 1 / (gam_pf * P.m); }
            }
            if (DEBUG && slot >= 0 && fin < 0) {
                int k = P.trace_cnt[slot];
                if (k < P.trace_max) {
                    McsTraceRec& r = P.trace_recs[(size_t)slot * P.trace_max + k];
                    r.x_cm = x; r.ptot_pf = ptot; r.pb_pf = pb; r.phi_rad = phi; r.acctime_sec = acct;
                    r.prp_x_cm = prp_x; r.i_grid = i_grid; r.helix_count = helix;
                    r.flags = (down ? 1 : 0) | (inj ? 2 : 0) | (went_retro ? 4 : 0) | ((i_return + 1) << 8);
                    r.n_draws = (int)rng.n;
                    P.trace_cnt[slot] = k + 1;
                }
            }
            if (fin < 0 && i_return == 0) { sum_p = true; fin = lose_pt ? 4 : 1; }
            if (DEBUG && fin < 0 && rng.exhausted) fin = MCS_FATE_ERROR;
        }
        if (moved) x_old_le0 = x_old <= 0.0;
        // ---- point B (converged): particles that left the loop ------------------------------------------------
        ev = 0;
        bool release = false;
        if (MCS_UNLIKELY(ip >= 0 && fin >= 0)) {
            if (DEBUG && rng.exhausted) { fin = MCS_FATE_ERROR; sum_p = false; }
            if (fin == 0) {  // particle_loop.jl:361-380
                P.l_save[ip] = 1;
                P.saved.weight[ip] = P.cur.weight[ip]; P.saved.ptot[ip] = ptot; P.saved.pb[ip] = pb; P.saved.x[ip] = x;
                P.saved.grid[ip] = i_grid; P.saved.down[ip] = down; P.saved.inj[ip] = inj;
                P.saved.xn_per[ip] = xsel == 0 ? P.xn_fine : (xsel == 1 ? P.xn_coarse : P.cur.xn_per[ip]);
                P.saved.prp_x[ip] = x < prp_x ? prp_x : x * 1.1;
                P.saved.acctime[ip] = acct; P.saved.phi[ip] = phi; P.saved.tcut[ip] = tcut;
            } else if (fin <= 4) {
                ev = EV_VALID | EV_FINISH | ((uint32_t)fin << EV_REASON_SHIFT) | (sum_p ? EV_SUMP : 0u);
            } else {
                count(P, CNT_ERR);
            }
            P.fate[ip] = fin; P.helix[ip] = helix; P.draws[ip] = rng.n;
            count(P, CNT_FATE0 + fin);
            count(P, CNT_HELIX, (unsigned long long)helix);
            { const long long rs = P.retro[ip]; if (rs) count(P, CNT_RETRO, (unsigned long long)rs); }
            release = true;  // ip is still needed by the event push below (weight is read from the population array)
        }
        {
            double ec = 1.0, es = 0.0;
            if (ev) sincos_bf(phi, &es, &ec);
            qn = push_events<false>(P, wm, qn, ev, ip, pb, pperp, gam_pf, ec, es, ptot, i_grid, i_grid_old, iz);
        }
        if (release) ip = -1;
        // a particle back from retro_time (i_return == 1) takes its follow-up pass here at once
        if (served) parked = !fast_ok || (ip >= 0 && i_return == 1);
    }
    l.rng_n = rng.n; l.rng_s2 = rng.s2; l.rng_s3 = rng.s3; l.rng_c1 = rng.c1; l.rng_ru = rng.ru; l.rng_rn = rng.rn;
    l.rng_exhausted = rng.exhausted;
    Lref = l;
    return all_done;
}

// optional per-pass features, as a compile-time mask of transport_kernel (FEAT)
enum : int { FEAT_AGE = 1, FEAT_TCUTS = 2, FEAT_FEB_DN = 4, FEAT_REFLECT = 8, FEAT_ETF = 16 };

// lane status bits of the fast loop
enum : uint32_t {
    ST_DOWN = 1u, ST_INJ = 2u, ST_XOLDLE0 = 4u, ST_PARKED = 8u, ST_NEEDPSP = 16u, ST_XSEL = 32u, ST_GTPMAX = 64u, ST_GTPCUT = 128u,
    ST_RAN = 256u,   // at least one fast pass committed in this residency (i_return = 2)
    ST_MUSN = 512u,  // mu / sn are newer than the record's pb / pperp
    ST_PHI = 1024u,  // the phase registers are newer than the record's angle (a boost without a committed pass after it)
    ST_ETF = 2048u,  // energy transfer is due before the next pass (particle_loop.jl:235): general pass
    ST_QEMPTY = 4096u,  // this lane found the warp's particle sequence exhausted
};
constexpr double COS_AT_LIMIT = 1.4901161193847656e-08;  // sqrt(1 - prevfloat(1.0)^2): cosine of the phase change at the clamp

// sin and cos of the scattering azimuth phi_s = 2 pi u - pi (scattering.jl:71) for u = w / 2^53, w the 53-bit random
// integer (hi:lo >> 11): the top 8 bits of w pick a table entry {sin A_k, cos A_k}, A_k = -pi + 2 pi (k + 1/2) / 256, the
// other 45 bits the offset |t| <= pi/256 from it, whose sine and cosine need three terms each; angle addition.  12 FP64
// operations and 6 constants instead of 26 and 16 for a general sincos; error <= 2.5 ulp of 1 against the exact azimuth
// (measured 2.45 on B200, tests/test_device_units.py), up to 2.36 of which is the table's: az_table rounds the bin centre to
// double before libm sees it.
__device__ __forceinline__ void az_sincos(const double2* __restrict__ tab, uint32_t hi, uint32_t lo, double& s_out, double& c_out) {
    const uint32_t k = hi >> 24;
    // f = bits 44..0 of w: bits 23..11 of hi (13 bits) above bits 31..11 of lo... as an exact double via the 2^52 trick
    const uint32_t f_hi = (hi >> 11) & 0x1fffu;             // bits 44..32 of f
    const uint32_t f_lo = (lo >> 11) | (hi << 21);          // bits 31..0 of f
    const double f = __hiloint2double((int)(0x43300000u | f_hi), (int)f_lo) - 4503599627370496.0;  // exact: f < 2^45
    const double t = fma(f, 6.975736996017264e-16, -0.01227184630308513);  // 2 pi / 256 / 2^45 * f - pi / 256
    const double z = t * t;
    const double ps = fma(z, 0.008333333333333333, -0.16666666666666666);
    const double st = fma(t * z, ps, t);
    double pc = fma(z, -0.001388888888888889, 0.041666666666666664);
    pc = fma(z, pc, -0.5);
    const double ct = fma(z, pc, 1.0);
    const double2 e = tab[k];
    s_out = fma(e.x, ct, e.y * st);
    c_out = fma(e.y, ct, -(e.x * st));
}
// the table az_sincos reads (DevParams.az_tab), built on the host with its libm
__host__ inline void az_table(double2 tab[AZ_N]) {
    for (int k = 0; k < AZ_N; k++) {
        const double a = -PI + TWO_PI * (k + 0.5) / AZ_N;
        tab[k].x = sin(a); tab[k].y = cos(a);
    }
}

// Base.mod2pi for -2pi < v < 4pi without branches (the general formula with k = -1, 0, 1 and the same roundings);
// ok = false when the result needs the final wrap of the general formula or v is outside that range: the lane parks.
__device__ __forceinline__ double mod2pi_bf(double v, bool& ok) {
    const double kd = v >= TWO_PI ? 1.0 : (v < 0.0 ? -1.0 : 0.0);
    double r = fma(-kd, TWO_PI, v);
    r = fma(-kd, TWO_PI_LO, r);
    ok = (r >= 0.0) & (r < TWO_PI);
    return r;
}

// ---------------------------------------------------------------------------------------------
// The transport kernel.
#ifdef MCS_MAXNREG
#define MCS_KERNEL_BOUNDS __maxnreg__(MCS_MAXNREG)
#else
#define MCS_KERNEL_BOUNDS __launch_bounds__(MCS_BLOCK, MCS_MIN_BLOCKS)
#endif
template <bool DEBUG, bool ELECTRON, bool OBLIQUE, bool SLIM, bool CUSTOM = false, int FEAT = -1>
__global__ void MCS_KERNEL_BOUNDS transport_kernel(const __grid_constant__ DevParams P) {
    extern __shared__ __align__(16) unsigned char mcs_smem[];
    const int ng = P.n_grid;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
    {   // zone table of the fast loop
        double2* za = reinterpret_cast<double2*>(mcs_smem);
        double2 *zb = za + (ng + 2), *zc = zb + (ng + 2);
        double* zd = reinterpret_cast<double*>(zc + (ng + 2));
        for (int i = threadIdx.x; i < ng + 2; i += blockDim.x) {
            za[i] = make_double2(P.ux[i], P.gsf[i]);
            zb[i] = make_double2(P.gef[i], P.costh[i]);
            zc[i] = make_double2(P.xg[i], i <= ng ? P.xg[i + 1] : __longlong_as_double(0x7ff0000000000000ll));
            zd[i] = 1 / (P.zz * P.bt[i]);
        }
        double2* az = reinterpret_cast<double2*>(mcs_smem + zone_tab_bytes(ng) - (size_t)AZ_N * 16);
        for (int i = threadIdx.x; i < AZ_N; i += blockDim.x) az[i] = P.az_tab[i];
    }
    const WarpMem wm = warp_mem(warp, ng);
    for (int i = lane; i < 3 * ng + SC_N; i += 32) wm.part[i] = 0.0;
    __syncthreads();
    const ZoneTab zt = zone_tab(ng);

    const uint32_t flags = P.flags;
    // the fast loop covers scattering configurations without per-pass field updates, detectors or debug streams
    // custom eps_B (field beyond the end of the grid falls off as sqrt(x_grid_stop / x): per-pass gyro-period) is a compile-time
    // variant of the fast loop: as a launch-uniform branch it cost the plain kernel 6 % (temporaries kept live, larger loop)
    const bool fast_ok = !DEBUG && !(flags & (F_DONT_SCATTER | F_NO_FAST_LOOP)) && P.n_xspec == 0 && (CUSTOM || !(flags & F_CUSTOM_EPSB));
    constexpr bool custom_cfg = CUSTOM;
    const bool rad_fast = ELECTRON && (flags & F_RAD_LOSSES);  // the fast loop applies radiation_loss itself, pass by pass
    const double inv_mc = 1 / P.mc;
    // FEAT >= 0: the host tells at compile time which optional features of a pass are switched on (FEAT_* bits: age limit,
    // tcut tracking, downstream FEB, reflection for no-DSA / partial injection, energy transfer) and the loop does not test
    // for the others.  As launch-uniform branches those five tests cost the plain configs 7-9 % (profiles/r02_variants.md).
    // FEAT < 0: the generic build, every feature decided at run time.
    constexpr bool known = FEAT >= 0;
    const bool reflect_cfg = known ? (FEAT & FEAT_REFLECT) != 0 : ((flags & F_DONT_DSA) || P.inj_frac < 1);
    const bool age_on = known ? (FEAT & FEAT_AGE) != 0 : P.age_max > 0, tcuts_on = known ? (FEAT & FEAT_TCUTS) != 0 : (flags & F_TCUTS) != 0,
               feb_dn_on = known ? (FEAT & FEAT_FEB_DN) != 0 : P.feb_dn > 0, etf_on = known ? (FEAT & FEAT_ETF) != 0 : P.energy_transfer_frac > 0;

    Lane L;
    L.ptot = 1; L.pb = 0; L.pperp = 0; L.x = 0; L.prp_x = 0; L.acct = 0; L.phi = 0;
    L.gam_pf = 1; L.gd = 0; L.grt = 0; L.gr = 0; L.gper = 0; L.t_step = 0; L.inv_ptot = 1; L.inv_gm = 1;
    L.ux = 0; L.gsf = 1; L.gef = 1; L.bsin = 0; L.bcos = 1;
    L.rng_ru = nullptr; L.rng_rn = 0;
    L.ip = -1; L.next_j = 0; L.iz = 0; L.i_grid = 0; L.i_grid_old = 0; L.helix = 0; L.tcut = 1; L.i_return = -1; L.xsel = 0;
    L.slot = -1; L.qn = 0;
    L.rng_n = 0; L.rng_s2 = 0; L.rng_s3 = 0; L.rng_c1 = 0;
    L.rng_exhausted = false; L.queue_empty = false; L.down = false; L.inj = false; L.x_old_le0 = true; L.parked = true;
    L.mu = 0; L.sn = 1; L.cph = 1; L.sph = 0; L.cs_valid = false; L.cs_flags = 0u;
#ifdef MCS_SCHED_COUNTERS
    unsigned long long c_fast_lane = 0, c_fast_iter = 0, c_sections = 0, c_wait = 0, c_idle = 0, c_psp = 0;
#define MCS_SC(x) x
#else
#define MCS_SC(x)
#endif

    for (;;) {
        MCS_SC(c_sections++;)
        if (general_section<DEBUG, ELECTRON>(P, L, fast_ok)) break;
        if constexpr (!DEBUG) {
            // ---- FAST LOOP -------------------------------------------------------------------------------------
            // Passes in which nothing rare happens (scatter, move, zone search, zone change without a boost, shock
            // crossing, PRP placement, the crossing event).  A lane that meets anything else commits nothing and PARKS;
            // when enough lanes wait, the warp leaves for the general section.  Per particle the sequence of operations
            // is the one of particle_loop.jl.  Register state: position, pitch (mu, sn = pb, pperp over ptot), phase,
            // clock, PRP, and three per-momentum constants; zone constants come from the shared zone table.
            int ip;
            double x, acct, prp_x, grt, t_step, mu, sn, vgm, gper;
            double cph, sph;  // gyro-phase as (cos, sin): the kick and the advance are rotations, no asin / mod2pi per pass
            int iz, helix;
            uint32_t gpack, rng_n, rng_s2, rng_s3, rng_c1;
            // status word; ST_GTPMAX / ST_GTPCUT / ST_ETF = "the general pass must see this particle before its next pass"
            // for the reasons that only change at a boost, a shock crossing or a zone change
            uint32_t st;
            // registers <- record (at entry, and for a lane refilled inside the loop)
#define MCS_LOAD_LANE()                                                                                                     \
    do {                                                                                                                    \
        ip = L.ip;                                                                                                          \
        x = L.x; acct = L.acct; prp_x = L.prp_x; grt = L.grt; t_step = L.t_step;                                            \
        vgm = L.ptot * L.inv_gm;                                                                                            \
        gper = (ELECTRON && L.ptot < P.pe_crit) ? TWO_PI * P.gam_e_crit * P.mc * L.gd : TWO_PI * L.gam_pf * P.mc * L.gd;    \
        if (L.cs_valid) { mu = L.mu; sn = L.sn; cph = L.cph; sph = L.sph; }                                                 \
        else { mu = L.pb * L.inv_ptot; sn = L.pperp * L.inv_ptot; sincos(L.phi, &sph, &cph); }                              \
        iz = L.iz; helix = L.helix;                                                                                         \
        gpack = (uint32_t)L.i_grid | ((uint32_t)L.i_grid_old << 16);                                                        \
        rng_n = L.rng_n; rng_s2 = L.rng_s2; rng_s3 = L.rng_s3; rng_c1 = L.rng_c1;                                           \
        st = (L.down ? ST_DOWN : 0u) | (L.inj ? ST_INJ : 0u) | (L.x_old_le0 ? ST_XOLDLE0 : 0u) | (L.xsel ? ST_XSEL : 0u) |  \
             (L.ptot > P.pmax_cutoff ? ST_GTPMAX : 0u) | (L.ptot > P.pcut ? ST_GTPCUT : 0u) | (L.queue_empty ? ST_QEMPTY : 0u) | \
             ((L.ip >= 0 && L.parked) ? ST_PARKED : 0u) | (L.cs_valid ? L.cs_flags : 0u);                                   \
        if (etf_on && !L.inj && L.x_old_le0 && L.i_grid_old != L.i_grid) st |= ST_ETF;                                      \
    } while (0)
            MCS_LOAD_LANE();
            int qn = L.qn;
#ifdef MCS_PREFETCH
            uint32_t q0, q1, q2, q3;
            philox4x32_10_rk((rng_n + (rng_n & 1u)) >> 1, rng_c1, P.ctr2, P.ctr3, P.rk, q0, q1, q2, q3);
#endif
            int n_act = __popc(__ballot_sync(FULL, ip >= 0));
            int park_t = min(MCS_PARK_T, (3 * n_act + 3) >> 2);
            int psp_debt = 0, wait_debt = 0;
            for (int it = 0; it < MCS_FAST_MAX; it++) {
                uint32_t fev = 0;   // crossing event produced by this pass
                int ev_old = 0;     // its zone before the move
                if (ip >= 0 && !(st & (ST_PARKED | ST_NEEDPSP))) {
                    const int ig = (int)(gpack & 0xffffu);
                    // what the general pass must see before this pass: helix cap, a momentum above a cut-off (saved when
                    // downstream), pending energy transfer, age
                    bool park = (helix >= P.helix_cap) || (st & (ST_GTPMAX | ST_ETF));
                    if (age_on) park = park || acct > P.age_max;
                    // downstream and above this pcut: the particle is saved by its next pass (particle_loop.jl:361-380): general pass.
                    // (Saving and refilling inside this loop was tried — MCS_TAIL, profiles/r02_variants.md — and lost 8 %:
                    // the extra vote per iteration and the larger loop cost more than the idle lanes it removed.)
                    park = park || ((st & (ST_DOWN | ST_GTPCUT)) == (ST_DOWN | ST_GTPCUT));
                    if (ig != iz && !park) {
                        // Code Block 3 zone change (particle_loop.jl:186-228): without a change of flow speed only the
                        // zone's constants change; with one, the momentum must be boosted (batched below)
                        if (zt.a[ig].x != zt.a[iz].x) st |= ST_NEEDPSP;
                        else {
                            const double gd_n = zt.gd[ig];
                            if (gd_n != zt.gd[iz])
                                gper = (ELECTRON && L.ptot < P.pe_crit) ? TWO_PI * P.gam_e_crit * P.mc * gd_n : TWO_PI * L.gam_pf * P.mc * gd_n;
                            iz = ig;
                        }
                    }
                    if (!(st & ST_NEEDPSP) && !park) {
                        // scattering.jl:29-101, same kick as the general pass.  Differences in form only: the azimuth's
                        // sine and cosine come from the table; sqrt(w) is w * rsqrt(w) and the three of them overlap
                        // (sin_new and the pair (sv, cv) = (sin, cos) of the phase change asin(sv) share one reciprocal
                        // square root of sn2); the phase change is applied as a rotation.
                        // Electrons with radiative losses (particle_loop.jl:578-592, applied where the general pass applies it:
                        // over the PREVIOUS pass's time step, after the zone change, before the kick).  The momentum and what
                        // hangs on it — Lorentz factor, gyro-radius, gyro-period, speed — become per-pass quantities; mu and sn
                        // do not change (pb and pperp shrink by the same factor).  Held in temporaries until the pass commits.
                        double p_use = 0.0, gam_use = 0.0, grt_u = grt, vgm_u = vgm, gper_u = gper;
                        bool lost_all = false;
                        if ((ELECTRON && rad_fast) || custom_cfg) {
                            // the field of this pass as the general pass takes it (particle_loop.jl:239-247): the zone's, or with
                            // custom eps_B beyond the end of the grid the last zone's falling off as sqrt(x_grid_stop / x)
                            const bool off_grid = custom_cfg && x > P.x_grid_stop;
                            const double bmag = off_grid ? P.bt[ng] * sqrt(P.x_grid_stop / x) : P.bt[iz];
                            const double gd_z = off_grid ? 1 / (P.zz * bmag) : zt.gd[iz];
                            if (ELECTRON && rad_fast) {
                                const double Bcmb = P.B_CMBz * zt.b[iz].x;
                                p_use = radiation_loss(P, bmag * bmag + Bcmb * Bcmb, L.ptot, t_step);
                                lost_all = !(p_use > 0.0);                           // fate 4: the general pass ends it
                                // gamma = sqrt(1 + (p/mc)^2) directly: p/mc is O(1e-2 .. 1e2) for an electron that still loses
                                // momentum, no overflow to guard against (library hypot was 14 % of this kernel's instructions)
                                const double r_mc = p_use * inv_mc;
                                gam_use = sqrt(fma(r_mc, r_mc, 1.0));
                                grt_u = p_use * P.c * gd_z;
                                vgm_u = p_use * (1 / (gam_use * P.m));
                            } else {
                                p_use = L.ptot; gam_use = L.gam_pf;
                            }
                            gper_u = (ELECTRON && p_use < P.pe_crit) ? TWO_PI * P.gam_e_crit * P.mc * gd_z : TWO_PI * gam_use * P.mc * gd_z;
                        } else if (ELECTRON) {
                            p_use = L.ptot; gam_use = L.gam_pf;
                        }
                        const bool xs_n = x > grt_u;                                 // particle_loop.jl:385, decided first
                        const int xi = xs_n ? 1 : 0;
                        const double t_n = gper_u * P.inv_xn[xi];
                        const double cd = P.cdphi[xi], sd = P.sdphi[xi];
                        const double omc = P.omc[(st & ST_XSEL) ? 1 : 0];
                        const uint32_t odd = rng_n & 1u;
#ifndef MCS_PREFETCH
                        uint32_t q0, q1, q2, q3;
                        philox4x32_10_rk((rng_n + odd) >> 1, rng_c1, P.ctr2, P.ctr3, P.rk, q0, q1, q2, q3);
#endif
                        const double u1 = odd ? u53(rng_s3, rng_s2) : u53(q1, q0);
                        double sps, cps;
                        az_sincos(zt.az, odd ? q1 : q3, odd ? q0 : q2, sps, cps);
                        const uint32_t l2 = q2, l3 = q3;                             // left over for an odd-aligned successor
#ifdef MCS_PREFETCH
                        philox4x32_10_rk(((rng_n + odd) >> 1) + 1u, rng_c1, P.ctr2, P.ctr3, P.rk, q0, q1, q2, q3);
#endif
                        const double cos_d = 1 - u1 * omc;
                        const double sd2 = 1 - cos_d * cos_d;
                        const double sin_d = sd2 * rsqrt_nr(sd2);                    // NaN for sd2 == 0: parks below
                        const double cos_new = mu * cos_d + sn * sin_d * cps;
                        const double sn2 = 1 - cos_new * cos_new;
                        const double a = sps * sin_d;
                        const double r = rsqrt_nr(sn2);
                        const double w2 = sn2 - a * a;
                        const double r2 = rsqrt_nr(w2);
                        const double sin_new = sn2 * r;
                        double sv = a * r;
                        double cv = (w2 * r2) * r;                                   // sqrt(1 - sv^2) = sqrt(sn2 - a^2) / sin_new
                        if (fabs(sv) > SIN_UPPER_LIMIT) sv = copysign(SIN_UPPER_LIMIT, sv);
                        cv = cv > COS_AT_LIMIT ? cv : COS_AT_LIMIT;                  // also catches the NaN of w2 <= 0 at the clamp
                        const double c1 = cph * cv - sph * sv, s1 = sph * cv + cph * sv;
                        // Code Block 2 move
                        const double cph_n = c1 * cd - s1 * sd, sph_n = s1 * cd + c1 * sd;
                        const double2 za = zt.a[iz], zb = zt.b[iz], zc = zt.c[iz];  // {ux, gsf} {gef, cos th} {xg[iz], xg[iz+1]}
                        const double x_move = (cos_new * vgm_u) * t_n;
                        double gyr = 0.0;
                        if (OBLIQUE) {
                            const double bsin = P.sinth[iz];
                            if (bsin != 0.0) gyr = L.gr * bsin * (cph_n - c1);
                        }
                        const double x_n = x + za.y * (x_move * zb.y - gyr + za.x * t_n);
                        double acct_n = acct;
                        if (st & ST_DOWN) {
                            acct_n = acct + t_step * zb.x;
                            if (tcuts_on) park = L.tcut <= P.n_tcuts && acct_n >= P.tcuts[L.tcut - 1];
                        }
                        // Is this a plain pass?  Same zone, and inside the grid or between its end and the PRP.
                        const bool dn = x_n > x;
                        const bool same = dn ? (zc.y > x_n) : (zc.x <= x_n);
                        // `other`: anything but a zone change inside the grid (also a NaN position: !(NaN < stop))
                        const bool beyond = !(x_n < P.x_grid_stop);
                        bool other = !(sn2 > 0.0) | park | (beyond & ((x < P.x_grid_stop) | !(x_n < prp_x) | ELECTRON));
                        if (ELECTRON) other |= lost_all;
                        if (st & ST_INJ) other |= x_n < P.feb_up;
                        if (feb_dn_on) other |= x_n > P.feb_dn;
                        if (reflect_cfg) other |= (x_n <= 0) & (x > 0);
                        int ig_new = iz;
                        double prp_n = prp_x;
                        uint32_t st_n = st;
                        bool go = true;
                        if (other | !same) {
                            // Runs in every other iteration of a warp (one lane or two): most often a zone boundary crossed
                            // inside the grid and nothing else, so everything else nests under `other`.
                            bool pk = false;
                            const bool cross_down = x < 0 && x_n >= 0;
                            if (cross_down) {  // particle_loop.jl:413-429: arrival downstream, make the region long enough
                                const double Ld = ELECTRON ? P.eta_mfp / 3 * grt_u * p_use / (P.m * gam_use * P.u2)
                                                           : P.eta_mfp / 3 * grt * L.ptot / (P.m * L.gam_pf * P.u2);
                                prp_n = fmax(prp_x, Ld);
                            }
                            if (other) {
                            // anything the general pass would have to act on after the move -> nothing is committed
                            pk = park | !(sn2 > 0.0) | !(x_n == x_n) | (reflect_cfg && x_n <= 0 && x > 0 && !(st & ST_INJ)) |
                                 (feb_dn_on && x_n > P.feb_dn) | (ELECTRON && lost_all);
                            // (not `other`: x_n < x_grid_stop <= prp_x, or x_grid_stop <= x, x_n < prp_x — neither test below fires)
                            if (x_n > 1.1 * prp_n) {
                                // downstream_test (particle_loop.jl:609-633): far beyond the PRP -> escapes beyond 6.91 L_diff
                                double v_fac;
                                if (ELECTRON && p_use < P.pe_crit) v_fac = (P.pe_crit * P.c * zt.gd[iz]) * P.pe_crit / (P.m * P.gam_e_crit * P.u2);
                                else if (ELECTRON) v_fac = grt_u * p_use / (P.m * gam_use * P.u2);
                                else v_fac = grt * L.ptot / (P.m * L.gam_pf * P.u2);
                                pk |= x_n > 6.91 * (P.eta_mfp / 3 * v_fac);
                            }
                            if (x_n >= P.x_grid_stop) {
                                if (x < P.x_grid_stop) {
                                    // prob_return.jl:59-84: just crossed the end of the grid -> place the PRP
                                    const double p_g = ELECTRON ? p_use : L.ptot, gam_g = ELECTRON ? gam_use : L.gam_pf;
                                    const double gyro_tmp = (custom_cfg && x_n > P.x_grid_stop) ? sqrt(P.x_grid_stop / x_n) : 1.0;
                                    const double g2 = p_g * P.c * gyro_tmp / (P.qcgs * P.bmag2);
                                    prp_n = x_n + 3 * (P.eta_mfp / 3 * g2 * p_g / (P.aa * P.mp * gam_g * P.u2));
                                } else {
                                    pk |= (x < prp_n && x_n >= prp_n) | ELECTRON;  // PRP crossing: probability-of-return test
                                }
                            }
                            }
                            if (!pk) {
                                // zone search (all_flux.jl:65-82) and the crossing event
                                if (!same) {
                                    // on the shared table {xg[j], xg[j+1]}, starting at the neighbour (the own zone is excluded)
                                    if (dn) { int j = iz + 1; while (j <= ng && !(zt.c[j].y > x_n)) j++; ig_new = j; }
                                    else { int j = iz - 1; while (j >= 0 && !(zt.c[j].x <= x_n)) j--; ig_new = j; }
                                }
                                if (cross_down) st_n |= ST_DOWN;
                                if ((st_n & ST_DOWN) && x_n < 0) st_n |= ST_INJ;  // particle_loop.jl:433-435 (before all_flux)
                                const bool below_feb = (st_n & ST_INJ) && x_n < P.feb_up;
                                const bool feb_x = below_feb && x >= P.feb_up;
                                if (ig_new != iz || (feb_x && ig_new <= P.i_grid_feb))
                                    fev = EV_VALID | ((st_n & ST_INJ) ? EV_INJ : 0u) | (dn ? 0u : EV_UP) | (feb_x ? EV_FEB_UP : 0u);
                                if (below_feb) st_n |= ST_PARKED;  // the next pass ends at the upstream FEB: general pass
                                // energy transfer is due at the next pass of a not yet injected particle that changed zone
                                // coming from x <= 0 (particle_loop.jl:235)
                                if (etf_on && !(st_n & ST_INJ) && x <= 0.0 && ig_new != iz) st_n |= ST_ETF;
                            }
                            go = !pk;
                        }
                        if (go) {
                            ev_old = iz;
                            st = (st_n & ~(ST_XOLDLE0 | ST_XSEL | ST_PHI)) | (x <= 0.0 ? ST_XOLDLE0 : 0u) | (xs_n ? ST_XSEL : 0u) | ST_RAN | ST_MUSN;
                            prp_x = prp_n;
                            helix++; MCS_SC(c_fast_lane++;)
                            acct = acct_n; t_step = t_n;
                            if (ELECTRON && rad_fast) {  // the loss of this pass becomes the particle's momentum
                                grt = grt_u; vgm = vgm_u; gper = gper_u;
                                L.ptot = p_use; L.gam_pf = gam_use; L.grt = grt_u;  // (the reciprocals of the record: at exit)
                            }
                            mu = cos_new; sn = sin_new; cph = cph_n; sph = sph_n; x = x_n;
                            gpack = (uint32_t)ig_new | ((uint32_t)iz << 16);
                            rng_n += 2; rng_s2 = l2; rng_s3 = l3;
                        } else if (ip >= 0) {
                            st |= ST_PARKED;  // (a prefetched block is stale now; it is rebuilt when the lane re-enters the loop)
                        }
                    } else if (park) {
                        st |= ST_PARKED;
                    }
                }
                // converged: queue the crossing events of this pass (state right after the move, as at point A)
                if (__any_sync(FULL, fev != 0u))
                    qn = push_events<true, SLIM>(P, wm, qn, fev, ip, L.ptot * mu, L.ptot * sn, L.gam_pf, cph, sph, L.ptot, (int)(gpack & 0xffffu), ev_old,
                                     ev_old);
                // leave the loop?  Enough lanes wait for the general pass, or few have waited long (short trajectories: many
                // refills), or the bound on consecutive iterations is reached
                MCS_SC(c_fast_iter++;)
                const int n_wait = __popc(__ballot_sync(FULL, ip >= 0 && (st & ST_PARKED)));
                MCS_SC(c_wait += n_wait; c_idle += __popc(__ballot_sync(FULL, ip < 0)); c_psp += __popc(__ballot_sync(FULL, (st & ST_NEEDPSP) != 0u));)
                wait_debt += n_wait;
                const bool leaving = (n_wait > 0 && n_wait >= park_t) || (MCS_WAIT_DEBT > 0 && wait_debt >= MCS_WAIT_DEBT) ||
                                     it == MCS_FAST_MAX - 1;
                {   // converged: pending boosts.  Waiting costs idle lanes, serving costs the whole warp ~250 issue slots:
                    // serve once the lanes have waited MCS_PSP_DEBT lane-iterations in total, or when fewer lanes run
                    // than wait — and always before leaving: a boost asked for in this loop is done by this loop, so WHICH
                    // of the two (mathematically equal) boost routines a particle meets never depends on its warp mates.
                    const unsigned mp = __ballot_sync(FULL, (st & ST_NEEDPSP) != 0u);
                    if (mp) {
                        const int n_psp = __popc(mp);
                        const int n_run = __popc(__ballot_sync(FULL, ip >= 0 && !(st & (ST_PARKED | ST_NEEDPSP))));
                        psp_debt += n_psp;
                        if (leaving || psp_debt >= MCS_PSP_DEBT || MCS_PSP_NUM * n_psp >= n_run) {
                            psp_debt = 0;
                            if (st & ST_NEEDPSP) {
                                st &= ~ST_NEEDPSP;
                                const int iz_old = iz;
                                iz = (int)(gpack & 0xffffu);
                                const double gd = zt.gd[iz];
                                MomCS mi;
                                mi.ptot = L.ptot; mi.gam_pf = L.gam_pf; mi.cphi = cph; mi.sphi = sph;
                                mi.pb = (st & ST_MUSN) ? L.ptot * mu : L.pb;
                                mi.pperp = (st & ST_MUSN) ? L.ptot * sn : L.pperp;
                                const MomCS mo = transform_p_PSP_cs(P, iz_old, iz, mi);
                                cph = mo.cphi; sph = mo.sphi;
                                L.ptot = mo.ptot; L.pb = mo.pb; L.pperp = mo.pperp; L.gam_pf = mo.gam_pf; L.gd = gd;
                                L.gr = mo.pperp * P.c * gd;
                                grt = mo.ptot * P.c * gd;
                                L.grt = grt;
                                const double inv_ptot = 1 / mo.ptot, inv_gm = 1 / (mo.gam_pf * P.m);
                                L.inv_ptot = inv_ptot; L.inv_gm = inv_gm;
                                mu = mo.pb * inv_ptot; sn = mo.pperp * inv_ptot;
                                vgm = mo.ptot * inv_gm;
                                gper = (ELECTRON && mo.ptot < P.pe_crit) ? TWO_PI * P.gam_e_crit * P.mc * gd : TWO_PI * mo.gam_pf * P.mc * gd;
                                // the boosted momentum may now exceed a cut-off: the pre-test of the next pass parks the lane
                                st = (st & ~(ST_MUSN | ST_GTPMAX | ST_GTPCUT)) | ST_PHI | (mo.ptot > P.pmax_cutoff ? ST_GTPMAX : 0u) |
                                     (mo.ptot > P.pcut ? ST_GTPCUT : 0u);
                            }
                        }
                    }
                }
                if (leaving) break;
            }
            // ---- back to the record ----
            L.ip = ip;
            if (st & ST_QEMPTY) L.queue_empty = true;
            if (ip >= 0) {
                L.x = x; L.acct = acct; L.prp_x = prp_x; L.t_step = t_step; L.gper = gper;
                if (st & (ST_PARKED | ST_NEEDPSP)) {
                    // the general pass takes this particle next: give it the record in the reference's terms
                    if (st & ST_PHI) {  // last touched by a boost: atan(...) - pi/2 lies in (-3 pi/2, pi/2] (transformers.jl:603-604)
                        double a = atan2(sph, cph);
                        if (a > HALF_PI) a -= TWO_PI;
                        L.phi = a;
                    } else if (st & ST_RAN) {  // last touched by a move: Base.mod2pi leaves it in [0, 2 pi)
                        double a = atan2(sph, cph);
                        if (a < 0.0) a += TWO_PI;
                        L.phi = a;
                    }
                    if (st & ST_MUSN) { L.pb = L.ptot * mu; L.pperp = L.ptot * sn; }
                    if (ELECTRON && rad_fast) L.gr = L.pperp * P.c * L.gd;
                    L.cs_valid = false;
                } else {
                    // the warp left because of other lanes: this one comes back with exactly these registers
                    L.mu = mu; L.sn = sn; L.cph = cph; L.sph = sph;
                    L.cs_valid = true; L.cs_flags = st & (ST_RAN | ST_MUSN | ST_PHI);
                }
                if (ELECTRON && rad_fast) { L.inv_ptot = 1 / L.ptot; L.inv_gm = 1 / (L.gam_pf * P.m); }  // not kept up to date per pass
                if (st & ST_RAN) L.i_return = 2;
                L.helix = helix;
                L.i_grid = (int)(gpack & 0xffffu); L.i_grid_old = (int)(gpack >> 16);
                if (iz != L.iz) {  // the general pass expects the constants of the zone in effect
                    L.iz = iz;
                    L.ux = P.ux[iz]; L.gsf = P.gsf[iz]; L.gef = P.gef[iz]; L.bsin = P.sinth[iz]; L.bcos = P.costh[iz];
                    L.gd = zt.gd[iz];
                }
                L.xsel = (st & ST_XSEL) ? 1 : 0;
                L.down = st & ST_DOWN; L.inj = st & ST_INJ; L.x_old_le0 = st & ST_XOLDLE0;
                L.parked = (st & (ST_PARKED | ST_NEEDPSP)) != 0u;  // a boost still pending: the general pass does the zone change
                L.rng_n = rng_n; L.rng_s2 = rng_s2; L.rng_s3 = rng_s3;
            }
            L.qn = qn;
        }
    }
    __syncwarp();
    if (L.qn > 0) process_events_ool(P, 0, L.qn);

    MCS_SC(count(P, CNT_FAST_LANE, c_fast_lane);
           if (lane == 0) { count(P, CNT_FAST_ITER, c_fast_iter); count(P, CNT_SLOW_SEC, c_sections);
                            count(P, CNT_PARK0, c_wait); count(P, CNT_PARK0 + 1, c_idle); count(P, CNT_PARK0 + 2, c_psp); })
    // ---- block partials -------------------------------------------------------------------------------
    __syncthreads();
    const int np = 3 * ng + SC_N;
    double* part = P.t.block_partials + (size_t)blockIdx.x * (size_t)np;
    for (int i = threadIdx.x; i < np; i += blockDim.x) {
        double s = 0.0;
        for (int w = 0; w < n_warps; w++) s += warp_mem(w, ng).part[i];  // fixed warp order
        part[i] = s;
    }
}

// Sum the per-block partials in block order (run-to-run deterministic) into the ion totals.
__global__ void reduce_partials_kernel(const double* __restrict__ partials, int n_blocks, int ng, double* pxx,
                                       double* pxz, double* efl, double* scalars) {
    const int np = 3 * ng + SC_N;
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= np) return;
    double s = 0.0;
    for (int b = 0; b < n_blocks; b++) s += partials[(size_t)b * np + i];
    double* dst = i < ng ? pxx + i : (i < 2 * ng ? pxz + (i - ng) : (i < 3 * ng ? efl + (i - 2 * ng) : scalars + (i - 3 * ng)));
    *dst += s;
}

// ---------------------------------------------------------------------------------------------
// new_pcut (cuts.jl:34-98) on device: order-preserving compaction of l_save, then i_mult clones each.
// COMPACT_TPB is the block size of all three compaction kernels (enqueue_compaction): one block count per COMPACT_TPB
// particles, and the scan walks the counts in tiles of COMPACT_TPB.
constexpr int COMPACT_TPB = 1024;
__global__ void count_saved_kernel(const uint8_t* __restrict__ l_save, long long n, int* block_counts) {
    __shared__ int sh[32];
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    int v = (i < n && l_save[i]) ? 1 : 0;
    unsigned b = __ballot_sync(0xffffffffu, v);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = __popc(b);
    __syncthreads();
    if (threadIdx.x < 32) {
        int s = threadIdx.x < (blockDim.x >> 5) ? sh[threadIdx.x] : 0;
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (threadIdx.x == 0) block_counts[blockIdx.x] = s;
    }
}

// single block: exclusive scan of block_counts (n_blocks entries) into block_offsets; total -> *total
__global__ void scan_blocks_kernel(const int* __restrict__ counts, int n_blocks, long long* offsets, long long* total) {
    __shared__ long long sh[COMPACT_TPB];
    __shared__ long long carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (int base = 0; base < n_blocks; base += blockDim.x) {
        int i = base + threadIdx.x;
        long long v = i < n_blocks ? counts[i] : 0;
        sh[threadIdx.x] = v;
        __syncthreads();
        for (int o = 1; o < blockDim.x; o <<= 1) {
            long long t = threadIdx.x >= o ? sh[threadIdx.x - o] : 0;
            __syncthreads();
            sh[threadIdx.x] += t;
            __syncthreads();
        }
        if (i < n_blocks) offsets[i] = carry + sh[threadIdx.x] - v;
        __syncthreads();
        if (threadIdx.x == 0) carry += sh[blockDim.x - 1];
        __syncthreads();
    }
    if (threadIdx.x == 0) *total = carry;
}

__global__ void compact_saved_kernel(const uint8_t* __restrict__ l_save, long long n, const long long* __restrict__ offsets,
                                     long long* saved_idx) {
    __shared__ int sh[32];
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    int v = (i < n && l_save[i]) ? 1 : 0;
    unsigned b = __ballot_sync(0xffffffffu, v);
    int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    if (lane == 0) sh[w] = __popc(b);
    __syncthreads();
    int before = 0;
    for (int k = 0; k < w; k++) before += sh[k];
    if (v) saved_idx[offsets[blockIdx.x] + before + __popc(b & ((1u << lane) - 1u))] = i;
}

// entries of the block_cnt / block_off buffers that enqueue_compaction needs for n particles
__host__ inline long long compaction_blocks(long long n) { return (n + COMPACT_TPB - 1) / COMPACT_TPB; }

// The order-preserving compaction, enqueued on `stream` (n >= 1): saved_idx[0..*total) = the indices i < n with l_save[i]
// set, in increasing order.  compact_saved_kernel reads offsets[blockIdx.x] under count_saved_kernel's block size, and the
// scan's shared array holds one tile of COMPACT_TPB counts, so these launch shapes are fixed here and nowhere else.
// Launch errors are left for the caller's cudaGetLastError.
__host__ inline void enqueue_compaction(const uint8_t* l_save, long long n, int* block_cnt, long long* block_off,
                                        long long* total, long long* saved_idx, cudaStream_t stream) {
    const int nb = (int)compaction_blocks(n);
    count_saved_kernel<<<nb, COMPACT_TPB, 0, stream>>>(l_save, n, block_cnt);
    scan_blocks_kernel<<<1, COMPACT_TPB, 0, stream>>>(block_cnt, nb, block_off, total);
    compact_saved_kernel<<<nb, COMPACT_TPB, 0, stream>>>(l_save, n, block_off, saved_idx);
}

// per-pcut exchange record of one rank, filled on the device so that the all-gather needs no host round trip first
__global__ void pack_counts_kernel(const unsigned long long* __restrict__ counters, unsigned long long saved0, long long n_use,
                                   long long err, long long* out) {
    out[0] = (long long)(counters[CNT_FATE0] - saved0);
    out[1] = n_use; out[2] = err; out[3] = 0;
}

// record o of dst = record j of src, the weight divided by i_mult (cuts.jl:77; exact for i_mult = 1)
__device__ __forceinline__ void copy_record(const PopPtrs& dst, long long o, const PopPtrs& src, long long j, long long i_mult) {
#define X(T, name, pub) T name = src.name[j];
    MCS_POP_FIELDS(X)
#undef X
    weight /= (double)i_mult;
#define X(T, name, pub) dst.name[o] = name;
    MCS_POP_FIELDS(X)
#undef X
}

// child o of the split = copy of saved record saved_idx[o / i_mult]
__global__ void clone_kernel(PopPtrs src, PopPtrs dst, const long long* __restrict__ saved_idx, long long n_out,
                             long long i_mult) {
    long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= n_out) return;
    copy_record(dst, o, src, saved_idx[o / i_mult], i_mult);
}

// Multi-GPU split with rebalancing: every rank packs its saved records into its block of an exchange buffer; block q is
// pop_view(buf + q * stride * POP_REC_BYTES, stride, 0).  After ncclAllGather each rank clones an equal contiguous slice of
// the GLOBAL child index range.
struct GatherPrefix { long long start[65]; int nranks; };

// record r of a rank's exchange block (`stride` records) = its saved record saved_idx[r], r < ns
__global__ void pack_saved_kernel(PopPtrs src, const long long* __restrict__ saved_idx, long long ns, unsigned char* block,
                                  long long stride) {
    long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= ns) return;
    copy_record(pop_view(block, stride, 0), r, src, saved_idx[r], 1);
}

__global__ void clone_gathered_kernel(unsigned char* buf, long long stride, GatherPrefix pre, PopPtrs dst, long long c0,
                                      long long n_out, long long i_mult) {
    long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= n_out) return;
    const long long sidx = (c0 + o) / i_mult;  // global rank of the saved parent (cuts.jl:69-91 order)
    int q = 0;
    while (q + 1 < pre.nranks && sidx >= pre.start[q + 1]) q++;
    copy_record(dst, o, pop_view(buf + (size_t)q * (size_t)stride * POP_REC_BYTES, stride, 0), sidx - pre.start[q], i_mult);
}

// Host plan of the rebalancing split for one rank, from every rank's saved count ns_all[0..nranks): the prefix of the
// gathered blocks, S saved in all, i_mult = max(target / S, 1) (cuts.jl:42 on the global count), C = S * i_mult children,
// this rank's slice [c0, c1) = [C r / N, C (r + 1) / N) and the gather stride (the largest ns rounded up to 16 records).
// Every rank computes the same plan but its slice, so all refuse together.  `pre` and S are filled on every path.
struct SplitPlan {
    GatherPrefix pre;
    long long S, i_mult, C, c0, c1, stride;
};
enum SplitPlanError {
    SPLIT_PLAN_OK = 0,
    SPLIT_PLAN_BAD_RANKS,      // nranks outside 1..64 or rank outside 0..nranks-1
    SPLIT_PLAN_NONE_SAVED,     // S == 0: nothing to split
    SPLIT_PLAN_OVER_CAPACITY,  // the largest slice exceeds n_pts_max
    SPLIT_PLAN_OVER_RANGE,     // C > 2^32: a child's global index would leave the RNG counter range
};
__host__ inline int split_plan(const long long* ns_all, int nranks, int rank, long long target, long long n_pts_max,
                               SplitPlan* p) {
    memset(p, 0, sizeof *p);
    if (nranks < 1 || nranks > 64 || rank < 0 || rank >= nranks) return SPLIT_PLAN_BAD_RANKS;
    p->pre.nranks = nranks;
    long long S = 0, max_ns = 0;
    for (int r = 0; r < nranks; r++) { p->pre.start[r] = S; S += ns_all[r]; if (ns_all[r] > max_ns) max_ns = ns_all[r]; }
    p->pre.start[nranks] = S;
    p->S = S;
    if (S <= 0) return SPLIT_PLAN_NONE_SAVED;
    long long i_mult = target / S;
    if (i_mult < 1) i_mult = 1;
    const long long C = S * i_mult;
    for (int r = 0; r < nranks; r++)  // the largest slice decides for everybody
        if (C * (r + 1) / nranks - C * r / nranks > n_pts_max) return SPLIT_PLAN_OVER_CAPACITY;
    if (C > 0x100000000ll) return SPLIT_PLAN_OVER_RANGE;
    p->i_mult = i_mult;
    p->C = C;
    p->c0 = C * rank / nranks;
    p->c1 = C * (rank + 1) / nranks;
    p->stride = pop_cap(max_ns);
    return SPLIT_PLAN_OK;
}

// brings the words of a cell to their unique form: 0 <= word < 2^32 below the top one, which carries the sign
__device__ __forceinline__ void acc_normalize(long long d[ACC_D]) {
#pragma unroll
    for (int k = 0; k + 1 < ACC_D; k++) {
        const long long carry = d[k] >> 32;  // arithmetic shift = floor
        d[k] -= carry << 32;
        d[k + 1] += carry;
    }
}

// End of the ion: fold the exact accumulators into the FP64 tally cells [c0, c1).  A cell becomes the correctly rounded
// double of the integer its words hold, so the result is a function of the accumulated VALUE only: the magnitude's 64 bits
// from the leading one down, with a sticky bit for everything below them, go through ONE round-to-nearest conversion and
// are then scaled by a power of two (exact: every nonzero result is >= 2^ACC_ELO, far above the subnormals).
__global__ void fold_accumulators_kernel(const long long* __restrict__ acc, size_t c0, size_t c1, double* tally) {
    const size_t c = c0 + (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= c1) return;
    long long d[ACC_D];
    bool any = false;
#pragma unroll
    for (int k = 0; k < ACC_D; k++) { d[k] = acc[c * ACC_D + k]; any |= d[k] != 0; }
    if (!any) { tally[c] = 0.0; return; }
    acc_normalize(d);
    const bool neg = d[ACC_D - 1] < 0;
    if (neg) {  // magnitude: negate word by word, then carry again
#pragma unroll
        for (int k = 0; k < ACC_D; k++) d[k] = -d[k];
        acc_normalize(d);
    }
    // the magnitude as ACC_D + 1 digits of 32 bits (the top word holds up to 63)
    uint32_t u[ACC_D + 1];
#pragma unroll
    for (int k = 0; k < ACC_D; k++) u[k] = (uint32_t)d[k];
    u[ACC_D] = (uint32_t)((unsigned long long)d[ACC_D - 1] >> 32);
    int h = ACC_D;
    while (h >= 0 && u[h] == 0) h--;
    if (h < 0) { tally[c] = 0.0; return; }  // the adds cancelled exactly: +0
    const int lz = __clz(u[h]);
    const uint32_t u1 = h >= 1 ? u[h - 1] : 0u, u2 = h >= 2 ? u[h - 2] : 0u;
    unsigned long long m = ((((unsigned long long)u[h] << 32) | u1) << lz) | ((unsigned long long)u2 >> (32 - lz));
    bool sticky = (uint32_t)(u2 << lz) != 0u;
    for (int k = 0; k + 2 < h; k++) sticky |= u[k] != 0u;
    m |= sticky ? 1ull : 0ull;
    const double v = scalbn(__ull2double_rn(m), ACC_ELO + 32 * (h - 1) - lz);
    tally[c] = neg ? -v : v;
}

// particle_counter.jl:81-85: shock-frame dN(p) of the cosmic rays = sum of the PSD over the angle bins
__global__ void sum_angle_kernel(const double* __restrict__ psd, int M2, int T2, int ng, double* dndp) {
    int idx = blockIdx.x * blockDim.x + threadIdx.x;  // k + M2 * i
    if (idx >= M2 * ng) return;
    const int k = idx % M2, i = idx / M2;
    double s = 0.0;
    for (int j = 0; j < T2; j++) {
        double v = psd[(size_t)k + (size_t)M2 * ((size_t)j + (size_t)T2 * (size_t)i)];
        if (v > 0) s += v;
    }
    dndp[idx] = s;
}

// the optional fields of a fresh record: upstream, not injected, the fine xn_per, prp_x at x_grid_stop, no age, tcut 1
__device__ __forceinline__ void set_optional_defaults(const PopPtrs& p, long long i, double xn_fine, double x_grid_stop) {
    p.down[i] = 0; p.inj[i] = 0; p.xn_per[i] = xn_fine; p.prp_x[i] = x_grid_stop; p.acctime[i] = 0.0; p.tcut[i] = 1;
}

__global__ void fill_defaults_kernel(PopPtrs p, long long n, double xn_fine, double x_grid_stop) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) set_optional_defaults(p, i, xn_fine, x_grid_stop);
}

// init_pop in run-length form (include/mcs.h McsInjection; initializers.jl:977-1134, ion_init.jl:29-53).  HBM-bound: 82 B
// written per particle, bins (<= 151 x 6 doubles) read through L1.  Every operation is an explicitly rounded IEEE one
// (no FMA contraction), so the population is bit-identical to the oracle's and the host mirror's.
struct InjDev {
    const double *ptot, *weight, *lo, *hi, *gfac;
    const long long* start;
    int n_bins, mode, perm_stride;
    long long n_total, grid;
    double x_cm, u_stop, c, xn_fine, x_grid_stop;
    uint32_t key0, key1, ctr2, ctr3;
};
__global__ void generate_population_kernel(PopPtrs p, long long n_local, long long first_global, InjDev J) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_local) return;
    long long s = first_global + i, j = s;
    if (J.perm_stride > 0) {
        const long long K = J.perm_stride, a = J.n_total / K, b = J.n_total % K;
        if (s < b * (a + 1)) j = s / (a + 1) + K * (s % (a + 1));
        else { s -= b * (a + 1); j = (b + s / a) + K * (s % a); }
    }
    int lo = 0, hi = J.n_bins;
    while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (J.start[mid] <= j) lo = mid; else hi = mid; }
    uint32_t o0, o1, o2, o3;
    philox4x32_10(0u, (uint32_t)j, J.ctr2, J.ctr3, J.key0, J.key1, o0, o1, o2, o3);
    const double u1 = u53(o1, o0), u2 = u53(o3, o2);
    const double ptot = J.ptot[lo];
    double pb;
    if (J.mode == MCS_INJ_UPSTREAM) pb = __dmul_rn(__dmul_rn(ptot, 2.0), __dadd_rn(u1, -0.5));
    else {
        const double l = J.lo[lo];
        const double vx = __dadd_rn(l, __dmul_rn(__dadd_rn(J.hi[lo], -l), __dsqrt_rn(u1)));
        if (J.mode == MCS_INJ_FASTPUSH_REL) {
            const double bu = __ddiv_rn(J.u_stop, J.c);
            const double vpf = __dmul_rn(__ddiv_rn(__dadd_rn(vx, -bu), __dadd_rn(1.0, -__dmul_rn(vx, bu))), J.c);
            pb = __dmul_rn(J.gfac[lo], vpf);
        } else pb = __dmul_rn(J.gfac[lo], __dadd_rn(vx, -J.u_stop));
    }
    p.weight[i] = J.weight[lo]; p.ptot[i] = ptot; p.pb[i] = pb; p.x[i] = J.x_cm; p.grid[i] = J.grid;
    p.phi[i] = __dmul_rn(TWO_PI, u2);
    set_optional_defaults(p, i, J.xn_fine, J.x_grid_stop);
}

// sqrt_nr / div_nr against the IEEE operations on operands spread over the fast loop's ranges (mcs_math.cuh).
__global__ void selftest_math_kernel(long long n, uint32_t key0, uint32_t key1, unsigned long long* bad) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t o0, o1, o2, o3;
    philox4x32_10((uint32_t)i, (uint32_t)(i >> 32), 0xABCDu, 7u, key0, key1, o0, o1, o2, o3);
    const double u = u53(o1, o0), v = u53(o3, o2);
    // operands: 1 - c^2 for c near +-1 (sin^2 of small and large angles), plain (0,1], and a wide log-uniform sweep
    double xs, a, b;
    switch (i & 3) {
        case 0: { const double c = 1 - u * exp2(-40.0 * v); xs = 1 - c * c; a = 2 * v - 1; b = sqrt(fmax(xs, 1e-300)); break; }
        case 1: xs = u; a = 2 * v - 1; b = 0.25 + 0.75 * u; break;
        case 2: xs = exp2(1900.0 * u - 950.0); a = (2 * v - 1) * exp2(200.0 * u - 100.0); b = exp2(200.0 * v - 100.0); break;
        default: xs = (1 - u) * 0.5; a = u * u * v; b = 1 - 0.7 * u; break;
    }
    if (xs >= 0x1.0p-960 && __double_as_longlong(sqrt_nr(xs)) != __double_as_longlong(sqrt(xs))) atomicAdd(&bad[0], 1ull);
    if (b != 0.0 && __double_as_longlong(div_nr(a, b)) != __double_as_longlong(a / b)) atomicAdd(&bad[1], 1ull);
}

// ---------------------------------------------------------------------------------------------
// Roofline denominators measured in place (MEASURED_PEAKS.json has no FP64 entry).
__global__ void dfma_peak_kernel(double* out, int iters) {
    double a0 = threadIdx.x * 1e-9, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
    const double b = 1.0000001, c = 1e-9;
    for (int i = 0; i < iters; i++) {
        a0 = fma(a0, b, c); a1 = fma(a1, b, c); a2 = fma(a2, b, c); a3 = fma(a3, b, c);
        a4 = fma(a4, b, c); a5 = fma(a5, b, c); a6 = fma(a6, b, c); a7 = fma(a7, b, c);
    }
    out[blockIdx.x * blockDim.x + threadIdx.x] = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
}

// The NECESSARY arithmetic of one bulk scattering step (SURVEY App. D) and nothing else: Philox block, pitch-angle kick,
// phase advance, move.  No zone test, no escape tests, no tallies, no refill.  Its rate on this GPU is the practical
// ceiling for the transport kernel's hot path and is reported next to the DFMA peak.
__global__ void __launch_bounds__(256, 2) scatter_only_kernel(double* out, int iters, double omc, double inv_xn, double dphi,
                                                             uint32_t key0, uint32_t key1) {
    const uint32_t tid = blockIdx.x * blockDim.x + threadIdx.x;
    double ptot = 1.0e-17, pb = 0.3e-17, pperp = sqrt(ptot * ptot - pb * pb), phi = 0.1, x = -1.0e12;
    const double inv_ptot = 1 / ptot, gper = 6.5e3, inv_gm = 1 / 1.67e-24, ux = 1.0e9, gsf = 1.0;
    double acc = 0.0;
    for (int i = 0; i < iters; i++) {
        uint32_t o0, o1, o2, o3;
        philox4x32_10((uint32_t)i, tid, 2u, 1u, key0, key1, o0, o1, o2, o3);
        const double u1 = u53(o1, o0), u2 = u53(o3, o2);
        const double cos_old = pb * inv_ptot, sin_old = pperp * inv_ptot;
        const double cos_d = 1 - u1 * omc;
        const double sin_d = sqrt_nr(fmax(1 - cos_d * cos_d, 0x1.0p-900));
        const double phi_s = u2 * TWO_PI - PI;
        double sps, cps;
        sincos_bf(phi_s, &sps, &cps);
        const double cos_new = cos_old * cos_d + sin_old * sin_d * cps;
        const double sin_new = sqrt_nr(fmax(1 - cos_new * cos_new, 0x1.0p-900));
        pb = ptot * cos_new;
        pperp = ptot * sin_new;
        double s = div_nr(sps * sin_d, sin_new);
        if (fabs(s) > SIN_UPPER_LIMIT) s = copysign(SIN_UPPER_LIMIT, s);
        phi = (phi + HALF_PI + asin_bf<true>(s)) - HALF_PI;
        const double t_step = gper * inv_xn;
        phi = mod2pi(phi + dphi);
        x = x + gsf * (pb * t_step * inv_gm + ux * t_step);
        acc += t_step;
    }
    out[tid] = x + phi + acc;
}

__global__ void atomic_peak_kernel(double* cells, long long n_cells, int iters) {
    uint32_t s = (blockIdx.x * blockDim.x + threadIdx.x) * 2654435761u + 12345u;
    for (int i = 0; i < iters; i++) {
        s = s * 1664525u + 1013904223u;
        long long idx = (long long)(((unsigned long long)s * (unsigned long long)n_cells) >> 32);
        red_add_f64(&cells[idx], 1.0);
    }
}

}  // namespace mcs
