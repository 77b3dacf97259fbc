// mcs_api.cu — C-ABI (include/mcs.h) of the B200 transport loop: device memory, launches, NCCL.
//
// Every entry point replaces a piece of /root/reference/src/main_loops.jl (see include/mcs.h).  The library
// owns all device state; callers pass plain host pointers.  NCCL is resolved with dlopen at mcs_comm_init so
// that single-GPU users need no NCCL at all and multi-GPU users share the libnccl their process already has.
#include <dlfcn.h>
#include <nccl.h>

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "mcs_device.cuh"
#include "mcs_thermo.cuh"

using namespace mcs;

static thread_local char g_err[768];
static int fail(int code, const char* fmt, const char* a = "", const char* b = "") {
    snprintf(g_err, sizeof g_err, fmt, a, b);
    return code;
}
#define CU(call)                                                                                       \
    do {                                                                                               \
        cudaError_t e_ = (call);                                                                       \
        if (e_ != cudaSuccess) return fail(MCS_ERR_CUDA, "CUDA error: %s at %s", cudaGetErrorString(e_), #call); \
    } while (0)

extern "C" const char* mcs_last_error(void) { return g_err; }
extern "C" const char* mcs_backend(void) { return "cuda-sm_100a"; }

extern "C" int mcs_abi_sizes(int32_t out[6]) {
    out[0] = (int32_t)sizeof(McsConfig); out[1] = (int32_t)sizeof(McsSpecies); out[2] = (int32_t)sizeof(McsTallies);
    out[3] = (int32_t)sizeof(McsPopulation); out[4] = (int32_t)sizeof(McsTraceRec); out[5] = (int32_t)sizeof(McsTiming);
    return MCS_OK;
}

extern "C" void mcs_default_config(McsConfig* c) {
    memset(c, 0, sizeof *c);
    c->abi_version = MCS_ABI_VERSION; c->device = -1;
    c->mp_g = 1.67262192369e-24; c->c_cms = 2.99792458e10; c->qcgs_esu = 4.80320471257e-10;
    c->E_rel_pt = 0.005;
    {
        double me = 9.1093837015e-28, sigT = 6.6524587321e-25, cc = c->c_cms;
        c->rad_loss_fac = 4.0 / 3.0 * cc * sigT / (cc * cc * cc * me * me * 8 * PI);  // constants.jl:30
    }
    c->eta_mfp = 1.0; c->xn_per_fine = 2000.0; c->xn_per_coarse = 100.0; c->age_max = -1.0;
    c->pe_crit = -1.0; c->gam_e_crit = -1.0;
    c->n_ions = 1; c->na_cr = 1000000; c->n_pts_max = 100000;
    for (int i = 0; i < MCS_MAX_IONS; i++) c->inj_fracs[i] = 1.0;
    c->do_retro = 1;
    c->helix_cap = 10000; c->retro_cap = 10000000; c->seed = 210; c->compat = MCS_COMPAT_DEFAULT;
    c->rng_mode = MCS_RNG_PHILOX; c->threads = 1; c->det_tallies = 1;
}

// ---------------------------------------------------------------------------------------------
struct NcclApi {
    void* lib = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
};
static NcclApi g_nccl;
static int nccl_load() {
    if (g_nccl.lib) return MCS_OK;
    const char* names[] = {getenv("MCS_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
    void* lib = nullptr;
    for (const char* n : names) {
        if (!n) continue;
        lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
        if (lib) break;
    }
    if (!lib) return fail(MCS_ERR_COMM, "cannot dlopen libnccl.so.2 (set MCS_NCCL_LIB): %s", dlerror());
#define SYM(field, name)                                                       \
    g_nccl.field = (decltype(g_nccl.field))dlsym(lib, name);                   \
    if (!g_nccl.field) return fail(MCS_ERR_COMM, "libnccl lacks %s", name);
    SYM(GetUniqueId, "ncclGetUniqueId") SYM(CommInitRank, "ncclCommInitRank") SYM(AllReduce, "ncclAllReduce")
    SYM(AllGather, "ncclAllGather") SYM(CommDestroy, "ncclCommDestroy") SYM(GetErrorString, "ncclGetErrorString")
#undef SYM
    g_nccl.lib = lib;
    return MCS_OK;
}
#define NC(call)                                                                                        \
    do {                                                                                                \
        ncclResult_t r_ = (call);                                                                       \
        if (r_ != ncclSuccess) return fail(MCS_ERR_COMM, "NCCL error: %s at %s", g_nccl.GetErrorString(r_), #call); \
    } while (0)

// ---------------------------------------------------------------------------------------------
struct McsHandle {
    McsConfig cfg;
    McsSpecies sp;
    int device = 0, n_sm = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev2 = nullptr, ev3 = nullptr, ev4 = nullptr, ev5 = nullptr;
    bool have_profile = false, have_ion = false;
    int i_iter = 0, i_ion = 0;
    int ng = 0, M = 0, T = 0;
    long long n_use = 0, first_global = 0, n_saved_last = 0, n_saved_global_last = 0;
    // device buffers
    double2* d_az = nullptr;   // azimuth table of the fast loop: {sin, cos} of the 256 bin centres of phi_s
    double* d_boost = nullptr; // 3 arrays of (ng+2): ux/ut, uz/ut, ux*uz/ut^2
    double* d_grid = nullptr;  // 10 arrays of (ng+2): xg ux uz ut gsf gef bt sinth costh (bef unused) + tcuts(NA_C)
    double* d_zone = nullptr;  // eps_target, recv_pool [ng] each
    unsigned char* d_pop = nullptr;  // the three population blocks, one after the other
    PopPtrs pop[3];            // views of them: cur, saved, next
    int cur = 0, nxt = 2;      // saved is always pop[1]
    uint8_t* d_l_save = nullptr;
    int *d_fate = nullptr, *d_helix = nullptr;
    long long *d_retro = nullptr, *d_draws = nullptr, *d_saved_idx = nullptr, *d_block_off = nullptr, *d_total = nullptr;
    int* d_block_cnt = nullptr;
    // tallies: one packed FP64 buffer (single all-reduce) + one packed u64 buffer
    double* d_tally = nullptr;
    long long* d_acc = nullptr;  // exact accumulators (cfg.det_tallies): ACC_D words per cell of d_tally from off_psd on
    size_t n_tally = 0, off_pxx = 0, off_pxz = 0, off_efl = 0, off_psd = 0, off_esc_up = 0, off_esc_dn = 0, off_en_eff = 0,
           off_num_eff = 0, off_wc = 0, off_sc = 0, off_pool = 0, off_sf = 0, off_pf = 0, off_scal = 0, off_thsf = 0, off_thpf = 0,
           off_dndp = 0;
    unsigned long long* d_u64 = nullptr;  // [ng crossings | CNT_N counters]
    unsigned long long h_counters[CNT_N];
    long long *d_tg = nullptr;
    double *d_tpx = nullptr, *d_tpt = nullptr, *d_tw = nullptr;
    double* d_partials = nullptr;
    int max_blocks = 0, block = 256, blocks_per_sm = 2;
    // debug
    double* d_replay_u = nullptr;
    double* d_inj = nullptr;  // packed injection bins (mcs_begin_ion_generate)
    long long* d_replay_off = nullptr;
    long long replay_n = 0;
    int* d_trace_slot = nullptr;
    McsTraceRec* d_trace_recs = nullptr;
    int* d_trace_cnt = nullptr;
    int n_trace = 0, trace_max = 0;
    std::vector<long long> trace_idx;
    // comm
    ncclComm_t comm = nullptr;
    int rank = 0, nranks = 1;
    long long* d_gather = nullptr;    // [64 ranks][4]: {n_saved, n_use, error flag, spare} of the current pcut
    unsigned char* d_xchg = nullptr;  // all-gather buffer of saved records for the rebalancing split
    size_t xchg_bytes = 0;
    bool reduced = false;             // mcs_end_ion already summed the tallies over ranks (idempotence)
    bool ended = false;               // mcs_end_ion has folded the accumulators: d_tally holds this ion's final FP64 tallies
    bool split_timed = false;         // ev2/ev3 bracket an un-timed split (elapsed time read at the next sync)
    unsigned long long steps0 = 0, saved0 = 0, reds0 = 0;  // counter values before the pcut in flight
    double last_steps_per_particle = 0;  // of the previous pcut of this ion (0: none yet); picks the kernel build
    McsTiming tm;
    DevParams P;
};

static int check_index_range(long long first_global, long long n);

static size_t psd_len(const McsHandle* h) { return (size_t)(h->M + 2) * (size_t)(h->T + 2) * (size_t)h->ng; }

extern "C" int mcs_destroy(McsHandle* h) {
    if (!h) return MCS_OK;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    if (h->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(h->comm);
    cudaFree(h->d_grid); cudaFree(h->d_boost); cudaFree(h->d_zone); cudaFree(h->d_az);
    cudaFree(h->d_pop); cudaFree(h->d_l_save); cudaFree(h->d_fate); cudaFree(h->d_helix); cudaFree(h->d_retro); cudaFree(h->d_draws);
    cudaFree(h->d_saved_idx); cudaFree(h->d_block_off); cudaFree(h->d_total); cudaFree(h->d_block_cnt);
    cudaFree(h->d_tally); cudaFree(h->d_acc); cudaFree(h->d_u64); cudaFree(h->d_tg); cudaFree(h->d_tpx); cudaFree(h->d_tpt); cudaFree(h->d_tw);
    cudaFree(h->d_inj); cudaFree(h->d_partials); cudaFree(h->d_replay_u); cudaFree(h->d_replay_off); cudaFree(h->d_trace_slot);
    cudaFree(h->d_trace_recs); cudaFree(h->d_trace_cnt); cudaFree(h->d_gather); cudaFree(h->d_xchg);
    if (h->ev0) cudaEventDestroy(h->ev0);
    if (h->ev1) cudaEventDestroy(h->ev1);
    if (h->ev2) cudaEventDestroy(h->ev2);
    if (h->ev3) cudaEventDestroy(h->ev3);
    if (h->ev4) cudaEventDestroy(h->ev4);
    if (h->ev5) cudaEventDestroy(h->ev5);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
    return MCS_OK;
}

static int env_int(const char* name, int dflt) {
    const char* s = getenv(name);
    return s && *s ? atoi(s) : dflt;
}

extern "C" int mcs_create(const McsConfig* cfg, McsHandle** out) {
    if (!cfg || !out) return fail(MCS_ERR_ARG, "null argument");
    if (cfg->abi_version != MCS_ABI_VERSION) return fail(MCS_ERR_ARG, "abi_version mismatch");
    if (cfg->n_grid < 1 || cfg->n_grid > 2048 || cfg->n_pts_max < 1 || cfg->n_ions < 1 || cfg->n_ions > MCS_MAX_IONS ||
        cfg->n_tcuts > MCS_NA_C || cfg->n_tcuts < 0 || cfg->n_xspec > MCS_MAX_XSPEC || cfg->n_xspec < 0 ||
        cfg->num_psd_mom_bins < 1 || cfg->num_psd_theta_bins < 1 || cfg->na_cr < 0)
        return fail(MCS_ERR_ARG, "bad sizes in McsConfig");
    if (cfg->use_custom_frg) return fail(MCS_ERR_UNSUPPORTED, "use_custom_frg: the reference errors too (scattering.jl:53)");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev < 1)
        return fail(MCS_ERR_CUDA, "no CUDA device: %s (this library has no CPU fallback)", cudaGetErrorString(e));
    int dev = cfg->device;
    if (dev < 0) {
        const char* lr = getenv("LOCAL_RANK");
        dev = lr ? atoi(lr) % ndev : 0;
    }
    if (dev >= ndev) return fail(MCS_ERR_ARG, "device ordinal out of range");
    CU(cudaSetDevice(dev));
    McsHandle* h = new McsHandle();
    memset(&h->tm, 0, sizeof h->tm);
    memset(h->pop, 0, sizeof h->pop);
    memset(h->h_counters, 0, sizeof h->h_counters);
    h->cfg = *cfg; h->device = dev;
    h->cfg.det_tallies = env_int("MCS_DET_TALLIES", cfg->det_tallies);  // tuning aid: 0 = FP64 red path
    h->ng = cfg->n_grid; h->M = cfg->num_psd_mom_bins; h->T = cfg->num_psd_theta_bins;
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, dev));
    h->n_sm = prop.multiProcessorCount;
    h->block = env_int("MCS_BLOCK", MCS_BLOCK);
    if (h->block > MCS_BLOCK || h->block < 32 || (h->block & 31)) h->block = MCS_BLOCK;
    h->blocks_per_sm = env_int("MCS_BLOCKS_PER_SM", MCS_MIN_BLOCKS);
    h->max_blocks = h->n_sm * h->blocks_per_sm;
#define CUA(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { fail(MCS_ERR_NOMEM, "CUDA alloc: %s at %s", cudaGetErrorString(e_), #call); mcs_destroy(h); return MCS_ERR_NOMEM; } } while (0)
    CUA(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
    CUA(cudaEventCreate(&h->ev0)); CUA(cudaEventCreate(&h->ev1)); CUA(cudaEventCreate(&h->ev2)); CUA(cudaEventCreate(&h->ev3)); CUA(cudaEventCreate(&h->ev4)); CUA(cudaEventCreate(&h->ev5));
    const int ng = h->ng, ng2 = ng + 2;
    const long long N = cfg->n_pts_max;
    CUA(cudaMalloc(&h->d_grid, (size_t)(9 * ng2 + MCS_NA_C) * 8));
    CUA(cudaMalloc(&h->d_boost, (size_t)3 * ng2 * 8));
    CUA(cudaMalloc(&h->d_zone, (size_t)2 * ng * 8));
    CUA(cudaMalloc(&h->d_az, (size_t)AZ_N * sizeof(double2)));
    const long long cap = pop_cap(N);
    CUA(cudaMalloc(&h->d_pop, (size_t)3 * (size_t)cap * POP_REC_BYTES));
    for (int k = 0; k < 3; k++) h->pop[k] = pop_view(h->d_pop + (size_t)k * (size_t)cap * POP_REC_BYTES, cap, 0);
    CUA(cudaMalloc(&h->d_l_save, (size_t)N)); CUA(cudaMalloc(&h->d_fate, (size_t)N * 4)); CUA(cudaMalloc(&h->d_helix, (size_t)N * 4));
    CUA(cudaMalloc(&h->d_retro, (size_t)N * 8)); CUA(cudaMalloc(&h->d_draws, (size_t)N * 8));
    CUA(cudaMalloc(&h->d_saved_idx, (size_t)N * 8));
    const long long scan_blocks = compaction_blocks(N);
    CUA(cudaMalloc(&h->d_block_cnt, (size_t)scan_blocks * 4)); CUA(cudaMalloc(&h->d_block_off, (size_t)scan_blocks * 8));
    CUA(cudaMalloc(&h->d_total, 8));
    // packed FP64 tally buffer
    size_t o = 0;
    auto take = [&](size_t n) { size_t r = o; o += n; return r; };
    h->off_pxx = take(ng); h->off_pxz = take(ng); h->off_efl = take(ng); h->off_psd = take(psd_len(h));
    h->off_esc_up = take((size_t)E1 * E1); h->off_esc_dn = take((size_t)E1 * E1); h->off_en_eff = take(E1);
    h->off_num_eff = take(E1); h->off_wc = take(MCS_NA_C); h->off_sc = take((size_t)E1 * MCS_NA_C); h->off_pool = take(ng);
    h->off_sf = take((size_t)E1 * MCS_MAX_XSPEC); h->off_pf = take((size_t)E1 * MCS_MAX_XSPEC); h->off_scal = take(SC_N);
    if (cfg->bin_thermal) { h->off_thsf = take(psd_len(h)); h->off_thpf = take(psd_len(h)); h->off_dndp = take((size_t)(h->M + 2) * ng); }
    h->n_tally = o;
    CUA(cudaMalloc(&h->d_tally, o * 8));
    if (h->cfg.det_tallies) CUA(cudaMalloc(&h->d_acc, o * ACC_D * 8));
    CUA(cudaMalloc(&h->d_u64, (size_t)(ng + CNT_N) * 8));
    const size_t L = (size_t)(cfg->na_cr > 0 ? cfg->na_cr : 1);
    CUA(cudaMalloc(&h->d_tg, L * 8)); CUA(cudaMalloc(&h->d_tpx, L * 8)); CUA(cudaMalloc(&h->d_tpt, L * 8)); CUA(cudaMalloc(&h->d_tw, L * 8));
    CUA(cudaMalloc(&h->d_partials, (size_t)h->max_blocks * (3 * ng + SC_N) * 8));
    CUA(cudaMalloc(&h->d_gather, 64 * 4 * 8));
    CUA(cudaMemsetAsync(h->d_tally, 0, o * 8, h->stream));
    CUA(cudaMemsetAsync(h->d_u64, 0, (size_t)(ng + CNT_N) * 8, h->stream));
    // large grids: fewer warps per block so that the per-warp flux partials still fit (the per-launch shared-memory
    // attribute is set in mcs_run_pcut: it belongs to the function and the device, not to this handle)
    while (h->block > 32 && block_smem_bytes(ng, h->block / 32) > (size_t)200 * 1024 / (size_t)h->blocks_per_sm) h->block /= 2;
#undef CUA
    // static part of the kernel parameters
    DevParams& P = h->P;
    memset(&P, 0, sizeof P);
    P.mp = cfg->mp_g; P.c = cfg->c_cms; P.qcgs = cfg->qcgs_esu; P.E_rel_pt = cfg->E_rel_pt; P.rad_loss_fac = cfg->rad_loss_fac;
    P.gam0 = cfg->gam0; P.u0 = cfg->u0; P.u2 = cfg->u2; P.bmag2 = cfg->bmag2; P.pe_crit = cfg->pe_crit;
    P.gam_e_crit = cfg->gam_e_crit; P.eta_mfp = cfg->eta_mfp;
    P.psd_mom_min = cfg->psd_mom_min; P.psd_cos_fine = cfg->psd_cos_fine; P.delta_cos = cfg->delta_cos;
    P.psd_theta_min = cfg->psd_theta_min; P.bpd_mom = (double)cfg->psd_bins_per_dec_mom; P.bpd_th = (double)cfg->psd_bins_per_dec_theta;
    P.energy_transfer_frac = cfg->energy_transfer_frac; P.feb_up = cfg->feb_upstream; P.feb_dn = cfg->feb_downstream;
    P.x_grid_stop = cfg->x_grid_stop; P.B_CMBz = cfg->B_CMBz; P.xn_fine = cfg->xn_per_fine; P.xn_coarse = cfg->xn_per_coarse;
    P.age_max = cfg->age_max;
    for (int i = 0; i < MCS_MAX_XSPEC; i++) P.x_spec[i] = cfg->x_spec[i];
    P.M = h->M; P.T = h->T; P.n_grid = ng; P.i_grid_feb = cfg->i_grid_feb; P.i_shock = cfg->i_shock; P.n_xspec = cfg->n_xspec;
    P.n_tcuts = cfg->n_tcuts; P.helix_cap = cfg->helix_cap; P.retro_cap = cfg->retro_cap;
    P.flags = (cfg->do_rad_losses ? F_RAD_LOSSES : 0) | (cfg->do_retro ? F_RETRO : 0) | (cfg->do_tcuts ? F_TCUTS : 0) |
              (cfg->dont_DSA ? F_DONT_DSA : 0) | (cfg->dont_scatter ? F_DONT_SCATTER : 0) |
              (cfg->use_custom_epsB ? F_CUSTOM_EPSB : 0) | ((cfg->compat & MCS_COMPAT_RETRO_KEEP_NEW_PITCH) ? F_KEEP_NEW_PITCH : 0) |
              (env_int("MCS_DYNAMIC_QUEUE", cfg->dynamic_queue) ? F_DYNAMIC_QUEUE : 0) |
              (env_int("MCS_NO_FAST_LOOP", 0) ? F_NO_FAST_LOOP : 0);
    {   // per-xn_per scattering constants, host libm (scattering.jl:46-60: the gyroradius cancels in vp_tg / lambda_mfp)
        const double xn[2] = {cfg->xn_per_fine, cfg->xn_per_coarse};
        for (int k = 0; k < 2; k++) {
            P.omc[k] = 1 - cos(sqrt(6 * (TWO_PI * 1.0) / (xn[k] * (cfg->eta_mfp * 1.0))));
            P.inv_xn[k] = 1.0 / xn[k];
            P.dphi[k] = TWO_PI / xn[k];
            P.cdphi[k] = cos(P.dphi[k]); P.sdphi[k] = sin(P.dphi[k]);
        }
    }
    P.key0 = (uint32_t)cfg->seed; P.key1 = (uint32_t)(cfg->seed >> 32);
    for (int r = 0; r < 10; r++) { P.rk[2 * r] = P.key0 + (uint32_t)r * 0x9E3779B9u; P.rk[2 * r + 1] = P.key1 + (uint32_t)r * 0xBB67AE85u; }
    double* g = h->d_grid;
    P.xg = g; P.ux = g + ng2; P.uz = g + 2 * ng2; P.ut = g + 3 * ng2; P.gsf = g + 4 * ng2; P.gef = g + 5 * ng2;
    P.bt = g + 6 * ng2; P.sinth = g + 7 * ng2; P.costh = g + 8 * ng2; P.tcuts = g + 9 * ng2;
    P.rxt = h->d_boost; P.rzt = h->d_boost + ng2; P.crt = h->d_boost + 2 * ng2;
    P.eps_target = h->d_zone; P.recv_pool = h->d_zone + ng;
    P.az_tab = h->d_az;
    P.l_save = h->d_l_save; P.fate = h->d_fate; P.helix = h->d_helix; P.retro = h->d_retro; P.draws = h->d_draws;
    TallyPtrs& t = P.t;
    double* b = h->d_tally;
    t.psd = b + h->off_psd; t.esc_up = b + h->off_esc_up; t.esc_dn = b + h->off_esc_dn; t.esc_en_eff = b + h->off_en_eff;
    t.esc_num_eff = b + h->off_num_eff; t.w_coupled = b + h->off_wc; t.s_coupled = b + h->off_sc; t.pool = b + h->off_pool;
    t.spec_sf = b + h->off_sf; t.spec_pf = b + h->off_pf;
    t.therm_sf = cfg->bin_thermal ? b + h->off_thsf : nullptr; t.therm_pf = cfg->bin_thermal ? b + h->off_thpf : nullptr;
    t.dndp_cr = cfg->bin_thermal ? b + h->off_dndp : nullptr;
    t.acc = h->d_acc; t.tally_base = h->d_tally;
    t.pxx = b + h->off_pxx; t.pxz = b + h->off_pxz; t.efl = b + h->off_efl; t.scal = b + h->off_scal;
    t.counters = h->d_u64 + ng;
    t.ncross = h->d_u64;
    t.tg = h->d_tg; t.tpx = h->d_tpx; t.tpt = h->d_tpt; t.tw = h->d_tw; t.na_cr = cfg->na_cr;
    t.block_partials = h->d_partials;
    {
        double2 az[AZ_N];  // sine and cosine of the bin centres of the scattering azimuth
        az_table(az);
        cudaError_t e2 = cudaMemcpyAsync(h->d_az, az, sizeof az, cudaMemcpyHostToDevice, h->stream);
        if (e2 == cudaSuccess) e2 = cudaStreamSynchronize(h->stream);
        if (e2 != cudaSuccess) { mcs_destroy(h); return fail(MCS_ERR_CUDA, "CUDA error: %s", cudaGetErrorString(e2)); }
    }
    {
        cudaError_t e2 = cudaMemcpyAsync((void*)P.tcuts, cfg->tcuts, MCS_NA_C * 8, cudaMemcpyHostToDevice, h->stream);
        if (e2 == cudaSuccess) e2 = cudaStreamSynchronize(h->stream);
        if (e2 != cudaSuccess) { mcs_destroy(h); return fail(MCS_ERR_CUDA, "CUDA error: %s", cudaGetErrorString(e2)); }
    }
    *out = h;
    return MCS_OK;
}

// ---------------------------------------------------------------------------------------------
extern "C" int mcs_comm_unique_id(void* id128) {
    int rc = nccl_load();
    if (rc) return rc;
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
    NC(g_nccl.GetUniqueId((ncclUniqueId*)id128));
    return MCS_OK;
}
extern "C" int mcs_comm_init(McsHandle* h, int rank, int nranks, const void* id128) {
    if (!h || nranks < 1 || rank < 0 || rank >= nranks || nranks > 64) return fail(MCS_ERR_ARG, "bad rank/nranks");
    h->rank = rank; h->nranks = nranks;
    if (nranks == 1) return MCS_OK;
    if (!id128) return fail(MCS_ERR_ARG, "null unique id");
    int rc = nccl_load();
    if (rc) return rc;
    CU(cudaSetDevice(h->device));
    ncclUniqueId id;
    memcpy(&id, id128, sizeof id);
    NC(g_nccl.CommInitRank(&h->comm, nranks, id, rank));
    // Exchange buffer of the rebalancing split, sized for the worst case (every rank saves its whole population) here,
    // where a failure is reported to each caller before any collective: inside the pcut loop a rank that bailed out
    // alone would leave the others blocked in the next all-gather.
    const size_t need = (size_t)pop_cap(h->cfg.n_pts_max) * POP_REC_BYTES * (size_t)nranks;
    cudaFree(h->d_xchg); h->d_xchg = nullptr; h->xchg_bytes = 0;
    if (cudaMalloc(&h->d_xchg, need) != cudaSuccess) return fail(MCS_ERR_NOMEM, "cannot allocate the split exchange buffer");
    h->xchg_bytes = need;
    return MCS_OK;
}

extern "C" int mcs_set_profile(McsHandle* h, int32_t n_grid, const double* xg, const double* ux, const double* uz,
                               const double* ut, const double* gsf, const double* gef, const double* bef, const double* bt,
                               const double* th, const double* eps_target, const double* recv_pool) {
    (void)bef;
    if (!h || n_grid != h->ng) return fail(MCS_ERR_ARG, "n_grid mismatch");
    if (!xg || !ux || !uz || !ut || !gsf || !gef || !bt || !th) return fail(MCS_ERR_ARG, "null profile array");
    CU(cudaSetDevice(h->device));
    const int ng2 = h->ng + 2;
    std::vector<double> buf((size_t)9 * ng2 + 2 * h->ng, 0.0);
    const double* src[7] = {xg, ux, uz, ut, gsf, gef, bt};
    for (int a = 0; a < 7; a++) memcpy(&buf[(size_t)a * ng2], src[a], (size_t)ng2 * 8);
    h->P.oblique = 0;
    for (int i = 0; i < ng2; i++) {  // per-zone sin/cos(theta_B) tables (particle_loop.jl:203-204), host libm
        buf[(size_t)7 * ng2 + i] = sin(th[i]);
        buf[(size_t)8 * ng2 + i] = cos(th[i]);
        if (buf[(size_t)7 * ng2 + i] != 0.0) h->P.oblique = 1;
    }
    if (eps_target) memcpy(&buf[(size_t)9 * ng2], eps_target, (size_t)h->ng * 8);
    if (recv_pool) memcpy(&buf[(size_t)9 * ng2 + h->ng], recv_pool, (size_t)h->ng * 8);
    std::vector<double> boost((size_t)3 * ng2);
    for (int i = 0; i < ng2; i++) {  // transformers.jl:553-560: the same three quotients for every particle entering zone i
        boost[i] = ux[i] / ut[i];
        boost[(size_t)ng2 + i] = uz[i] / ut[i];
        boost[(size_t)2 * ng2 + i] = ux[i] * uz[i] / (ut[i] * ut[i]);
    }
    CU(cudaMemcpyAsync(h->d_boost, boost.data(), (size_t)3 * ng2 * 8, cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(h->d_grid, buf.data(), (size_t)9 * ng2 * 8, cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(h->d_zone, &buf[(size_t)9 * ng2], (size_t)2 * h->ng * 8, cudaMemcpyHostToDevice, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    h->have_profile = true;
    return MCS_OK;
}

// The start of an ion, shared by mcs_begin_ion and mcs_begin_ion_generate: resets the handle's ion state, clears the
// tallies (clear_psd!, ion_init.jl:1-16) and every other per-ion sum, then runs `setup`, which fills the current population
// with its n particles.  The time from the reset to the end of `setup` goes to h2d_ms.
template <class Setup>
static int begin_ion(McsHandle* h, int32_t i_iter, int32_t i_ion, const McsSpecies* sp, long long n, long long first_global,
                     Setup&& setup) {
    CU(cudaSetDevice(h->device));
    h->sp = *sp; h->i_iter = i_iter; h->i_ion = i_ion; h->reduced = false; h->ended = false; h->split_timed = false; h->last_steps_per_particle = 0;
    h->n_use = n; h->first_global = first_global; h->n_saved_last = 0; h->n_saved_global_last = 0;
    CU(cudaMemsetAsync(h->d_tally, 0, h->n_tally * 8, h->stream));
    if (h->d_acc) CU(cudaMemsetAsync(h->d_acc, 0, h->n_tally * ACC_D * 8, h->stream));
    CU(cudaMemsetAsync(h->d_u64, 0, (size_t)(h->ng + CNT_N) * 8, h->stream));
    memset(h->h_counters, 0, sizeof h->h_counters);
    CU(cudaEventRecord(h->ev2, h->stream));
    const int rc = setup(h->pop[h->cur]);
    if (rc) return rc;
    CU(cudaEventRecord(h->ev3, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    float ms = 0;
    CU(cudaEventElapsedTime(&ms, h->ev2, h->ev3));
    h->tm.h2d_ms += ms;
    h->have_ion = true;
    return MCS_OK;
}

extern "C" int mcs_begin_ion(McsHandle* h, int32_t i_iter, int32_t i_ion, const McsSpecies* sp, int64_t n, int64_t first_global,
                             const McsPopulation* pop) {
    if (!h || !sp || !pop) return fail(MCS_ERR_ARG, "null argument");
    if (!h->have_profile) return fail(MCS_ERR_STATE, "mcs_set_profile first");
    if (n < 0 || n > h->cfg.n_pts_max) return fail(MCS_ERR_ARG, "n_pts exceeds n_pts_max");
    if (i_ion < 1 || i_ion > h->cfg.n_ions) return fail(MCS_ERR_ARG, "i_ion out of range");
    if (n > 0 && (!pop->weight || !pop->ptot_pf || !pop->pb_pf || !pop->x_cm || !pop->grid || !pop->phi_rad))
        return fail(MCS_ERR_ARG, "weight/ptot_pf/pb_pf/x_cm/grid/phi_rad are required");
    for (int64_t i = 0; i < n; i++)
        if (pop->grid[i] < 0 || pop->grid[i] > h->ng + 1) return fail(MCS_ERR_ARG, "grid index out of range");
    { int rcg = check_index_range(first_global, n); if (rcg) return rcg; }
    return begin_ion(h, i_iter, i_ion, sp, n, first_global, [&](const PopPtrs& p) {
        if (n == 0) return MCS_OK;
        // every optional field gets its default first: the uploads of the fields the caller gives overwrite them
        fill_defaults_kernel<<<(unsigned)((n + 255) / 256), 256, 0, h->stream>>>(p, n, h->cfg.xn_per_fine, h->cfg.x_grid_stop);
        CU(cudaGetLastError());
        h->tm.other_launches++;
#define X(T, name, pub) \
        if (pop->pub) CU(cudaMemcpyAsync(p.name, pop->pub, (size_t)n * sizeof(T), cudaMemcpyHostToDevice, h->stream));
        MCS_POP_FIELDS(X)
#undef X
        return MCS_OK;
    });
}

extern "C" int mcs_begin_ion_generate(McsHandle* h, int32_t i_iter, int32_t i_ion, const McsSpecies* sp, int64_t first_global,
                                      int64_t n_local, const McsInjection* inj) {
    if (!h || !sp || !inj) return fail(MCS_ERR_ARG, "null argument");
    if (!h->have_profile) return fail(MCS_ERR_STATE, "mcs_set_profile first");
    if (i_ion < 1 || i_ion > h->cfg.n_ions) return fail(MCS_ERR_ARG, "i_ion out of range");
    if (inj->n_bins < 1 || !inj->bin_ptot || !inj->bin_weight || !inj->bin_start) return fail(MCS_ERR_ARG, "injection bins missing");
    if (inj->mode < 0 || inj->mode > 2) return fail(MCS_ERR_ARG, "injection mode");
    if (inj->mode != MCS_INJ_UPSTREAM && (!inj->bin_lo || !inj->bin_hi || !inj->bin_gfac)) return fail(MCS_ERR_ARG, "fast-push bins missing");
    const int nb = inj->n_bins;
    const int64_t n_total = inj->bin_start[nb];
    if (n_local < 0 || first_global < 0 || first_global + n_local > n_total) return fail(MCS_ERR_ARG, "shard outside the population");
    if (n_local > h->cfg.n_pts_max) return fail(MCS_ERR_ARG, "n_pts exceeds n_pts_max");
    if (inj->grid < 0 || inj->grid > h->ng + 1) return fail(MCS_ERR_ARG, "grid index out of range");
    { int rcg = check_index_range(first_global, n_local); if (rcg) return rcg; }
    if (n_total > 0x100000000ll) return fail(MCS_ERR_ARG, "global particle index exceeds 2^32 (RNG counter width)");
    return begin_ion(h, i_iter, i_ion, sp, n_local, first_global, [&](const PopPtrs& p) {
        // bins: one packed upload [ptot | weight | lo | hi | gfac | start]
        std::vector<double> pack((size_t)nb * 5 + (size_t)nb + 1, 0.0);
        for (int b = 0; b < nb; b++) {
            pack[b] = inj->bin_ptot[b]; pack[nb + b] = inj->bin_weight[b];
            if (inj->mode != MCS_INJ_UPSTREAM) { pack[2 * nb + b] = inj->bin_lo[b]; pack[3 * nb + b] = inj->bin_hi[b]; pack[4 * nb + b] = inj->bin_gfac[b]; }
        }
        memcpy(&pack[(size_t)5 * nb], inj->bin_start, (size_t)(nb + 1) * 8);
        cudaFree(h->d_inj); h->d_inj = nullptr;
        CU(cudaMalloc(&h->d_inj, pack.size() * 8));
        CU(cudaMemcpyAsync(h->d_inj, pack.data(), pack.size() * 8, cudaMemcpyHostToDevice, h->stream));
        InjDev J;
        J.ptot = h->d_inj; J.weight = h->d_inj + nb; J.lo = h->d_inj + 2 * nb; J.hi = h->d_inj + 3 * nb; J.gfac = h->d_inj + 4 * nb;
        J.start = reinterpret_cast<const long long*>(h->d_inj + 5 * nb);
        J.n_bins = nb; J.mode = inj->mode; J.perm_stride = inj->perm_stride; J.n_total = n_total; J.grid = inj->grid;
        J.x_cm = inj->x_cm; J.u_stop = inj->u_stop; J.c = h->cfg.c_cms; J.xn_fine = h->cfg.xn_per_fine; J.x_grid_stop = h->cfg.x_grid_stop;
        J.key0 = h->P.key0; J.key1 = h->P.key1; J.ctr2 = (uint32_t)i_ion << 16; J.ctr3 = (uint32_t)i_iter;
        if (n_local > 0) {
            generate_population_kernel<<<(unsigned)((n_local + 255) / 256), 256, 0, h->stream>>>(p, n_local, first_global, J);
            CU(cudaGetLastError());
            h->tm.other_launches++;
        }
        return MCS_OK;
    });
}

static int read_counters(McsHandle* h) {
    CU(cudaMemcpyAsync(h->h_counters, h->d_u64 + h->ng, CNT_N * 8, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return MCS_OK;
}

// RNG counters hold the GLOBAL particle index in 32 bits and the pcut in 16: refuse anything that would wrap and
// silently reuse a stream.
static int check_index_range(long long first_global, long long n) {
    if (n > 0x7fffffffll) return fail(MCS_ERR_ARG, "more than 2^31-1 particles on one rank");
    if (first_global < 0 || first_global + n > 0x100000000ll) return fail(MCS_ERR_ARG, "global particle index exceeds 2^32 (RNG counter width)");
    return MCS_OK;
}

// Launch the transport kernel of one pcut and the ordered reduction of its block partials; no host synchronisation.
static int launch_pcut(McsHandle* h, int32_t i_pcut, double pcut, double pcut_prev) {
    if (i_pcut < 0 || i_pcut > 0xFFFF) return fail(MCS_ERR_ARG, "i_pcut outside the RNG counter's 16-bit field");
    const long long n = h->n_use;
    h->steps0 = h->h_counters[CNT_HELIX] + h->h_counters[CNT_RETRO];
    h->saved0 = h->h_counters[CNT_FATE0];
    h->reds0 = h->h_counters[CNT_RED];
    DevParams& P = h->P;
    P.aa = h->sp.aa; P.zz = h->sp.zz_esu; P.n0 = h->sp.n0; P.pmax_cutoff = h->sp.pmax_cutoff; P.ewf = h->sp.electron_weight_fac;
    P.m = P.aa * P.mp; P.mc = P.m * P.c; P.inj_frac = h->cfg.inj_fracs[h->i_ion - 1];
    P.pcut = pcut; P.pcut_prev = pcut_prev;
    P.ctr2 = ((uint32_t)i_pcut & 0xFFFFu) | ((uint32_t)h->i_ion << 16); P.ctr3 = (uint32_t)h->i_iter;
    P.first_global = h->first_global; P.n_use = n;
    P.cur = h->pop[h->cur]; P.saved = h->pop[1];
    const bool debug = h->cfg.rng_mode == MCS_RNG_REPLAY || h->n_trace > 0;
    P.replay_u = h->cfg.rng_mode == MCS_RNG_REPLAY ? h->d_replay_u : nullptr;
    P.replay_off = h->d_replay_off; P.replay_n = h->replay_n;
    if (h->cfg.rng_mode == MCS_RNG_REPLAY && !h->d_replay_u) return fail(MCS_ERR_STATE, "replay mode without mcs_replay_set_stream");
    P.trace_slot = nullptr; P.trace_recs = h->d_trace_recs; P.trace_cnt = h->d_trace_cnt; P.trace_max = h->trace_max;
    if (h->n_trace > 0 && n > 0) {
        std::vector<int> slot((size_t)n, -1);
        for (int t = 0; t < h->n_trace; t++)
            if (h->trace_idx[t] >= 0 && h->trace_idx[t] < n) slot[(size_t)h->trace_idx[t]] = t;
        cudaFree(h->d_trace_slot); h->d_trace_slot = nullptr;
        CU(cudaMalloc(&h->d_trace_slot, (size_t)n * 4));
        CU(cudaMemcpyAsync(h->d_trace_slot, slot.data(), (size_t)n * 4, cudaMemcpyHostToDevice, h->stream));
        CU(cudaMemsetAsync(h->d_trace_cnt, 0, (size_t)h->n_trace * 4, h->stream));
        CU(cudaStreamSynchronize(h->stream));
        P.trace_slot = h->d_trace_slot;
    }
    // l_save .= false (main_loops.jl:184); the *_saved arrays are only read where l_save is set
    CU(cudaMemsetAsync(h->d_l_save, 0, (size_t)(n > 0 ? n : 1), h->stream));
    CU(cudaMemsetAsync(h->d_u64 + h->ng + CNT_QUEUE, 0, 8, h->stream));
    CU(cudaEventRecord(h->ev0, h->stream));
    if (n > 0) {
        long long want = (n + h->block - 1) / h->block;
        int blocks = (int)(want < h->max_blocks ? want : h->max_blocks);
        const size_t smem = block_smem_bytes(h->ng, h->block / 32);
        const bool electron = h->sp.aa < 1;
        const bool obl = P.oblique != 0;  // only the fast loop reads it: the debug build has none
        // SLIM build of the fast loop (drain helpers out of line) for short trajectories, where the warps go back and forth
        // between the loop and the general section and wait for instruction fetch; the arithmetic is the same.  Chosen from
        // the previous pcut of this ion: fewer than 2000 scattering steps per particle (MCS_SLIM_DRAIN=0/1 forces it).
        const int slim_env = env_int("MCS_SLIM_DRAIN", -1);
        const bool slim = slim_env >= 0 ? slim_env != 0 : (h->last_steps_per_particle > 0 && h->last_steps_per_particle < 2000.0);
        // which optional per-pass features this launch needs; the two commonest masks have their own builds of the kernel
        const int feat = (P.age_max > 0 ? FEAT_AGE : 0) | ((P.flags & F_TCUTS) ? FEAT_TCUTS : 0) | (P.feb_dn > 0 ? FEAT_FEB_DN : 0) |
                         (((P.flags & F_DONT_DSA) || P.inj_frac < 1) ? FEAT_REFLECT : 0) | (P.energy_transfer_frac > 0 ? FEAT_ETF : 0);
        const bool spec = env_int("MCS_PLAIN", 1) != 0 && !obl && (feat == 0 || feat == FEAT_ETF);
        const bool custom = h->cfg.use_custom_epsB != 0 && !obl;  // custom eps_B build of the fast loop (parallel shocks; else general pass)
        void (*kern)(const DevParams) =
            debug ? (electron ? transport_kernel<true, true, false, false> : transport_kernel<true, false, false, false>)
            : custom ? (electron ? transport_kernel<false, true, false, false, true> : transport_kernel<false, false, false, false, true>)
            : (spec && feat == 0)
                ? (slim ? (electron ? transport_kernel<false, true, false, true, false, 0> : transport_kernel<false, false, false, true, false, 0>)
                        : (electron ? transport_kernel<false, true, false, false, false, 0> : transport_kernel<false, false, false, false, false, 0>))
            : spec
                ? (slim ? (electron ? transport_kernel<false, true, false, true, false, FEAT_ETF> : transport_kernel<false, false, false, true, false, FEAT_ETF>)
                        : (electron ? transport_kernel<false, true, false, false, false, FEAT_ETF> : transport_kernel<false, false, false, false, false, FEAT_ETF>))
            : slim ? (electron ? (obl ? transport_kernel<false, true, true, true> : transport_kernel<false, true, false, true>)
                               : (obl ? transport_kernel<false, false, true, true> : transport_kernel<false, false, false, true>))
                   : (electron ? (obl ? transport_kernel<false, true, true, false> : transport_kernel<false, true, false, false>)
                               : (obl ? transport_kernel<false, false, true, false> : transport_kernel<false, false, false, false>));
        // per function and per device, not per handle: set for THIS launch (another handle may have a smaller grid)
        CU(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        CU(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        kern<<<blocks, h->block, smem, h->stream>>>(P);
        CU(cudaEventRecord(h->ev1, h->stream));
        CU(cudaGetLastError());
        double* b = h->d_tally;
        reduce_partials_kernel<<<(3 * h->ng + SC_N + 127) / 128, 128, 0, h->stream>>>(
            h->d_partials, blocks, h->ng, b + h->off_pxx, b + h->off_pxz, b + h->off_efl, b + h->off_scal);
        CU(cudaGetLastError());
        h->tm.transport_launches++; h->tm.other_launches++;
    } else {
        CU(cudaEventRecord(h->ev1, h->stream));
    }
    return MCS_OK;
}

// After a synchronisation that brought h_counters back: book-keeping of the pcut just run.
static int finish_pcut(McsHandle* h, int64_t* n_saved, int64_t* n_steps) {
    float ms = 0;
    CU(cudaEventElapsedTime(&ms, h->ev0, h->ev1));
    h->tm.transport_ms += ms;
    if (h->split_timed) {
        CU(cudaEventElapsedTime(&ms, h->ev2, h->ev3));
        h->tm.split_ms += ms;
        h->split_timed = false;
    }
    const int64_t st = (int64_t)(h->h_counters[CNT_HELIX] + h->h_counters[CNT_RETRO] - h->steps0);
    h->n_saved_last = (long long)(h->h_counters[CNT_FATE0] - h->saved0);
    h->tm.local_steps += st;
    h->tm.local_particles += h->n_use;
    h->last_steps_per_particle = h->n_use > 0 ? (double)st / (double)h->n_use : 0.0;
    h->tm.local_reds += (int64_t)(h->h_counters[CNT_RED] - h->reds0);
    if (n_saved) *n_saved = h->n_saved_last;
    if (n_steps) *n_steps = st;
    return MCS_OK;
}

extern "C" int mcs_run_pcut(McsHandle* h, int32_t i_pcut, double pcut, double pcut_prev, int64_t* n_saved, int64_t* n_steps) {
    if (!h || !h->have_ion) return fail(MCS_ERR_STATE, "mcs_begin_ion first");
    if (h->reduced) return fail(MCS_ERR_STATE, "mcs_end_ion already summed this ion's tallies: mcs_begin_ion first");
    CU(cudaSetDevice(h->device));
    int rc = launch_pcut(h, i_pcut, pcut, pcut_prev);
    if (rc) return rc;
    rc = read_counters(h);
    if (rc) return rc;
    return finish_pcut(h, n_saved, n_steps);
}

// Local part of new_pcut: order-preserving list of the saved indices (h->d_saved_idx[0..ns))
static int compact_saved(McsHandle* h) {
    const long long n = h->n_use;
    if (h->n_saved_last > 0) {
        enqueue_compaction(h->d_l_save, n, h->d_block_cnt, h->d_block_off, h->d_total, h->d_saved_idx, h->stream);
        CU(cudaGetLastError());
        h->tm.other_launches += 3;
    }
    return MCS_OK;
}

// The end of an enqueued split: ev3 closes its timing bracket (opened with ev2) and the n_out children, the first of them
// global index first_global, become the current population.
static int finish_split(McsHandle* h, long long n_out, long long first_global, int64_t* n_new_local) {
    CU(cudaEventRecord(h->ev3, h->stream));
    h->split_timed = true;
    int t = h->cur; h->cur = h->nxt; h->nxt = t;
    h->n_use = n_out; h->first_global = first_global;
    if (n_new_local) *n_new_local = n_out;
    return MCS_OK;
}

// Single-rank split, enqueued only (the caller synchronises).  ev2/ev3 bracket it.
static int split_local_async(McsHandle* h, int64_t i_mult, int64_t first_global_child, int64_t* n_new_local) {
    if (i_mult < 1) return fail(MCS_ERR_ARG, "i_mult < 1");
    const long long ns = h->n_saved_last, n_out = ns * i_mult;
    if (n_out > h->cfg.n_pts_max) return fail(MCS_ERR_ARG, "split population exceeds n_pts_max");
    int rc = check_index_range(first_global_child, n_out);
    if (rc) return rc;
    CU(cudaEventRecord(h->ev2, h->stream));
    if (ns > 0) {
        rc = compact_saved(h);
        if (rc) return rc;
        clone_kernel<<<(unsigned)((n_out + 255) / 256), 256, 0, h->stream>>>(h->pop[1], h->pop[h->nxt], h->d_saved_idx, n_out, i_mult);
        CU(cudaGetLastError());
        h->tm.other_launches++;
    }
    return finish_split(h, n_out, first_global_child, n_new_local);
}

static int sync_split_time(McsHandle* h) {
    CU(cudaStreamSynchronize(h->stream));
    if (h->split_timed) {
        float ms = 0;
        CU(cudaEventElapsedTime(&ms, h->ev2, h->ev3));
        h->tm.split_ms += ms;
        h->split_timed = false;
    }
    return MCS_OK;
}

extern "C" int mcs_split_explicit(McsHandle* h, int64_t i_mult, int64_t first_global_child, int64_t* n_new_local) {
    if (!h || !h->have_ion) return fail(MCS_ERR_STATE, "mcs_begin_ion first");
    CU(cudaSetDevice(h->device));
    int rc = split_local_async(h, i_mult, first_global_child, n_new_local);
    if (rc) return rc;
    return sync_split_time(h);
}

// Multi-GPU split with rebalancing, enqueued only: all-gather the saved records, every rank clones an equal slice of the
// GLOBAL child range.  `ns_all` = saved particles per rank (identical on every rank), so every decision below — i_mult,
// the slices, the capacity check — comes out the same everywhere and no rank can leave the collective alone.
static int split_multi_async(McsHandle* h, const long long* ns_all, int64_t n_pts_target, int64_t* n_new_local,
                             int64_t* n_new_global, int64_t* i_mult_out) {
    SplitPlan plan;
    const int pe = split_plan(ns_all, h->nranks, h->rank, n_pts_target, h->cfg.n_pts_max, &plan);
    h->n_saved_global_last = plan.S;
    if (pe == SPLIT_PLAN_BAD_RANKS) return fail(MCS_ERR_STATE, "bad rank/nranks");
    if (pe == SPLIT_PLAN_NONE_SAVED) return fail(MCS_ERR_STATE, "no saved particles to split");
    if (pe == SPLIT_PLAN_OVER_CAPACITY) return fail(MCS_ERR_ARG, "split population exceeds n_pts_max");
    if (pe == SPLIT_PLAN_OVER_RANGE) return fail(MCS_ERR_ARG, "global particle index exceeds 2^32 (RNG counter width)");
    const GatherPrefix& pre = plan.pre;
    const long long i_mult = plan.i_mult, C = plan.C, c0 = plan.c0, n_out = plan.c1 - plan.c0, stride = plan.stride;
    const size_t block_bytes = (size_t)stride * POP_REC_BYTES;
    if (block_bytes * (size_t)h->nranks > h->xchg_bytes) return fail(MCS_ERR_STATE, "split exchange buffer too small");
    CU(cudaEventRecord(h->ev2, h->stream));
    int rc = compact_saved(h);
    if (rc) return rc;
    unsigned char* mine = h->d_xchg + (size_t)h->rank * block_bytes;
    if (h->n_saved_last > 0) {
        pack_saved_kernel<<<(unsigned)((h->n_saved_last + 255) / 256), 256, 0, h->stream>>>(h->pop[1], h->d_saved_idx, h->n_saved_last,
                                                                                        mine, stride);
        CU(cudaGetLastError());
        h->tm.other_launches++;
    }
    NC(g_nccl.AllGather(mine, h->d_xchg, block_bytes, ncclUint8, h->comm, h->stream));
    if (n_out > 0) {
        clone_gathered_kernel<<<(unsigned)((n_out + 255) / 256), 256, 0, h->stream>>>(h->d_xchg, stride, pre, h->pop[h->nxt], c0, n_out,
                                                                                   i_mult);
        CU(cudaGetLastError());
        h->tm.other_launches++;
    }
    rc = finish_split(h, n_out, c0, n_new_local);
    if (rc) return rc;
    if (n_new_global) *n_new_global = C;
    if (i_mult_out) *i_mult_out = i_mult;
    return MCS_OK;
}

// ONE exchange per pcut: every rank contributes {n_saved, n_use, error flag}; all ranks get all triples.
// n_saved is computed on the device from the counter (so no host round trip is needed before the gather) when
// `from_device` is set, else taken from h->n_saved_last.
static int gather_counts(McsHandle* h, bool from_device, long long local_err, long long* ns_all, long long* used_g, long long* err_any) {
    long long all[64 * 4];
    if (from_device) {
        pack_counts_kernel<<<1, 1, 0, h->stream>>>(h->d_u64 + h->ng, h->saved0, h->n_use, local_err, h->d_gather + 4 * h->rank);
        CU(cudaGetLastError());
        h->tm.other_launches++;
    } else {
        long long v[4] = {h->n_saved_last, h->n_use, local_err, 0};
        CU(cudaMemcpyAsync(h->d_gather + 4 * h->rank, v, 32, cudaMemcpyHostToDevice, h->stream));
    }
    NC(g_nccl.AllGather(h->d_gather + 4 * h->rank, h->d_gather, 4, ncclInt64, h->comm, h->stream));
    CU(cudaMemcpyAsync(all, h->d_gather, (size_t)h->nranks * 32, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaMemcpyAsync(h->h_counters, h->d_u64 + h->ng, CNT_N * 8, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    long long u = 0, e = 0;
    for (int r = 0; r < h->nranks; r++) { ns_all[r] = all[4 * r]; u += all[4 * r + 1]; e |= all[4 * r + 2]; }
    *used_g = u; *err_any = e;
    return MCS_OK;
}

extern "C" int mcs_split(McsHandle* h, int64_t n_pts_target, int64_t* n_new_local, int64_t* n_new_global, int64_t* i_mult_out) {
    if (!h || !h->have_ion) return fail(MCS_ERR_STATE, "mcs_begin_ion first");
    CU(cudaSetDevice(h->device));
    if (h->nranks == 1) {
        const long long ns = h->n_saved_last;
        h->n_saved_global_last = ns;
        if (ns <= 0) return fail(MCS_ERR_STATE, "no saved particles to split");
        long long i_mult = n_pts_target / ns;  // cuts.jl:42
        if (i_mult < 1) i_mult = 1;
        int64_t k = 0;
        int rc = split_local_async(h, i_mult, 0, &k);
        if (rc) return rc;
        if (n_new_local) *n_new_local = k;
        if (n_new_global) *n_new_global = k;
        if (i_mult_out) *i_mult_out = i_mult;
        return sync_split_time(h);
    }
    long long ns_all[64], used_g = 0, err_any = 0;
    int rc = gather_counts(h, false, 0, ns_all, &used_g, &err_any);
    if (rc) return rc;
    rc = split_multi_async(h, ns_all, n_pts_target, n_new_local, n_new_global, i_mult_out);
    if (rc) return rc;
    return sync_split_time(h);
}

// Whole pcut loop of one ion (main_loops.jl:179-317).  Host synchronisations: ONE per pcut (the counts), none for the split.
extern "C" int mcs_run_ion(McsHandle* h, const double* pcuts, int32_t n_pcuts, double p_pcut_hi, int64_t n_pts_pcut,
                           int64_t n_pts_pcut_hi, int32_t* n_run, int64_t* n_used, int64_t* n_saved_arr) {
    if (!h || !pcuts || n_pcuts < 1 || n_pcuts > MCS_NA_C) return fail(MCS_ERR_ARG, "bad pcuts");
    if (!h->have_ion) return fail(MCS_ERR_STATE, "mcs_begin_ion first");
    if (h->reduced) return fail(MCS_ERR_STATE, "mcs_end_ion already summed this ion's tallies: mcs_begin_ion first");
    int32_t k = 0;
    CU(cudaSetDevice(h->device));
    CU(cudaEventRecord(h->ev4, h->stream));
    int rc_out = MCS_OK;
    for (int32_t i = 1; i <= n_pcuts; i++) {
        int64_t ns = 0;
        long long used_g = h->n_use, ns_g = 0, ns_all[64], err_any = 0;
        // A failure that only this rank sees must not make it leave before the exchange: it is carried as a flag
        // through the gather so that every rank returns together.
        int rc = launch_pcut(h, i, pcuts[i - 1], i > 1 ? pcuts[i - 2] : 0.0);
        if (h->nranks == 1) {
            if (rc) return rc;
            rc = read_counters(h);
            if (rc) return rc;
            rc = finish_pcut(h, &ns, nullptr);
            if (rc) return rc;
            ns_g = ns;
        } else {
            int rc2 = gather_counts(h, true, rc != MCS_OK, ns_all, &used_g, &err_any);
            if (rc2) return rc2;
            if (err_any) { rc_out = rc ? rc : fail(MCS_ERR_COMM, "another rank failed in this pcut"); break; }
            rc = finish_pcut(h, &ns, nullptr);
            if (rc) return rc;
            for (int r = 0; r < h->nranks; r++) ns_g += ns_all[r];
        }
        if (n_used) n_used[i - 1] = used_g;
        if (n_saved_arr) n_saved_arr[i - 1] = ns_g;
        k = i;
        if (ns_g == 0) break;  // pcut_finalize: break_pcut (decided on the global count: every rank takes the same branch)
        const int64_t target = pcuts[i - 1] < p_pcut_hi ? n_pts_pcut : n_pts_pcut_hi;
        if (h->nranks == 1) {
            long long i_mult = target / ns_g;  // cuts.jl:42
            if (i_mult < 1) i_mult = 1;
            h->n_saved_global_last = ns_g;
            rc = split_local_async(h, i_mult, 0, nullptr);
        } else {
            rc = split_multi_async(h, ns_all, target, nullptr, nullptr, nullptr);  // errors here are decided identically on every rank
        }
        if (rc) { rc_out = rc; break; }
    }
    CU(cudaEventRecord(h->ev5, h->stream));
    int rc = sync_split_time(h);
    if (rc) return rc;
    float ms_loop = 0;
    CU(cudaEventElapsedTime(&ms_loop, h->ev4, h->ev5));
    h->tm.ion_loop_ms += ms_loop;
    if (n_run) *n_run = k;
    return rc_out;
}

extern "C" int mcs_end_ion(McsHandle* h, McsTallies* t) {
    if (!h || !t) return fail(MCS_ERR_ARG, "null argument");
    if (!h->have_ion) return fail(MCS_ERR_STATE, "mcs_begin_ion first");
    CU(cudaSetDevice(h->device));
    // thermal log count is rank-local: read it before the counters are summed over ranks
    int rc = read_counters(h);
    if (rc) return rc;
    const long long log_claimed = (long long)h->h_counters[CNT_LOG];
    const long long n_log = log_claimed < h->cfg.na_cr ? log_claimed : h->cfg.na_cr;
    if (h->nranks > 1 && !h->reduced) {  // SURVEY 8e(ii): ONE all-reduce over the packed FP64 tallies (+ one for the integer counts)
        h->reduced = true;  // a second call returns the same sums; further pcuts need mcs_begin_ion
        CU(cudaEventRecord(h->ev2, h->stream));
        NC(g_nccl.AllReduce(h->d_tally, h->d_tally, h->n_tally, ncclFloat64, ncclSum, h->comm, h->stream));
        if (h->d_acc)  // the exact accumulators: integer sum, hence the same words on any number of ranks
            NC(g_nccl.AllReduce(h->d_acc + h->off_psd * ACC_D, h->d_acc + h->off_psd * ACC_D, (h->n_tally - h->off_psd) * ACC_D, ncclInt64,
                                ncclSum, h->comm, h->stream));
        NC(g_nccl.AllReduce(h->d_u64, h->d_u64, (size_t)(h->ng + CNT_N), ncclUint64, ncclSum, h->comm, h->stream));
        CU(cudaEventRecord(h->ev3, h->stream));
        CU(cudaStreamSynchronize(h->stream));
        float ms = 0;
        CU(cudaEventElapsedTime(&ms, h->ev2, h->ev3));
        h->tm.comm_ms += ms;
        rc = read_counters(h);
        if (rc) return rc;
    }
    CU(cudaEventRecord(h->ev2, h->stream));
    const size_t ng = (size_t)h->ng;
    double* b = h->d_tally;
    if (h->d_acc) {  // exact accumulators -> FP64 cells (everything but the flux arrays and the scalars)
        const size_t r0[2] = {h->off_psd, h->off_thsf}, r1[2] = {h->off_scal, h->off_dndp};
        for (int k = 0; k < (h->cfg.bin_thermal ? 2 : 1); k++) {
            const size_t n = r1[k] - r0[k];
            fold_accumulators_kernel<<<(unsigned)((n + 255) / 256), 256, 0, h->stream>>>(h->d_acc, r0[k], r1[k], h->d_tally);
            CU(cudaGetLastError());
            h->tm.other_launches++;
        }
    }
    if (h->cfg.bin_thermal) {
        const int M2 = h->M + 2, T2 = h->T + 2;
        sum_angle_kernel<<<(M2 * h->ng + 255) / 256, 256, 0, h->stream>>>(b + h->off_psd, M2, T2, h->ng, b + h->off_dndp);
        CU(cudaGetLastError());
        h->tm.other_launches++;
    }
#define DN(dst, src, count) do { if (dst && (count) > 0) CU(cudaMemcpyAsync(dst, src, (size_t)(count) * 8, cudaMemcpyDeviceToHost, h->stream)); } while (0)
    DN(t->pxx_flux, b + h->off_pxx, ng); DN(t->pxz_flux, b + h->off_pxz, ng); DN(t->energy_flux, b + h->off_efl, ng);
    DN(t->psd, b + h->off_psd, psd_len(h)); DN(t->num_crossings, h->d_u64, ng);
    DN(t->therm_grid, h->d_tg, n_log); DN(t->therm_px_sk, h->d_tpx, n_log); DN(t->therm_ptot_sk, h->d_tpt, n_log);
    DN(t->therm_weight, h->d_tw, n_log);
    DN(t->esc_psd_feb_upstream, b + h->off_esc_up, (size_t)E1 * E1); DN(t->esc_psd_feb_downstream, b + h->off_esc_dn, (size_t)E1 * E1);
    DN(t->esc_energy_eff, b + h->off_en_eff, E1); DN(t->esc_num_eff, b + h->off_num_eff, E1);
    DN(t->weight_coupled, b + h->off_wc, MCS_NA_C); DN(t->spectra_coupled, b + h->off_sc, (size_t)E1 * MCS_NA_C);
    DN(t->energy_transfer_pool, b + h->off_pool, ng);
    DN(t->spectra_sf, b + h->off_sf, (size_t)E1 * h->cfg.n_xspec); DN(t->spectra_pf, b + h->off_pf, (size_t)E1 * h->cfg.n_xspec);
    if (h->cfg.bin_thermal) {
        DN(t->therm_d2N_sf, b + h->off_thsf, psd_len(h)); DN(t->therm_d2N_pf, b + h->off_thpf, psd_len(h));
        DN(t->dNdp_cr_sf, b + h->off_dndp, (size_t)(h->M + 2) * ng);
    }
    double sc[SC_N];
    CU(cudaMemcpyAsync(sc, b + h->off_scal, SC_N * 8, cudaMemcpyDeviceToHost, h->stream));
#undef DN
    CU(cudaEventRecord(h->ev3, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    float ms = 0;
    CU(cudaEventElapsedTime(&ms, h->ev2, h->ev3));
    h->tm.d2h_ms += ms;
    t->n_cr_count = n_log; t->n_cr_overflow = log_claimed - n_log;
    t->esc_flux = sc[SC_ESC_FLUX]; t->px_esc_feb = sc[SC_PX_ESC_FEB]; t->energy_esc_feb = sc[SC_EN_ESC_FEB];
    t->sum_P_downstream = sc[SC_SUMP]; t->sum_KE_downstream = sc[SC_SUMKE];
    t->px_esc_upstream = sc[SC_PX_ESC_UP]; t->energy_esc_upstream = sc[SC_EN_ESC_UP];
    const unsigned long long* c = h->h_counters;
    if (env_int("MCS_SCHED_STATS", 0))
    {
        fprintf(stderr, "[mcs] lane-passes: fast %llu general %llu | warp iterations: fast %llu general %llu\n", c[CNT_FAST_LANE],
                c[CNT_SLOW_LANE], c[CNT_FAST_ITER], c[CNT_SLOW_SEC]);
        fprintf(stderr, "[mcs] lane-iterations not spent on a pass: waiting for the general section %llu, without a particle %llu, waiting for a boost %llu\n",
                c[CNT_PARK0], c[CNT_PARK0 + 1], c[CNT_PARK0 + 2]);
    }
    t->n_helix_steps = (int64_t)c[CNT_HELIX]; t->n_retro_steps = (int64_t)c[CNT_RETRO];
    t->n_warn_pperp = (int64_t)c[CNT_W_PPERP]; t->n_warn_psd_mom = (int64_t)c[CNT_W_PSDMOM]; t->n_neg_sqrt = (int64_t)c[CNT_NEGSQRT];
    t->n_retro_capped = (int64_t)c[CNT_RETRO_CAP]; t->n_errors = (int64_t)c[CNT_ERR];
    for (int i = 0; i < 6; i++) t->n_fate[i] = (int64_t)c[CNT_FATE0 + i];
    h->ended = true;
    return MCS_OK;
}

// SURVEY 8(f1): thermo_calcs.jl:31-355 on the tallies where they lie (kernel in mcs_thermo.cuh)
extern "C" int mcs_thermo(McsHandle* h, const McsThermoIn* in, double* P_par, double* P_perp, double* e_dens, double* d2N_pop) {
    if (!h || !in || !in->cos_center || !in->pt_center || !in->zone_pop) return fail(MCS_ERR_ARG, "null argument");
    if (!h->cfg.bin_thermal) return fail(MCS_ERR_ARG, "mcs_thermo needs cfg.bin_thermal = 1");
    if (!h->have_profile) return fail(MCS_ERR_STATE, "mcs_set_profile first");
    const bool resident = !(in->psd && in->therm_d2N_pf && in->num_crossings);
    if (resident && (in->psd || in->therm_d2N_pf || in->num_crossings))
        return fail(MCS_ERR_ARG, "give psd, therm_d2N_pf and num_crossings together or none of them");
    if (resident && !h->ended) return fail(MCS_ERR_STATE, "mcs_end_ion first: the tallies are not folded / summed over ranks yet");
    CU(cudaSetDevice(h->device));
    const size_t ng = (size_t)h->ng, np = psd_len(h), nT = (size_t)h->T + 1, nM = (size_t)h->M + 1;
    // one scratch allocation: slab | cos | pt | zone_pop | 4 outputs | [psd | therm | ncross]
    const size_t n_d = np + nT + nM + ng + 4 * ng + (resident ? 0 : 2 * np + ng);
    double* d = nullptr;
    CU(cudaMalloc(&d, n_d * 8));
    double *slab = d, *d_cos = slab + np, *d_pt = d_cos + nT, *d_zp = d_pt + nM, *d_out = d_zp + ng, *d_in = d_out + 4 * ng;
    cudaError_t e = cudaSuccess;
#define UP(dst, src, count) if (e == cudaSuccess) e = cudaMemcpyAsync(dst, src, (size_t)(count) * 8, cudaMemcpyHostToDevice, h->stream)
    UP(d_cos, in->cos_center, nT); UP(d_pt, in->pt_center, nM); UP(d_zp, in->zone_pop, ng);
    if (!resident) { UP(d_in, in->psd, np); UP(d_in + np, in->therm_d2N_pf, np); UP(d_in + 2 * np, in->num_crossings, ng); }
#undef UP
    ThermoParams P;
    P.ng = h->ng; P.T = h->T; P.M = h->M;
    P.c = h->cfg.c_cms; P.m = h->sp.aa * h->cfg.mp_g; P.n0 = h->sp.n0; P.gam0 = h->cfg.gam0; P.beta0 = h->cfg.beta0;
    P.temperature_K = in->temperature_K;
    P.psd_mom_min = h->P.psd_mom_min; P.bpd_mom = h->P.bpd_mom; P.psd_cos_fine = h->P.psd_cos_fine; P.delta_cos = h->P.delta_cos;
    P.psd_theta_min = h->P.psd_theta_min; P.bpd_th = h->P.bpd_th;
    P.gsf = h->P.gsf; P.ux = h->P.ux;
    P.cos_center = d_cos; P.pt_center = d_pt; P.zone_pop = d_zp;
    P.psd = resident ? h->d_tally + h->off_psd : d_in;
    P.therm_pf = resident ? h->d_tally + h->off_thpf : d_in + np;
    P.ncross = resident ? h->d_u64 : (const unsigned long long*)(d_in + 2 * np);
    P.slab = slab;
    P.P_par = d_out; P.P_perp = d_out + ng; P.e_dens = d_out + 2 * ng; P.pop = d_out + 3 * ng;
    if (e == cudaSuccess) {
        thermo_kernel<<<(unsigned)h->ng, 256, 0, h->stream>>>(P);
        e = cudaGetLastError();
        h->tm.other_launches++;
    }
#define DN(dst, k) if (e == cudaSuccess && dst) e = cudaMemcpyAsync(dst, d_out + (k) * ng, ng * 8, cudaMemcpyDeviceToHost, h->stream)
    DN(P_par, 0); DN(P_perp, 1); DN(e_dens, 2); DN(d2N_pop, 3);
#undef DN
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    cudaFree(d);
    if (e != cudaSuccess) return fail(MCS_ERR_CUDA, "mcs_thermo: %s", cudaGetErrorString(e));
    return MCS_OK;
}

extern "C" int mcs_get_population(McsHandle* h, int32_t which, int64_t n, McsPopulation* o, uint8_t* l_save) {
    if (!h || !o) return fail(MCS_ERR_ARG, "null argument");
    if (n < 0 || n > h->cfg.n_pts_max) return fail(MCS_ERR_ARG, "n out of range");
    CU(cudaSetDevice(h->device));
    const PopPtrs& p = which == 0 ? h->pop[h->cur] : h->pop[1];
    if (n > 0) {
#define X(T, name, pub) if (o->pub) CU(cudaMemcpyAsync(o->pub, p.name, (size_t)n * sizeof(T), cudaMemcpyDeviceToHost, h->stream));
        MCS_POP_FIELDS(X)
#undef X
        if (l_save) CU(cudaMemcpyAsync(l_save, h->d_l_save, (size_t)n, cudaMemcpyDeviceToHost, h->stream));
    }
    CU(cudaStreamSynchronize(h->stream));
    if (which == 1 && l_save) {  // reference zeroes the *_saved arrays (main_loops.jl:186-197): mask unsaved slots
        for (int64_t i = 0; i < n; i++) {
            if (l_save[i]) continue;
#define X(T, name, pub) if (o->pub) o->pub[i] = 0;
            MCS_POP_FIELDS(X)
#undef X
        }
    }
    return MCS_OK;
}
extern "C" int64_t mcs_population_size(McsHandle* h) { return h ? h->n_use : -1; }

extern "C" int mcs_get_fates(McsHandle* h, int64_t n, int32_t* fate, int32_t* helix, int64_t* retro, int64_t* draws) {
    if (!h || n < 0 || n > h->cfg.n_pts_max) return fail(MCS_ERR_ARG, "bad argument");
    CU(cudaSetDevice(h->device));
    if (n > 0) {
        if (fate) CU(cudaMemcpyAsync(fate, h->d_fate, (size_t)n * 4, cudaMemcpyDeviceToHost, h->stream));
        if (helix) CU(cudaMemcpyAsync(helix, h->d_helix, (size_t)n * 4, cudaMemcpyDeviceToHost, h->stream));
        if (retro) CU(cudaMemcpyAsync(retro, h->d_retro, (size_t)n * 8, cudaMemcpyDeviceToHost, h->stream));
        if (draws) CU(cudaMemcpyAsync(draws, h->d_draws, (size_t)n * 8, cudaMemcpyDeviceToHost, h->stream));
    }
    CU(cudaStreamSynchronize(h->stream));
    return MCS_OK;
}

extern "C" int mcs_replay_set_stream(McsHandle* h, const double* u, const int64_t* off, int64_t n) {
    if (!h || !u || !off || n < 0) return fail(MCS_ERR_ARG, "bad argument");
    CU(cudaSetDevice(h->device));
    cudaFree(h->d_replay_u); cudaFree(h->d_replay_off);
    h->d_replay_u = nullptr; h->d_replay_off = nullptr;
    const int64_t tot = off[n];
    CU(cudaMalloc(&h->d_replay_u, (size_t)(tot > 0 ? tot : 1) * 8));
    CU(cudaMalloc(&h->d_replay_off, (size_t)(n + 1) * 8));
    CU(cudaMemcpyAsync(h->d_replay_u, u, (size_t)tot * 8, cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(h->d_replay_off, off, (size_t)(n + 1) * 8, cudaMemcpyHostToDevice, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    h->replay_n = n;
    return MCS_OK;
}

extern "C" int mcs_trace_enable(McsHandle* h, const int64_t* idx, int32_t n_trace, int32_t max_steps) {
    if (!h || n_trace < 0 || max_steps < 0) return fail(MCS_ERR_ARG, "bad argument");
    CU(cudaSetDevice(h->device));
    cudaFree(h->d_trace_recs); cudaFree(h->d_trace_cnt);
    h->d_trace_recs = nullptr; h->d_trace_cnt = nullptr;
    h->n_trace = n_trace; h->trace_max = max_steps;
    h->trace_idx.assign(idx, idx + n_trace);
    if (n_trace == 0) return MCS_OK;
    CU(cudaMalloc(&h->d_trace_recs, (size_t)n_trace * (size_t)(max_steps > 0 ? max_steps : 1) * sizeof(McsTraceRec)));
    CU(cudaMalloc(&h->d_trace_cnt, (size_t)n_trace * 4));
    CU(cudaMemset(h->d_trace_cnt, 0, (size_t)n_trace * 4));
    return MCS_OK;
}
extern "C" int mcs_trace_get(McsHandle* h, McsTraceRec* recs, int32_t* n_rec) {
    if (!h || !h->n_trace) return fail(MCS_ERR_STATE, "trace not enabled");
    CU(cudaSetDevice(h->device));
    if (recs) CU(cudaMemcpy(recs, h->d_trace_recs, (size_t)h->n_trace * h->trace_max * sizeof(McsTraceRec), cudaMemcpyDeviceToHost));
    if (n_rec) CU(cudaMemcpy(n_rec, h->d_trace_cnt, (size_t)h->n_trace * 4, cudaMemcpyDeviceToHost));
    return MCS_OK;
}

extern "C" int mcs_get_timing(McsHandle* h, McsTiming* out, int32_t reset) {
    if (!h) return fail(MCS_ERR_ARG, "null handle");
    if (out) *out = h->tm;
    if (reset) memset(&h->tm, 0, sizeof h->tm);
    return MCS_OK;
}

extern "C" int mcs_measure_fp64_peak(McsHandle* h, double* tflops) {
    if (!h || !tflops) return fail(MCS_ERR_ARG, "null argument");
    CU(cudaSetDevice(h->device));
    const int blocks = h->n_sm * 8, threads = 256, iters = 1 << 15;
    double* d = nullptr;
    CU(cudaMalloc(&d, (size_t)blocks * threads * 8));
    double best = 0;
    for (int rep = 0; rep < 4; rep++) {
        CU(cudaEventRecord(h->ev2, h->stream));
        dfma_peak_kernel<<<blocks, threads, 0, h->stream>>>(d, iters);
        CU(cudaEventRecord(h->ev3, h->stream));
        CU(cudaStreamSynchronize(h->stream));
        float ms = 0;
        CU(cudaEventElapsedTime(&ms, h->ev2, h->ev3));
        double tf = 2.0 * 8.0 * iters * (double)blocks * threads / (ms * 1e-3) / 1e12;
        if (rep > 0 && tf > best) best = tf;
    }
    cudaFree(d);
    *tflops = best;
    return MCS_OK;
}

extern "C" int mcs_measure_atomic_peak(McsHandle* h, int64_t n_cells, double* gops) {
    if (!h || !gops || n_cells < 1) return fail(MCS_ERR_ARG, "bad argument");
    CU(cudaSetDevice(h->device));
    const int blocks = h->n_sm * 8, threads = 256, iters = 2048;
    double* d = nullptr;
    CU(cudaMalloc(&d, (size_t)n_cells * 8));
    CU(cudaMemset(d, 0, (size_t)n_cells * 8));
    double best = 0;
    for (int rep = 0; rep < 4; rep++) {
        CU(cudaEventRecord(h->ev2, h->stream));
        atomic_peak_kernel<<<blocks, threads, 0, h->stream>>>(d, n_cells, iters);
        CU(cudaEventRecord(h->ev3, h->stream));
        CU(cudaStreamSynchronize(h->stream));
        float ms = 0;
        CU(cudaEventElapsedTime(&ms, h->ev2, h->ev3));
        double g = (double)iters * blocks * threads / (ms * 1e-3) / 1e9;
        if (rep > 0 && g > best) best = g;
    }
    cudaFree(d);
    *gops = best;
    return MCS_OK;
}

extern "C" int mcs_measure_scatter_peak(McsHandle* h, double* steps_per_s) {
    if (!h || !steps_per_s) return fail(MCS_ERR_ARG, "null argument");
    CU(cudaSetDevice(h->device));
    const int blocks = h->n_sm * 2, threads = 256, iters = 20000;
    double* d = nullptr;
    CU(cudaMalloc(&d, (size_t)blocks * threads * 8));
    double best = 0;
    for (int rep = 0; rep < 4; rep++) {
        CU(cudaEventRecord(h->ev2, h->stream));
        scatter_only_kernel<<<blocks, threads, 0, h->stream>>>(d, iters, h->P.omc[0], h->P.inv_xn[0], h->P.dphi[0], h->P.key0, h->P.key1);
        CU(cudaEventRecord(h->ev3, h->stream));
        CU(cudaStreamSynchronize(h->stream));
        float ms = 0;
        CU(cudaEventElapsedTime(&ms, h->ev2, h->ev3));
        double r = (double)iters * blocks * threads / (ms * 1e-3);
        if (rep > 0 && r > best) best = r;
    }
    cudaFree(d);
    *steps_per_s = best;
    return MCS_OK;
}

extern "C" int mcs_selftest_math(McsHandle* h, int64_t n, int64_t* n_bad_sqrt, int64_t* n_bad_div) {
    if (!h || !n_bad_sqrt || !n_bad_div || n <= 0) return fail(MCS_ERR_ARG, "bad argument");
    CU(cudaSetDevice(h->device));
    unsigned long long* d = nullptr;
    unsigned long long out[2] = {0, 0};
    CU(cudaMalloc(&d, 16));
    CU(cudaMemsetAsync(d, 0, 16, h->stream));
    selftest_math_kernel<<<(unsigned)((n + 255) / 256), 256, 0, h->stream>>>((long long)n, h->P.key0, h->P.key1, d);
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(out, d, 16, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    cudaFree(d);
    *n_bad_sqrt = (int64_t)out[0]; *n_bad_div = (int64_t)out[1];
    return MCS_OK;
}
