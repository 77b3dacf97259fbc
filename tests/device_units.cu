// Device unit harness: the primitives of csrc/mcs_device.cuh and csrc/mcs_math.cuh called one by one, so that
// tests/test_device_units.py can hold each to an exact reference.  It includes the header itself and is built with the
// library's flags (FMA contraction on), so it runs exactly the code the library inlines.  Every entry point copies its
// inputs in, runs one kernel, copies the results out and returns the CUDA error code.
#include <cstring>

#include "../montecarloscattering.jl_b200/csrc/mcs_device.cuh"

using namespace mcs;

namespace {

constexpr int TPB = 256;
unsigned blocks(long n) { return (unsigned)((n + TPB - 1) / TPB); }

__global__ void k_acc_add(const __grid_constant__ DevParams P, const long long* cell, const double* v, long n) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) acc_add(P, (size_t)cell[i], v[i]);
}
__global__ void k_az_sincos(const double2* tab, const uint32_t* hi, const uint32_t* lo, long n, double* s, double* c) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) az_sincos(tab, hi[i], lo[i], s[i], c[i]);
}
// y0 = rsqrt_nr(x), y1 = x * rsqrt_nr(x) (the fast loop's square root), y2 = sqrt_nr(x)
__global__ void k_roots(const double* x, long n, double* y0, double* y1, double* y2) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double r = rsqrt_nr(x[i]);
    y0[i] = r; y1[i] = x[i] * r; y2[i] = sqrt_nr(x[i]);
}
__global__ void k_sincos_bf(const double* x, long n, double* s, double* c) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) sincos_bf(x[i], &s[i], &c[i]);
}
template <bool NR>
__global__ void k_asin_bf(const double* x, long n, double* y) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) y[i] = asin_bf<NR>(x[i]);
}

// The split entry points take and return populations as three host arrays: the f64 fields, the i64 fields and the u8
// fields, each field `cap` records long, in PopPtrs order.  They are the three consecutive byte ranges of one population
// block of pop_view's layout, at[k]..at[k + 1], which start at its first field of each type.
struct PopRanges {
    unsigned char* at[4];
    PopRanges(unsigned char* block, long long cap) {
        const PopPtrs v = pop_view(block, cap, 0);
        at[0] = reinterpret_cast<unsigned char*>(v.weight); at[1] = reinterpret_cast<unsigned char*>(v.grid); at[2] = v.down;
        at[3] = block + (size_t)cap * POP_REC_BYTES;
    }
};

// device buffers of one call, freed on every path out
struct Bufs {
    void* p[16] = {};
    int n = 0;
    cudaError_t err = cudaSuccess;
    template <class T> T* in(const T* h, size_t count) {
        T* d = alloc<T>(count);
        if (d && h) err = cudaMemcpy(d, h, count * sizeof(T), cudaMemcpyHostToDevice);
        return err == cudaSuccess ? d : nullptr;
    }
    template <class T> T* alloc(size_t count) {
        if (err != cudaSuccess) return nullptr;
        void* d = nullptr;
        err = cudaMalloc(&d, count ? count * sizeof(T) : 1);
        if (err == cudaSuccess) err = cudaMemset(d, 0, count ? count * sizeof(T) : 1);
        if (err != cudaSuccess) return nullptr;
        p[n++] = d;
        return static_cast<T*>(d);
    }
    template <class T> void out(T* h, const T* d, size_t count) {
        if (err == cudaSuccess) err = cudaMemcpy(h, d, count * sizeof(T), cudaMemcpyDeviceToHost);
    }
    // a population block of `cap` records from the three host arrays (PopRanges), and back
    unsigned char* pop_in(const double* f64, const long long* i64, const uint8_t* u8, long long cap) {
        unsigned char* d = alloc<unsigned char>((size_t)cap * POP_REC_BYTES);
        if (!d) return nullptr;
        const PopRanges r(d, cap);
        const void* h[3] = {f64, i64, u8};
        for (int k = 0; k < 3; k++)
            if (err == cudaSuccess && r.at[k + 1] > r.at[k]) err = cudaMemcpy(r.at[k], h[k], r.at[k + 1] - r.at[k], cudaMemcpyHostToDevice);
        return err == cudaSuccess ? d : nullptr;
    }
    void pop_out(double* f64, long long* i64, uint8_t* u8, unsigned char* d, long long cap) {
        const PopRanges r(d, cap);
        void* h[3] = {f64, i64, u8};
        for (int k = 0; k < 3; k++)
            if (err == cudaSuccess && r.at[k + 1] > r.at[k]) err = cudaMemcpy(h[k], r.at[k], r.at[k + 1] - r.at[k], cudaMemcpyDeviceToHost);
    }
    int launched() {
        if (err == cudaSuccess) err = cudaGetLastError();
        if (err == cudaSuccess) err = cudaDeviceSynchronize();
        return err;
    }
    ~Bufs() { for (int i = 0; i < n; i++) cudaFree(p[i]); }
};

}  // namespace

extern "C" {

// acc_add of v[i] into cell[i] of n_cells zeroed accumulator cells; returns the words (n_cells x ACC_D) and CNT_ERR
int du_acc_add(const long long* cell, const double* v, long n, long n_cells, long long* words, unsigned long long* n_err) {
    Bufs b;
    const long long* d_cell = b.in(cell, n);
    const double* d_v = b.in(v, n);
    long long* d_acc = b.alloc<long long>((size_t)n_cells * ACC_D);
    unsigned long long* d_cnt = b.alloc<unsigned long long>(CNT_N);
    if (b.err) return b.err;
    DevParams P;
    memset(&P, 0, sizeof P);
    P.t.acc = d_acc; P.t.tally_base = nullptr; P.t.counters = d_cnt;
    if (n > 0) k_acc_add<<<blocks(n), TPB>>>(P, d_cell, d_v, n);
    b.launched();
    b.out(words, d_acc, (size_t)n_cells * ACC_D);
    b.out(n_err, d_cnt + CNT_ERR, 1);
    return b.err;
}

// fold_accumulators_kernel over n_cells cells of ACC_D words each
int du_fold(const long long* words, long n_cells, double* out) {
    Bufs b;
    const long long* d_acc = b.in(words, (size_t)n_cells * ACC_D);
    double* d_out = b.alloc<double>(n_cells);
    if (b.err) return b.err;
    fold_accumulators_kernel<<<blocks(n_cells), TPB>>>(d_acc, 0, (size_t)n_cells, d_out);
    b.launched();
    b.out(out, d_out, n_cells);
    return b.err;
}

// the library's azimuth table (az_table) and az_sincos on it
int du_az_table(double* tab) {
    az_table(reinterpret_cast<double2*>(tab));
    return 0;
}
int du_az_sincos(const uint32_t* hi, const uint32_t* lo, long n, double* s, double* c) {
    double2 tab[AZ_N];
    az_table(tab);
    Bufs b;
    const double2* d_tab = b.in(tab, AZ_N);
    const uint32_t* d_hi = b.in(hi, n);
    const uint32_t* d_lo = b.in(lo, n);
    double* d_s = b.alloc<double>(n);
    double* d_c = b.alloc<double>(n);
    if (b.err) return b.err;
    k_az_sincos<<<blocks(n), TPB>>>(d_tab, d_hi, d_lo, n, d_s, d_c);
    b.launched();
    b.out(s, d_s, n); b.out(c, d_c, n);
    return b.err;
}

int du_roots(const double* x, long n, double* rsqrt, double* sqrt_rsqrt, double* sqrt_nr_out) {
    Bufs b;
    const double* d_x = b.in(x, n);
    double* d_0 = b.alloc<double>(n);
    double* d_1 = b.alloc<double>(n);
    double* d_2 = b.alloc<double>(n);
    if (b.err) return b.err;
    k_roots<<<blocks(n), TPB>>>(d_x, n, d_0, d_1, d_2);
    b.launched();
    b.out(rsqrt, d_0, n); b.out(sqrt_rsqrt, d_1, n); b.out(sqrt_nr_out, d_2, n);
    return b.err;
}

int du_sincos_bf(const double* x, long n, double* s, double* c) {
    Bufs b;
    const double* d_x = b.in(x, n);
    double* d_s = b.alloc<double>(n);
    double* d_c = b.alloc<double>(n);
    if (b.err) return b.err;
    k_sincos_bf<<<blocks(n), TPB>>>(d_x, n, d_s, d_c);
    b.launched();
    b.out(s, d_s, n); b.out(c, d_c, n);
    return b.err;
}

// asin_bf<nr != 0>
int du_asin_bf(const double* x, long n, int nr, double* y) {
    Bufs b;
    const double* d_x = b.in(x, n);
    double* d_y = b.alloc<double>(n);
    if (b.err) return b.err;
    if (nr) k_asin_bf<true><<<blocks(n), TPB>>>(d_x, n, d_y);
    else k_asin_bf<false><<<blocks(n), TPB>>>(d_x, n, d_y);
    b.launched();
    b.out(y, d_y, n);
    return b.err;
}

// ---------------------------------------------------------------------------------------------------------------------
// The split of new_pcut.  Populations are held in blocks of pop_view's layout, as in the library.

// enqueue_compaction on l_save[0..n): saved_idx gets all n entries (zero past *total)
int du_compact(const uint8_t* l_save, long n, long long* saved_idx, long long* total) {
    Bufs b;
    const uint8_t* d_l = b.in(l_save, n);
    const long long nb = compaction_blocks(n);
    int* d_cnt = b.alloc<int>(nb);
    long long* d_off = b.alloc<long long>(nb);
    long long* d_total = b.alloc<long long>(1);
    long long* d_idx = b.alloc<long long>(n);
    if (b.err) return b.err;
    if (n > 0) enqueue_compaction(d_l, n, d_cnt, d_off, d_total, d_idx, 0);
    b.launched();
    b.out(total, d_total, 1);
    b.out(saved_idx, d_idx, n);
    return b.err;
}

// the single-rank split (the library's split_local_async): compaction, then clone_kernel into n_out = *total * i_mult
// children; fails with cudaErrorInvalidValue if they do not fit in `cap` records
int du_split_local(const double* f64, const long long* i64, const uint8_t* u8, const uint8_t* l_save, long n, long i_mult,
                   long cap, double* out_f64, long long* out_i64, uint8_t* out_u8, long long* total) {
    if (i_mult < 1) return cudaErrorInvalidValue;
    Bufs b;
    unsigned char* d_pop = b.pop_in(f64, i64, u8, n);
    const uint8_t* d_l = b.in(l_save, n);
    const long long nb = compaction_blocks(n);
    int* d_cnt = b.alloc<int>(nb);
    long long* d_off = b.alloc<long long>(nb);
    long long* d_total = b.alloc<long long>(1);
    long long* d_idx = b.alloc<long long>(n);
    unsigned char* o_pop = b.alloc<unsigned char>((size_t)cap * POP_REC_BYTES);
    if (b.err) return b.err;
    if (n > 0) enqueue_compaction(d_l, n, d_cnt, d_off, d_total, d_idx, 0);
    b.launched();
    b.out(total, d_total, 1);
    if (b.err) return b.err;
    const long long n_out = *total * i_mult;
    if (n_out > cap) return cudaErrorInvalidValue;
    if (n_out > 0)
        clone_kernel<<<blocks(n_out), TPB>>>(pop_view(d_pop, n, 0), pop_view(o_pop, cap, 0), d_idx, n_out, i_mult);
    b.launched();
    b.pop_out(out_f64, out_i64, out_u8, o_pop, cap);
    return b.err;
}

// The rebalancing split (the library's split_multi_async) of `nranks` ranks emulated on one device; rank q holds records
// [first_q, first_q + n_per_rank[q]) of the concatenated population.  Each rank compacts its own l_save, which gives
// ns_all, and plans with split_plan; rank q packs its saved records into block q of one exchange buffer, which is then
// byte for byte what the all-gather leaves on every rank; then every rank clones its slice [c0, c1) of the global child
// range out of it.  The slices land at records [c0, c1) of the output (cap records), n_out[r] = c1 - c0.  A refused plan
// or C > cap gives cudaErrorInvalidValue.
int du_split_ranks(int nranks, const long long* n_per_rank, const uint8_t* l_save, const double* f64, const long long* i64,
                   const uint8_t* u8, long long target, long long n_pts_max, long cap, double* out_f64, long long* out_i64,
                   uint8_t* out_u8, long long* n_out, long long* i_mult) {
    if (nranks < 1 || nranks > 64) return cudaErrorInvalidValue;
    long long first[65] = {0}, nb_max = 1;
    for (int q = 0; q < nranks; q++) {
        first[q + 1] = first[q] + n_per_rank[q];
        if (compaction_blocks(n_per_rank[q]) > nb_max) nb_max = compaction_blocks(n_per_rank[q]);
    }
    const long long N = first[nranks];
    Bufs b;
    unsigned char* d_pop = b.pop_in(f64, i64, u8, N);
    const uint8_t* d_l = b.in(l_save, N);
    int* d_cnt = b.alloc<int>(nb_max);
    long long* d_off = b.alloc<long long>(nb_max);
    long long* d_total = b.alloc<long long>(nranks);
    long long* d_idx = b.alloc<long long>(N);
    if (b.err) return b.err;
    for (int q = 0; q < nranks; q++)
        if (n_per_rank[q] > 0) enqueue_compaction(d_l + first[q], n_per_rank[q], d_cnt, d_off, d_total + q, d_idx + first[q], 0);
    b.launched();
    long long ns_all[64];
    b.out(ns_all, d_total, nranks);
    if (b.err) return b.err;
    SplitPlan plan[64];
    for (int r = 0; r < nranks; r++)
        if (split_plan(ns_all, nranks, r, target, n_pts_max, &plan[r]) != SPLIT_PLAN_OK) return cudaErrorInvalidValue;
    const long long stride = plan[0].stride;
    if (plan[0].C > cap) return cudaErrorInvalidValue;
    unsigned char* d_x = b.alloc<unsigned char>((size_t)nranks * (size_t)stride * POP_REC_BYTES);
    unsigned char* o_pop = b.alloc<unsigned char>((size_t)cap * POP_REC_BYTES);
    if (b.err) return b.err;
    for (int q = 0; q < nranks; q++)
        if (ns_all[q] > 0)
            pack_saved_kernel<<<blocks(ns_all[q]), TPB>>>(pop_view(d_pop, N, first[q]), d_idx + first[q], ns_all[q],
                                                          d_x + (size_t)q * (size_t)stride * POP_REC_BYTES, stride);
    for (int r = 0; r < nranks; r++) {
        n_out[r] = plan[r].c1 - plan[r].c0;
        if (n_out[r] > 0)
            clone_gathered_kernel<<<blocks(n_out[r]), TPB>>>(d_x, stride, plan[r].pre, pop_view(o_pop, cap, plan[r].c0), plan[r].c0,
                                                             n_out[r], plan[r].i_mult);
    }
    b.launched();
    b.pop_out(out_f64, out_i64, out_u8, o_pop, cap);
    *i_mult = plan[0].i_mult;
    return b.err;
}

// split_plan alone (host code, no device needed): returns its SplitPlanError; out = {S, i_mult, C, c0, c1, stride},
// start = the gather prefix start[0..nranks]
int du_split_plan(const long long* ns_all, int nranks, int rank, long long target, long long n_pts_max, long long* out,
                  long long* start) {
    SplitPlan p;
    const int rc = split_plan(ns_all, nranks, rank, target, n_pts_max, &p);
    const long long v[6] = {p.S, p.i_mult, p.C, p.c0, p.c1, p.stride};
    memcpy(out, v, sizeof v);
    if (p.pre.nranks > 0) memcpy(start, p.pre.start, (size_t)(p.pre.nranks + 1) * sizeof(long long));
    return rc;
}

}  // extern "C"
