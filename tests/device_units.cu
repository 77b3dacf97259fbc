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

// device buffers of one call, freed on every path out
struct Bufs {
    void* p[8] = {};
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

}  // extern "C"
