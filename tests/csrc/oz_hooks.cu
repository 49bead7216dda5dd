// Test hooks for the tcgen05 int8 Ozaki kernels (stheno.jl_b200/csrc/ozaki.cu).
//
// A small extern "C" surface over host buffers, so that tests/test_gpu_ozaki_exact.py can drive every
// kernel instance with hand-made digit planes and compare the result with the exact NumPy model in
// oracle/device_algorithms.py.  Every call allocates device buffers, copies its inputs in, launches the
// shipped launcher on a stream of its own, synchronises, copies the outputs back and frees; it returns
// the CUDA status (0 on success, a negative value when a launcher refused) and leaves the message in
// oz_hooks_last_error().
//
// This file calls the launchers exported by libstheno_b200.so and is linked against that library; it
// adds nothing to the product ABI (include/stheno_b200.h).
#include <cstdio>
#include <vector>

#include "../../stheno.jl_b200/csrc/sb_common.cuh"

using namespace sb;

namespace {

constexpr int S = 7;          // digit planes
constexpr int KMAX = 512;     // bytes per plane row

char g_msg[512] = "";

int fail(cudaError_t e, const char* what) {
    snprintf(g_msg, sizeof g_msg, "%s: %s", what, cudaGetErrorString(e));
    return (int)e;
}
int refuse(int rc, const char* what) {
    snprintf(g_msg, sizeof g_msg, "%s returned %d", what, rc);
    return rc < 0 ? rc : -rc;
}

// device copies of the host buffers of one call, freed on scope exit
struct Dev {
    std::vector<void*> p;
    ~Dev() {
        for (void* q : p) cudaFree(q);
    }
    template <class T>
    cudaError_t in(T** d, const T* h, size_t n) {
        void* q = nullptr;
        cudaError_t e = cudaMalloc(&q, n * sizeof(T) > 0 ? n * sizeof(T) : 1);
        if (e != cudaSuccess) return e;
        p.push_back(q);
        *d = static_cast<T*>(q);
        return h ? cudaMemcpy(q, h, n * sizeof(T), cudaMemcpyHostToDevice) : cudaMemset(q, 0, n * sizeof(T));
    }
};

struct Stream {
    cudaStream_t s = nullptr;
    ~Stream() {
        if (s) cudaStreamDestroy(s);
    }
};

#define HK(call)                                       \
    do {                                               \
        cudaError_t e_ = (call);                       \
        if (e_ != cudaSuccess) return fail(e_, #call); \
    } while (0)

// launch errors of the library's own kernels surface here or at the synchronise
int finish(Stream& st) {
    HK(cudaGetLastError());
    HK(cudaStreamSynchronize(st.s));
    return 0;
}

}  // namespace

extern "C" {

const char* oz_hooks_last_error() { return g_msg; }

int oz_hooks_sm_count(int* out) {
    int dev = 0;
    HK(cudaGetDevice(&dev));
    HK(cudaDeviceGetAttribute(out, cudaDevAttrMultiProcessorCount, dev));
    return 0;
}

// launch_oz_slice.  src holds every segment (n_src doubles); segment q starts at element src_off[q] and
// has leading dimension ld[q] and row-block stride rbs[q].  planes [7][plane_rows][512], scale and expo
// [plane_rows] are in/out: what the kernels do not write comes back as it went in.
int oz_hooks_slice(const double* src, int64_t n_src, int nseg, const int64_t* src_off, const int64_t* ld,
                   const int64_t* rbs, int64_t rb_lo, int64_t nrb, int64_t out_row_base, int64_t plane_rows,
                   signed char* planes, double* scale, int* expo) {
    Dev d;
    Stream st;
    double *dsrc, *dscale;
    int* dexpo;
    signed char* dplanes;
    HK(cudaStreamCreateWithFlags(&st.s, cudaStreamNonBlocking));
    HK(d.in(&dsrc, src, (size_t)n_src));
    HK(d.in(&dplanes, planes, (size_t)S * plane_rows * KMAX));
    HK(d.in(&dscale, scale, (size_t)plane_rows));
    HK(d.in(&dexpo, expo, (size_t)plane_rows));
    OzSrc s{};
    s.nseg = nseg;
    for (int q = 0; q < nseg; q++) { s.base[q] = dsrc + src_off[q]; s.ld[q] = ld[q]; s.rbs[q] = rbs[q]; }
    launch_oz_slice(s, rb_lo, nrb, out_row_base, plane_rows, dscale, dexpo, dplanes, st.s);
    if (int rc = finish(st)) return rc;
    HK(cudaMemcpy(planes, dplanes, (size_t)S * plane_rows * KMAX, cudaMemcpyDeviceToHost));
    HK(cudaMemcpy(scale, dscale, (size_t)plane_rows * sizeof(double), cudaMemcpyDeviceToHost));
    HK(cudaMemcpy(expo, dexpo, (size_t)plane_rows * sizeof(int), cudaMemcpyDeviceToHost));
    return 0;
}

// launch_syrk_ozaki on a packed lower matrix of order Np (in/out, Np (Np + 128) / 2 doubles) with the digit
// planes [7][Np][512] and row scales [Np] given.  dbg: null, or [7][128][64] int32 (in/out) that receives
// the raw accumulators of tile 0.
int oz_hooks_syrk_packed(double* packed, int64_t Np, const signed char* planes, const double* scale, int64_t k,
                         int nseg, int64_t jlo, int64_t jhi, int rank, int world, int tma_mode, int reserve_sms,
                         int64_t tile_lo, int64_t tile_hi, int* dbg) {
    Dev d;
    Stream st;
    Packed P{nullptr, Np};
    double* dscale;
    signed char* dplanes;
    int* ddbg = nullptr;
    HK(cudaStreamCreateWithFlags(&st.s, cudaStreamNonBlocking));
    HK(d.in(&P.base, packed, (size_t)P.total()));
    HK(d.in(&dplanes, planes, (size_t)S * Np * KMAX));
    HK(d.in(&dscale, scale, (size_t)Np));
    if (dbg) HK(d.in(&ddbg, dbg, (size_t)S * 128 * 64));
    OzMaps maps;
    OzDesc desc;
    if (int rc = oz_make_maps(dplanes, Np, tma_mode, &maps)) return refuse(rc, "oz_make_maps");
    oz_default_desc(&desc, tma_mode);
    if (int rc = launch_syrk_ozaki(P, k, nseg, jlo, jhi, rank, world, &maps, dscale, &desc, tma_mode, st.s, reserve_sms,
                                   ddbg, tile_lo, tile_hi))
        return refuse(rc, "launch_syrk_ozaki");
    if (int rc = finish(st)) return rc;
    HK(cudaMemcpy(packed, P.base, (size_t)P.total() * sizeof(double), cudaMemcpyDeviceToHost));
    if (dbg) HK(cudaMemcpy(dbg, ddbg, (size_t)S * 128 * 64 * sizeof(int), cudaMemcpyDeviceToHost));
    return 0;
}

// launch_gemm_ozaki: C[M x Ncols] (column-major, ldc, in/out) -= A B^T, A = plane rows [rowA0, rowA0 + M) of
// the set (planesA [7][rowsA][512], scaleA [rowsA]), B = plane rows [rowB0, rowB0 + Ncols) of the B set.
int oz_hooks_gemm_plain(double* C, int64_t ldc, int64_t M, int64_t Ncols, int nseg, const signed char* planesA,
                        const double* scaleA, int64_t rowsA, int64_t rowA0, const signed char* planesB,
                        const double* scaleB, int64_t rowsB, int64_t rowB0, int tma_mode) {
    Dev d;
    Stream st;
    double *dC, *dsA, *dsB;
    signed char *dpA, *dpB;
    HK(cudaStreamCreateWithFlags(&st.s, cudaStreamNonBlocking));
    HK(d.in(&dC, C, (size_t)ldc * Ncols));
    HK(d.in(&dpA, planesA, (size_t)S * rowsA * KMAX));
    HK(d.in(&dsA, scaleA, (size_t)rowsA));
    HK(d.in(&dpB, planesB, (size_t)S * rowsB * KMAX));
    HK(d.in(&dsB, scaleB, (size_t)rowsB));
    OzMaps mA, mB;
    OzDesc desc;
    if (int rc = oz_make_maps(dpA, rowsA, tma_mode, &mA)) return refuse(rc, "oz_make_maps(A)");
    if (int rc = oz_make_maps(dpB, rowsB, tma_mode, &mB)) return refuse(rc, "oz_make_maps(B)");
    oz_default_desc(&desc, tma_mode);
    if (int rc = launch_gemm_ozaki(dC, ldc, M, Ncols, nseg, &mA, dsA, rowA0, &mB, dsB, rowB0, &desc, tma_mode, st.s))
        return refuse(rc, "launch_gemm_ozaki");
    if (int rc = finish(st)) return rc;
    HK(cudaMemcpy(C, dC, (size_t)ldc * Ncols * sizeof(double), cudaMemcpyDeviceToHost));
    return 0;
}

// launch_panel_solve_ozaki: X[M x 512] = A W^T written over four block columns X[q] (column-major, ldx[q] >= M,
// 128 columns each, in/out), A = plane rows [rowA0, rowA0 + M) of (planesA, scaleA), W = the 512 plane rows of
// (planesW [7][512][512], scaleW [512]).
int oz_hooks_panel_solve(double* const* X, const int64_t* ldx, int64_t M, const signed char* planesA,
                         const double* scaleA, int64_t rowsA, int64_t rowA0, const signed char* planesW,
                         const double* scaleW) {
    constexpr int64_t WD = 4 * NB;
    Dev d;
    Stream st;
    double* dX[4];
    double *dsA, *dsW;
    signed char *dpA, *dpW;
    HK(cudaStreamCreateWithFlags(&st.s, cudaStreamNonBlocking));
    for (int q = 0; q < 4; q++) HK(d.in(&dX[q], X[q], (size_t)ldx[q] * NB));
    HK(d.in(&dpA, planesA, (size_t)S * rowsA * KMAX));
    HK(d.in(&dsA, scaleA, (size_t)rowsA));
    HK(d.in(&dpW, planesW, (size_t)S * WD * KMAX));
    HK(d.in(&dsW, scaleW, (size_t)WD));
    OzMaps mA, mW;
    OzDesc desc;
    if (int rc = oz_make_maps(dpA, rowsA, 8, &mA)) return refuse(rc, "oz_make_maps(A)");
    if (int rc = oz_make_maps(dpW, WD, 8, &mW)) return refuse(rc, "oz_make_maps(W)");
    oz_default_desc(&desc, 8);
    if (int rc = launch_panel_solve_ozaki(dX, ldx, M, &mA, dsA, rowA0, &mW, dsW, &desc, st.s))
        return refuse(rc, "launch_panel_solve_ozaki");
    if (int rc = finish(st)) return rc;
    for (int q = 0; q < 4; q++)
        HK(cudaMemcpy(X[q], dX[q], (size_t)ldx[q] * NB * sizeof(double), cudaMemcpyDeviceToHost));
    return 0;
}

}  // extern "C"
