// Standalone timing of the tcgen05 int8-Ozaki trailing update (stheno.jl_b200/csrc/ozaki.cu) next to the
// fp64 DMMA trailing kernel (gemm_nt.cu) on the same panels.  Correctness of every kernel instance is
// tests/test_gpu_ozaki_exact.py (bit-for-bit against the exact model).  Build: tools/Makefile (links build/*.o).
//   oz_test [Np=16384] [nseg=4]     (OZ_TEST_RESERVE: see below)
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "../stheno.jl_b200/csrc/sb_common.cuh"

using namespace sb;

#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e_), __FILE__, __LINE__); return 1; } } while (0)

static double urand(uint64_t& s) {
    s = s * 6364136223846793005ULL + 1442695040888963407ULL;
    return (double)(s >> 11) / 9007199254740992.0;
}

struct Problem {
    int64_t Np, nblk, k0;
    int nseg;
    double* dP[4] = {nullptr, nullptr, nullptr, nullptr};
    const double** dPt = nullptr;  // device array of panel pointers
    double *A1 = nullptr, *A2 = nullptr;
    double* scale = nullptr;
    int* expo = nullptr;
    signed char* planes = nullptr;
    Packed P1, P2;
};

static int setup(Problem& pr, int64_t Np, int nseg) {
    pr.Np = Np; pr.nblk = Np / NB; pr.k0 = 0; pr.nseg = nseg;
    const int64_t pe = tiled_panel_elems(Np);
    uint64_t seed = 12345;
    std::vector<double> hP(pe);
    for (int q = 0; q < nseg; q++) {
        std::fill(hP.begin(), hP.end(), 0.0);
        for (int64_t rb = 0; rb < pr.nblk; rb++)
            for (int k = 0; k < NB; k++)
                for (int r = 0; r < NB; r++) {
                    // rows with very different magnitudes + a few exact zeros / tiny values
                    double mag = std::pow(10.0, -3.0 * ((rb * NB + r) % 7) / 7.0) * ((r % 13 == 5) ? 1e-6 : 1.0);
                    double v = (urand(seed) * 2 - 1) * mag;
                    if ((r + k) % 97 == 0) v = 0.0;
                    hP[((rb * NB + k) * (int64_t)(NB + 4)) + r] = v;
                }
        CK(cudaMalloc(&pr.dP[q], pe * 8));
        CK(cudaMemcpy(pr.dP[q], hP.data(), pe * 8, cudaMemcpyHostToDevice));
    }
    CK(cudaMalloc(&pr.dPt, 4 * sizeof(double*)));
    CK(cudaMemcpy(pr.dPt, pr.dP, 4 * sizeof(double*), cudaMemcpyHostToDevice));
    pr.P1.Np = pr.P2.Np = Np;
    const int64_t tot = pr.P1.total();
    CK(cudaMalloc(&pr.A1, tot * 8));
    CK(cudaMalloc(&pr.A2, tot * 8));
    {
        std::vector<double> h(tot);
        for (int64_t i = 0; i < tot; i++) h[i] = urand(seed) * 2 - 1;
        CK(cudaMemcpy(pr.A1, h.data(), tot * 8, cudaMemcpyHostToDevice));
        CK(cudaMemcpy(pr.A2, h.data(), tot * 8, cudaMemcpyHostToDevice));
    }
    pr.P1.base = pr.A1; pr.P2.base = pr.A2;
    CK(cudaMalloc(&pr.scale, Np * 8));
    CK(cudaMalloc(&pr.expo, Np * 4));
    CK(cudaMalloc(&pr.planes, oz_planes_bytes(Np)));
    CK(cudaMemset(pr.planes, 0, oz_planes_bytes(Np)));
    CK(cudaMemset(pr.scale, 0, Np * 8));
    return 0;
}

static void teardown(Problem& pr) {
    for (int q = 0; q < 4; q++) if (pr.dP[q]) cudaFree(pr.dP[q]);
    cudaFree(pr.dPt); cudaFree(pr.A1); cudaFree(pr.A2); cudaFree(pr.scale); cudaFree(pr.expo); cudaFree(pr.planes);
}

// OZ_TEST_RESERVE: > 0 leaves that many SMs free (persistent grid), < 0 launches chunked CTAs of -value tiles
static int g_reserve = 0;

int main(int argc, char** argv) {
    if (getenv("OZ_TEST_RESERVE")) g_reserve = atoi(getenv("OZ_TEST_RESERVE"));
    const int64_t NpT = argc > 1 ? atoll(argv[1]) : 16384;
    const int nseg = argc > 2 ? atoi(argv[2]) : 4;
    cudaStream_t st;
    CK(cudaStreamCreate(&st));
    {
        Problem pr;
        if (setup(pr, NpT, nseg)) return 1;
        const int64_t jt = nseg;
        const double* Pt[4] = {pr.dP[0], pr.dP[1], pr.dP[2], pr.dP[3]};
        const double tiles = (double)syrk_packed_tiles(pr.nblk, 0, jt, pr.nblk, 0, 1);
        const double flops = tiles * 2.0 * NB * NB * (128.0 * nseg);
        cudaEvent_t e0, e1;
        cudaEventCreate(&e0); cudaEventCreate(&e1);
        float ms;
        for (int rep = 0; rep < 3; rep++) {
            cudaEventRecord(e0, st);
            launch_syrk_packed(pr.P1, 0, Pt, nseg, jt, pr.nblk, 0, 1, st);
            cudaEventRecord(e1, st);
            CK(cudaStreamSynchronize(st));
            cudaEventElapsedTime(&ms, e0, e1);
            printf("[time] Np=%lld DMMA   %.3f ms  %.2f TFLOP/s\n", (long long)NpT, ms, flops / ms * 1e-9);
        }
        cudaEventRecord(e0, st);
        launch_oz_slice(oz_src_tiled(Pt, nseg), nseg - 1, pr.nblk - nseg, (int64_t)NB, NpT, pr.scale, pr.expo, pr.planes, st);
        cudaEventRecord(e1, st);
        CK(cudaStreamSynchronize(st));
        cudaEventElapsedTime(&ms, e0, e1);
        printf("[time] slice kernels %.3f ms\n", ms);
        for (int mode : {8, 12, 16}) {
            OzMaps maps; OzDesc d;
            if (oz_make_maps(pr.planes, NpT, mode, &maps)) { printf("map fail\n"); continue; }
            oz_default_desc(&d, mode);
            for (int rep = 0; rep < 3; rep++) {
                cudaEventRecord(e0, st);
                launch_syrk_ozaki(pr.P2, 0, nseg, jt, pr.nblk, 0, 1, &maps, pr.scale, &d, mode, st, g_reserve);
                cudaEventRecord(e1, st);
                cudaError_t e = cudaStreamSynchronize(st);
                if (e != cudaSuccess) { printf("ozaki timing run failed: %s\n", cudaGetErrorString(e)); return 3; }
                cudaEventElapsedTime(&ms, e0, e1);
                printf("[time] Np=%lld OZAKI(mode %d) %.3f ms  %.2f TFLOP/s fp64-equivalent (%.0f int8 TOP/s)\n", (long long)NpT,
                       mode, ms, flops / ms * 1e-9, flops * 28 / ms * 1e-9);
            }
        }
        teardown(pr);
    }
    return 0;
}
