// gather_probe — what bounds the SpMV over the gapped array: the stream or the per-cell gathers of x?
// Synthetic stand-in for config 2: 2^24 cells, 60 % live, keys uniform in [1, 1e5], x = 1e5 doubles (800 KB, L2-resident).
// Variants of (cell format) x (gather path); each prints its time per launch.  Build: nvcc -O3 -gencode arch=compute_100a,code=sm_100a
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <vector>
#include "../dynamicsparsearrays.jl_b200/csrc/pcsr.cuh"   // the product kernels, timed on the same synthetic arrays
namespace dsa { Prof& prof() { static Prof p; return p; } DevicePool& device_pool(int) { static DevicePool* p = new DevicePool(); return *p; } }

#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { printf("%s: %s\n", #x, cudaGetErrorString(e)); exit(1); } } while (0)

enum { G_NONE = 0, G_LDG = 1, G_CG = 2, G_TEX = 3, G_SMEM = 4, G_NOALLOC = 5 };

__device__ __forceinline__ double ld_cg(const double* p) {
    double v;
    asm volatile("ld.global.cg.f64 %0, [%1];" : "=d"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ double ld_noalloc(const double* p) {
    double v;
    asm volatile("ld.global.nc.L1::no_allocate.f64 %0, [%1];" : "=d"(v) : "l"(p));
    return v;
}

template <typename KEY, int GATHER, int STEPS>
__global__ void __launch_bounds__(1024) k_probe(const KEY* __restrict__ keys, const double* __restrict__ vals, int64_t cap,
                                               const double* __restrict__ x, cudaTextureObject_t tx, int nx, int nsm,
                                               double* __restrict__ out) {
    extern __shared__ double sx[];
    if (GATHER == G_SMEM) {
        for (int i = threadIdx.x; i < nsm; i += blockDim.x) sx[i] = x[i];
        __syncthreads();
    }
    const int lane = threadIdx.x & 31;
    const int64_t nchunks = cap / (32 * STEPS);
    const int64_t wstride = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t chunk = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; chunk < nchunks; chunk += wstride) {
        const int64_t base = chunk * 32 * STEPS;
        KEY k[STEPS];
        double t[STEPS];
#pragma unroll
        for (int s = 0; s < STEPS; ++s) {
            k[s] = __ldcs(keys + base + s * 32 + lane);
            t[s] = __ldcs(vals + base + s * 32 + lane);
        }
        double acc = 0.0;
#pragma unroll
        for (int s = 0; s < STEPS; ++s) {
            const int64_t kk = (int64_t)k[s];
            if (kk > 0) {
                double xv = 1.0;
                if (GATHER == G_LDG) xv = __ldg(x + (kk - 1));
                if (GATHER == G_CG) xv = ld_cg(x + (kk - 1));
                if (GATHER == G_NOALLOC) xv = ld_noalloc(x + (kk - 1));
                if (GATHER == G_TEX) {
                    const int2 r = tex1Dfetch<int2>(tx, (int)(kk - 1));
                    xv = __hiloint2double(r.y, r.x);
                }
                if (GATHER == G_SMEM) xv = (kk - 1 < nsm) ? sx[kk - 1] : __ldg(x + (kk - 1));
                acc += xv * t[s];
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (lane == 0) out[chunk] = acc;
    }
}

template <typename KEY, int GATHER, int STEPS>
static void run(const char* name, const KEY* keys, const double* vals, int64_t cap, const double* x, cudaTextureObject_t tx, int nx, int nsm,
                double* out, int grid, size_t smem, double bytes, int block = 256) {
    if (smem > 48 * 1024) CK(cudaFuncSetAttribute(k_probe<KEY, GATHER, STEPS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0));
    CK(cudaEventCreate(&e1));
    for (int i = 0; i < 3; ++i) k_probe<KEY, GATHER, STEPS><<<grid, block, smem>>>(keys, vals, cap, x, tx, nx, nsm, out);
    CK(cudaDeviceSynchronize());
    const int reps = 20;
    CK(cudaEventRecord(e0));
    for (int i = 0; i < reps; ++i) k_probe<KEY, GATHER, STEPS><<<grid, block, smem>>>(keys, vals, cap, x, tx, nx, nsm, out);
    CK(cudaEventRecord(e1));
    CK(cudaDeviceSynchronize());
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, e0, e1));
    const double us = 1e3 * ms / reps;
    printf("%-44s grid %6d smem %6zu : %8.2f us  stream %7.1f GB/s\n", name, grid, smem, us, bytes / us * 1e-3);
}

int main() {
    const int64_t cap = 1 << 24;
    const int nx = 100000;
    std::vector<int64_t> hk(cap);
    std::vector<int32_t> hk32(cap);
    std::vector<double> hv(cap), hx(nx);
    uint64_t s = 88172645463325252ull;
    auto rnd = [&]() { s ^= s << 13; s ^= s >> 7; s ^= s << 17; return s; };
    for (int64_t i = 0; i < cap; ++i) {
        const bool live = (rnd() % 1000) < 602;
        const int64_t k = live ? (int64_t)(rnd() % nx) + 1 : INT64_MIN;
        hk[i] = k;
        hk32[i] = live ? (int32_t)k : INT32_MIN;
        hv[i] = (double)(rnd() % 1000) * 1e-3;
    }
    for (int i = 0; i < nx; ++i) hx[i] = (double)(rnd() % 1000) * 1e-3;
    int64_t* dk; int32_t* dk32; double *dv, *dx, *dout;
    CK(cudaMalloc(&dk, cap * 8)); CK(cudaMalloc(&dk32, cap * 4)); CK(cudaMalloc(&dv, cap * 8)); CK(cudaMalloc(&dx, nx * 8));
    CK(cudaMalloc(&dout, (cap / 32) * 8));
    CK(cudaMemcpy(dk, hk.data(), cap * 8, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dk32, hk32.data(), cap * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dv, hv.data(), cap * 8, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dx, hx.data(), nx * 8, cudaMemcpyHostToDevice));
    cudaResourceDesc rd = {};
    rd.resType = cudaResourceTypeLinear;
    rd.res.linear.devPtr = dx;
    rd.res.linear.desc = cudaCreateChannelDesc<int2>();
    rd.res.linear.sizeInBytes = (size_t)nx * 8;
    cudaTextureDesc td = {};
    td.readMode = cudaReadModeElementType;
    cudaTextureObject_t tx = 0;
    CK(cudaCreateTextureObject(&tx, &rd, &td, nullptr));
    int nsmc = 0;
    CK(cudaDeviceGetAttribute(&nsmc, cudaDevAttrMultiProcessorCount, 0));
    const double b16 = 16.0 * cap, b12 = 12.0 * cap;
    const int full4 = (int)(cap / (32 * 4) / 8), full8 = (int)(cap / (32 * 8) / 8);
    printf("SMs %d\n", nsmc);
    run<int64_t, G_NONE, 4>("i64 keys, stream only, 4 steps", dk, dv, cap, dx, tx, nx, 0, dout, full4, 0, b16);
    run<int32_t, G_NONE, 4>("i32 keys, stream only, 4 steps", dk32, dv, cap, dx, tx, nx, 0, dout, full4, 0, b12);
    run<int32_t, G_NONE, 8>("i32 keys, stream only, 8 steps", dk32, dv, cap, dx, tx, nx, 0, dout, full8, 0, b12);
    run<int64_t, G_LDG, 4>("i64 keys, ldg gather, 4 steps (round 1)", dk, dv, cap, dx, tx, nx, 0, dout, full4, 0, b16);
    run<int32_t, G_LDG, 4>("i32 keys, ldg gather, 4 steps", dk32, dv, cap, dx, tx, nx, 0, dout, full4, 0, b12);
    run<int32_t, G_LDG, 8>("i32 keys, ldg gather, 8 steps", dk32, dv, cap, dx, tx, nx, 0, dout, full8, 0, b12);
    run<int32_t, G_CG, 4>("i32 keys, ld.cg gather, 4 steps", dk32, dv, cap, dx, tx, nx, 0, dout, full4, 0, b12);
    run<int32_t, G_NOALLOC, 4>("i32 keys, ld.nc.L1::no_allocate, 4 steps", dk32, dv, cap, dx, tx, nx, 0, dout, full4, 0, b12);
    run<int32_t, G_TEX, 4>("i32 keys, tex1Dfetch gather, 4 steps", dk32, dv, cap, dx, tx, nx, 0, dout, full4, 0, b12);
    run<int32_t, G_TEX, 8>("i32 keys, tex1Dfetch gather, 8 steps", dk32, dv, cap, dx, tx, nx, 0, dout, full8, 0, b12);
    // part of x in shared memory (persistent CTAs: x is loaded once per CTA)
    for (int kb : {64, 128, 200}) {
        const int nsm = kb * 1024 / 8;
        char nm[96];
        snprintf(nm, sizeof nm, "i32 keys, %d KB of x in smem + ldg, 4 steps", kb);
        const int ctas = kb <= 100 ? 2 : 1;
        run<int32_t, G_SMEM, 4>(nm, dk32, dv, cap, dx, tx, nx, nsm, dout, nsmc * ctas, (size_t)nsm * 8, b12, 1024);
    }
    {   // persistent grids without smem, for comparison with the smem variants
        run<int32_t, G_LDG, 4>("i32 keys, ldg gather, persistent 2x1024/SM", dk32, dv, cap, dx, tx, nx, 0, dout, nsmc * 2, 0, b12, 1024);
        run<int32_t, G_TEX, 4>("i32 keys, tex gather, persistent 2x1024/SM", dk32, dv, cap, dx, tx, nx, 0, dout, nsmc * 2, 0, b12, 1024);
    }
    {   // the product SpMV kernels on a row-major-like array: a semaphore cell (key 0, value = partition id) every ~166 cells
        int64_t nparts = 0;
        for (int64_t i = 0; i < cap; i += 166) { hk[i] = 0; hv[i] = (double)(++nparts); }
        CK(cudaMemcpy(dk, hk.data(), cap * 8, cudaMemcpyHostToDevice));
        CK(cudaMemcpy(dv, hv.data(), cap * 8, cudaMemcpyHostToDevice));
        double *yslot, *carry; int32_t *ycnt, *ccnt, *clast;
        CK(cudaMalloc(&yslot, (nparts + 1) * 8)); CK(cudaMalloc(&ycnt, (nparts + 1) * 4));
        CK(cudaMalloc(&carry, (cap / 64) * 8)); CK(cudaMalloc(&ccnt, (cap / 64) * 4)); CK(cudaMalloc(&clast, (cap / 64) * 4));
        cudaEvent_t e0, e1;
        CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
        auto timeit = [&](const char* name, auto launch) {
            for (int i = 0; i < 3; ++i) launch();
            CK(cudaDeviceSynchronize());
            CK(cudaEventRecord(e0));
            for (int i = 0; i < 20; ++i) launch();
            CK(cudaEventRecord(e1));
            CK(cudaDeviceSynchronize());
            float ms = 0;
            CK(cudaEventElapsedTime(&ms, e0, e1));
            printf("%-60s : %8.2f us\n", name, 1e3 * ms / 20);
        };
        const int64_t nch4 = cap / 128, nch8 = cap / 256;
        timeit("product k_spmv_blocked<false,4>", [&] {
            dsa::k_spmv_blocked<0, 4><<<(unsigned)(nch4 * 32 / 256), 256>>>(dk, dv, cap, dx, nullptr, nullptr, nx, yslot, ycnt, carry, ccnt, clast, nch4); });
        timeit("product k_spmv_blocked<false,8>", [&] {
            dsa::k_spmv_blocked<0, 8><<<(unsigned)(nch8 * 32 / 256), 256>>>(dk, dv, cap, dx, nullptr, nullptr, nx, yslot, ycnt, carry, ccnt, clast, nch8); });
        timeit("product k_spmv_blocked<false,4> + fixup", [&] {
            dsa::k_spmv_blocked<0, 4><<<(unsigned)(nch4 * 32 / 256), 256>>>(dk, dv, cap, dx, nullptr, nullptr, nx, yslot, ycnt, carry, ccnt, clast, nch4);
            dsa::k_spmv_fixup<<<(unsigned)((nch4 + 255) / 256), 256>>>(yslot, ycnt, carry, ccnt, clast, nch4); });
    }
    return 0;
}
