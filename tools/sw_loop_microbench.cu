// What does one main-pass step of vtx_k_sw_fold cost when nothing but the arithmetic is there?  The kernel's SASS model
// (DESIGN.md section 4) charges 2 ALU-pipe cycles per DPX instruction and 1 per plain add; the kernel reaches ~0.79 of it.
// This probe runs the same cell update (same device functions, the kernel's 288 threads x 2 CTAs = 18 warps/SM) on
// registers only and then adds the other ingredients of the step one at a time: the profile merge, the shared-memory
// profile loads, the boundary shuffles, the boundary store.  Level 5 is the whole step with the profile pre-merged over
// (forward code, reverse code) pairs: one code byte and 3 LDS.128 from a 17-row table, no merge.  Output: cycles per
// warp-step per SMSP.  Design aid, not product code.
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -o sw_loop_microbench tools/sw_loop_microbench.cu
#include <cstdio>
#include <cstdint>
#include <cuda_runtime.h>
#include "../vartrix_b200/csrc/vtx_sw.cuh"

using namespace vtx;

constexpr int kThreads = 288;

template <int LEVEL>
__global__ void __launch_bounds__(kThreads, 2) k_loop(uint32_t* out, int steps, long long* cyc, uint32_t k64k, uint32_t one, const uint8_t* codes_g)
{
    constexpr int C1 = 12;
    __shared__ __align__(16) uint32_t prof[2 * 5 * 96];                 // forward + reverse profile (shared by the warps: read only)
    __shared__ __align__(16) uint32_t pm[17 * 96];                      // pre-merged {fwd, rev} rows (level 5)
    __shared__ uint2 bnd[(kThreads / 32) * 160];
    __shared__ uint8_t codes[2 * 4 * 168];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, u = lane >> 3, g = lane & 7;
    uint32_t* profF = prof;
    uint32_t* profR = profF + 5 * 96;
    for (int i = threadIdx.x; i < 5 * 96; i += blockDim.x) { profF[i] = (i * 7) % 5 == 0 ? 7u : 1u; profR[i] = (i * 3) % 4 == 0 ? 7u : 1u; }
    for (int i = threadIdx.x; i < 17 * 96; i += blockDim.x) pm[i] = profF[i % (5 * 96)] + (profR[(i * 5) % (5 * 96)] << 16);
    uint8_t* cw = codes;
    for (int i = threadIdx.x; i < 2 * 4 * 168; i += blockDim.x) cw[i] = codes_g[i % 1024] % (LEVEL == 5 ? 17 : 5);
    __syncthreads();
    uint32_t hg[C1], f[C1];
#pragma unroll
    for (int c = 0; c < C1; ++c) { hg[c] = kGOE2 + lane; f[c] = kNEG2; }
    uint32_t hg_last = kGOE2, e_last = kNEG2, diag_save = kGOE2, best = kBIAS2;
    const uint8_t* cA = cw + (2 * u) * 168 + 8 - g;
    const uint8_t* cB = cA + 168;
    const uint32_t* lane_f = profF + g * C1;
    const uint32_t* lane_r = profR + g * C1;
    uint2* my_bnd = bnd + warp * 160;
    uint32_t s_reg[C1];
#pragma unroll
    for (int c = 0; c < C1; ++c) s_reg[c] = pack2(1 + 6 * ((c + lane) & 1), 1 + 6 * ((c * 3 + lane) & 1));
    const long long t0 = clock64();
#pragma unroll 1
    for (int t = 0; t < steps; ++t) {
        uint32_t hl = hg_last, el = e_last;
        if (LEVEL >= 3) {
            hl = __shfl_up_sync(0xffffffffu, hg_last, 1, 8);
            el = __shfl_up_sync(0xffffffffu, e_last, 1, 8);
            if (g == 0) { hl = kGOE2; el = kNEG2; }
        }
        const int tt = t & 127;
        const uint32_t kk = k64k + uint32_t(t & 1) * 0;      // opaque per step (t & 1 is not folded): the merge stays one IMAD per cell
        asm volatile("" : "+r"(const_cast<uint32_t&>(kk)));
        const uint4* pa = reinterpret_cast<const uint4*>(lane_f + (LEVEL >= 2 && LEVEL < 5 ? uint32_t(cA[tt]) * 96 : 0));
        const uint4* pb = reinterpret_cast<const uint4*>(lane_r + (LEVEL >= 2 && LEVEL < 5 ? uint32_t(cB[tt]) * 96 : 0));
        const uint4* pp = reinterpret_cast<const uint4*>(pm + g * C1 + (LEVEL == 5 ? uint32_t(cA[tt]) * 96 : 0));
        uint32_t diag = diag_save;
        diag_save = hl;
        uint32_t e = el, eg = hl, hleft = hl;
#pragma unroll
        for (int q = 0; q < C1 / 4; ++q) {
            uint32_t sv[4];
            if (LEVEL == 5) {
                const uint4 p4 = pp[q];
                sv[0] = p4.x; sv[1] = p4.y; sv[2] = p4.z; sv[3] = p4.w;
            } else if (LEVEL >= 2) {
                const uint4 a4 = pa[q], b4 = pb[q];
                sv[0] = b4.x * k64k + a4.x; sv[1] = b4.y * k64k + a4.y; sv[2] = b4.z * k64k + a4.z; sv[3] = b4.w * k64k + a4.w;
            } else if (LEVEL == 1) {
#pragma unroll
                for (int k = 0; k < 4; ++k) sv[k] = (s_reg[4 * q + k] >> 16) * kk + (s_reg[4 * q + k] & 0xFFFFu);
            } else {
#pragma unroll
                for (int k = 0; k < 4; ++k) sv[k] = s_reg[4 * q + k];
            }
            uint32_t hh[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int c = 4 * q + k;
                const uint32_t fc = __viaddmax_s16x2(f[c], kGE2, hg[c]);
                e = __viaddmax_s16x2(e, kGE2, eg);
                const uint32_t h = sw_h(diag, one, sv[k], fc, e);
                hh[k] = h;
                diag = hg[c];
                hleft = hadd(h, one, c);
                eg = hleft;
                hg[c] = hleft;
                f[c] = fc;
            }
            best = __vimax3_s16x2(best, hh[0], hh[1]);
            best = __vimax3_s16x2(best, hh[2], hh[3]);
        }
        hg_last = hleft;
        e_last = e;
        if (LEVEL >= 4 && g == 7) my_bnd[tt] = make_uint2(hleft, e);
    }
    const long long t1 = clock64();
    __syncwarp();
    uint32_t s = best ^ hg_last ^ e_last ^ my_bnd[lane].x ^ my_bnd[lane + 32].y;
#pragma unroll
    for (int c = 0; c < C1; ++c) s ^= hg[c] ^ f[c];
    out[blockIdx.x * blockDim.x + threadIdx.x] = s;
    if (threadIdx.x == 0) cyc[blockIdx.x] = t1 - t0;
}

template <int LEVEL> void run(const char* name, const uint8_t* codes)
{
    int n_sm = 0; cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, 0);
    const int blocks = n_sm * 2, steps = 20000;
    uint32_t* out; long long* cyc; cudaMalloc(&out, size_t(blocks) * kThreads * 4); cudaMalloc(&cyc, blocks * 8);
    k_loop<LEVEL><<<blocks, kThreads>>>(out, 200, cyc, 65536u, 1u, codes);
    k_loop<LEVEL><<<blocks, kThreads>>>(out, steps, cyc, 65536u, 1u, codes);
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) { printf("%s: %s\n", name, cudaGetErrorString(e)); return; }
    static long long h[1024]; cudaMemcpy(h, cyc, blocks * 8, cudaMemcpyDeviceToHost);
    double avg = 0; for (int i = 0; i < blocks; ++i) avg += h[i]; avg /= blocks;
    // 2 CTAs x 9 warps = 4.5 warps per SMSP share one ALU pipe: cycles per warp-step per SMSP
    printf("%-64s %7.1f cycles per warp-step per SMSP\n", name, avg / (double(steps) * (2.0 * kThreads / 32 / 4)));
    cudaFree(out); cudaFree(cyc);
}

int main()
{
    uint8_t hc[1024]; for (int i = 0; i < 1024; ++i) hc[i] = uint8_t((i * 2654435761u) >> 13);
    uint8_t* dc; cudaMalloc(&dc, 1024); cudaMemcpy(dc, hc, 1024, cudaMemcpyHostToDevice);
    int dev = 0; cudaDeviceProp prop; cudaGetDeviceProperties(&prop, dev);
    printf("%s; fold main-pass step, 12 cells per lane, %d threads x 2 CTAs = %d warps/SM; SASS model: 54 DPX x 2 + ~19 plain = ~127 ALU-pipe cycles\n",
           prop.name, kThreads, 2 * kThreads / 32);
    run<0>("cells only (substitution words in registers)", dc);
    run<1>("+ 12 merge IMADs", dc);
    run<2>("+ profile rows from shared memory (6 LDS.128, 2 LDS.U8)", dc);
    run<3>("+ boundary shuffles (2 SHFL.UP + 2 SEL)", dc);
    run<4>("+ boundary store (STS.64 by lane 7)  = the kernel's step", dc);
    run<5>("level 4 with a pre-merged profile (3 LDS.128, 1 LDS.U8, no merge)", dc);
    return 0;
}
