// csrc/scaled.cu -- reduced-size decode in the DCT domain (HJD_FLAG_SCALE_1_2 / _1_4 / _1_8, include/hjd.h).
//
// Replaces the fused kernel (kernels 2+3) when a scale flag is set: one thread per MCU de-quantises the top-left
// N x N coefficients of each block (N = 4, 2, 1), runs the reference's direct-form IDCT on them with N in place of 8
// (loadjpg.cpp:105-140 with cosf(... / 2N)), replicates chroma by the reference's rule with 8 replaced by N
// (loadjpg.cpp:911-912) and converts to RGB with the reference's float expressions (loadjpg.cpp:873-879).
// Every product and sum is rounded once, in the reference's order (__fmul_rn / __fadd_rn: nvcc must not contract),
// so the bytes are exactly those the definition in include/hjd.h gives.
#include "scaled.cuh"
#include "kernels.cuh"
#include "device_common.cuh"
#include <cuda_runtime.h>

static __constant__ float c_sc_cos4[16];   // cos4[p * 4 + k] = cosf(((2p+1) * k * 3.14f) / 8)
static __constant__ float c_sc_cos2[4];    // cos2[p * 2 + k] = cosf(((2p+1) * k * 3.14f) / 4)
static __constant__ float c_sc_cos1[1];    // cosf(0) = 1
static __constant__ float c_sc_cc[16];     // cc[u * 4 + v] = C(u) * C(v)

cudaError_t hjd_set_scaled_constants(const float cos4[16], const float cos2[4], const float cos1[1], const float cc[16])
{
    cudaError_t e = cudaMemcpyToSymbol(c_sc_cos4, cos4, 16 * sizeof(float));
    if (e == cudaSuccess) e = cudaMemcpyToSymbol(c_sc_cos2, cos2, 4 * sizeof(float));
    if (e == cudaSuccess) e = cudaMemcpyToSymbol(c_sc_cos1, cos1, sizeof(float));
    if (e == cudaSuccess) e = cudaMemcpyToSymbol(c_sc_cc, cc, 16 * sizeof(float));
    return e;
}

template <int N>
__device__ __forceinline__ float sc_cos(int p, int k)
{
    if (N == 4) return c_sc_cos4[p * 4 + k];
    if (N == 2) return c_sc_cos2[p * 2 + k];
    return c_sc_cos1[0];
}

// Zig-zag position of natural (row v, column u), v, u < 4: the reference's ZigZagArray (loadjpg.cpp:56-66).
// Called with unrolled loop indices only, so it folds to a constant.
__device__ __forceinline__ int sc_zz(int v, int u)
{
    switch (v * 4 + u) {
        case 0: return 0;   case 1: return 1;   case 2: return 5;   case 3: return 6;
        case 4: return 2;   case 5: return 4;   case 6: return 7;   case 7: return 13;
        case 8: return 3;   case 9: return 8;   case 10: return 12; case 11: return 17;
        case 12: return 9;  case 13: return 11; case 14: return 18; default: return 24;
    }
}

__device__ __forceinline__ int sc_lo(uint32_t w) { return (int)(int16_t)(w & 0xFFFFu); }
__device__ __forceinline__ int sc_hi(uint32_t w) { return (int)w >> 16; }

// The zig-zag coefficients the reduced block reads, and no others: 0..24 (N = 4), 0..4 (N = 2; 3 is not used), 0 (N = 1).
template <int N> struct ScCoef { static constexpr int K = N == 4 ? 25 : (N == 2 ? 5 : 1); };

template <int N>
__device__ __forceinline__ void sc_load(const int16_t* __restrict__ blk, int* c)
{
    if constexpr (N == 4) {
        const uint4* p = (const uint4*)blk;
#pragma unroll
        for (int j = 0; j < 3; j++) {
            const uint4 w = p[j];
            c[8 * j + 0] = sc_lo(w.x); c[8 * j + 1] = sc_hi(w.x); c[8 * j + 2] = sc_lo(w.y); c[8 * j + 3] = sc_hi(w.y);
            c[8 * j + 4] = sc_lo(w.z); c[8 * j + 5] = sc_hi(w.z); c[8 * j + 6] = sc_lo(w.w); c[8 * j + 7] = sc_hi(w.w);
        }
        c[24] = blk[24];
    } else if constexpr (N == 2) {
        const uint2 w = *(const uint2*)blk;
        c[0] = sc_lo(w.x); c[1] = sc_hi(w.x); c[2] = sc_lo(w.y); c[3] = sc_hi(w.y);
        c[4] = blk[4];
    } else {
        c[0] = blk[0];
    }
}

// One block: de-quantisation (int16 wrap, loadjpg.cpp:150), the reduced direct-form IDCT in the reference's order
// (u outer, v inner, each term ((cc * arr) * cos[x][u]) * cos[y][v]), (int16)(int)(0.25 * sum) + 128 (int16), clamp.
// out[y * N + x] = sample (x horizontal).
template <int N>
__device__ __forceinline__ void sc_idct(const int16_t* __restrict__ blk, const uint16_t* __restrict__ q, int* out)
{
    int c[ScCoef<N>::K];
    sc_load<N>(blk, c);
    float t[N][N];                                     // t[u][v] = cc[u][v] * arr[u][v]; arr[u][v] = natural[v][u]
#pragma unroll
    for (int u = 0; u < N; u++)
#pragma unroll
        for (int v = 0; v < N; v++) {
            const int z = sc_zz(v, u);
            const int a = (int)(int16_t)(c[z] * (int)q[z]);          // exact: |c * q| < 2^23, as in float
            t[u][v] = __fmul_rn(c_sc_cc[u * 4 + v], (float)a);
        }
#pragma unroll
    for (int x = 0; x < N; x++) {
        float r[N][N];
#pragma unroll
        for (int u = 0; u < N; u++)
#pragma unroll
            for (int v = 0; v < N; v++) r[u][v] = __fmul_rn(t[u][v], sc_cos<N>(x, u));
#pragma unroll
        for (int y = 0; y < N; y++) {
            float s = 0.0f;
#pragma unroll
            for (int u = 0; u < N; u++)
#pragma unroll
                for (int v = 0; v < N; v++) s = __fadd_rn(s, __fmul_rn(r[u][v], sc_cos<N>(y, v)));
            int val = (int)(int16_t)__float2int_rz(__fmul_rn(0.25f, s));   // 0.25 * sum is exact, as in double
            val = (int)(int16_t)(val + 128);
            out[y * N + x] = min(max(val, 0), 255);
        }
    }
}

// YCrCb_to_RGB (loadjpg.cpp:873-879 with the argument swap of the call at 918 resolved), scalar, each operation
// rounded once; (int) truncates, then the clamp of loadjpg.cpp:83-91.
__device__ __forceinline__ void sc_ycc(int y, int cb, int cr, int* o)
{
    const float fy = (float)y, fcb = (float)(cb - 128), fcr = (float)(cr - 128);
    const int r = __float2int_rz(__fadd_rn(fy, __fmul_rn(1.402f, fcr)));
    const int g = __float2int_rz(__fsub_rn(__fsub_rn(fy, __fmul_rn(0.34414f, fcb)), __fmul_rn(0.71414f, fcr)));
    const int b = __float2int_rz(__fadd_rn(fy, __fmul_rn(1.772f, fcb)));
    o[0] = min(max(r, 0), 255);
    o[1] = min(max(g, 0), 255);
    o[2] = min(max(b, 0), 255);
}

// One thread = one MCU, as hjd_k_mcu_rgb (kernels.cu), with its two grid shapes (device_common.cuh).  Consecutive
// threads take consecutive MCUs of a row, so the row segments a warp stores are adjacent.  Each luma block is stored as
// soon as its IDCT is done.  RGB: the chroma tiles (N x N each) go to a thread-private shared-memory region (an odd
// number of words per thread: no bank conflicts), and the luma samples are converted with them.  GRAY
// (HJD_FLAG_GRAY_OUT): no chroma IDCT, no colour conversion and no shared memory; the luma samples are stored as they
// are, one byte per pixel.
template <int N, bool GRAY, bool FLAT>
__global__ void __launch_bounds__(HJD_MCU_THREADS)
hjd_k_mcu_scaled(const int16_t* __restrict__ coef, const HjdImageDesc* __restrict__ imgs,
                 const HjdQuantSet* __restrict__ qsets, uint8_t* __restrict__ out,
                 const uint32_t* __restrict__ mcu_prefix, int n_images, int img_base)
{
    constexpr uint32_t D = 8 / N;                       // scale denominator
    constexpr int C = GRAY ? 1 : 3;                     // bytes per output pixel
    const HjdImageDesc* d;
    uint32_t m;
    if (!hjd_locate<FLAT, HJD_MCU_THREADS>(imgs, mcu_prefix, n_images, img_base, d, m)) return;
    if (m >= d->n_mcus || d->blocks_per_mcu == 0) return;
    const uint32_t hf = d->hf, vf = d->vf, bpm = d->blocks_per_mcu;
    const bool mono = d->ncomp == 1;                    // one-component file
    const uint32_t ny = mono ? 1u : hf * vf;
    const uint32_t my = m / d->mcus_x, mx = m - my * d->mcus_x;
    const int hs = (int)hf - 1, vs = (int)vf - 1;
    const HjdQuantSet* qs = qsets + d->quant_set;
    const int16_t* cp = coef + (d->block_base + (uint64_t)m * bpm) * 64;
    const uint32_t ow = (d->width + D - 1) / D, oh = (d->height + D - 1) / D;   // jdiv_round_up(W, d)
    uint8_t *tcb = nullptr, *tcr = nullptr;
    if constexpr (!GRAY) {
        constexpr int CW = (N * N + 3) / 4;             // words of one chroma tile
        constexpr int S = (2 * CW) | 1;                 // words per thread
        __shared__ uint32_t s_c[S * HJD_MCU_THREADS];
        tcb = (uint8_t*)(s_c + threadIdx.x * S);
        tcr = tcb + 4 * CW;
        if (!mono) {
            int v[N * N];
            sc_idct<N>(cp + ny * 64, qs->q[1], v);      // q[1]: Cr's table (loadjpg.cpp:984)
#pragma unroll
            for (int i = 0; i < N * N; i++) tcb[i] = (uint8_t)v[i];
            sc_idct<N>(cp + (ny + 1) * 64, qs->q[2], v);
#pragma unroll
            for (int i = 0; i < N * N; i++) tcr[i] = (uint8_t)v[i];
        }
    }
    uint8_t* img_out = out + d->rgb_off;
#pragma unroll 1
    for (uint32_t bi = 0; bi < ny; bi++) {
        const uint32_t bx = bi % hf, by = bi / hf;
        const uint32_t x0 = (mx * hf + bx) * N, y0 = (my * vf + by) * N;
        if (x0 >= ow || y0 >= oh) continue;             // pixels at or beyond the output size are not written
        int v[N * N];
        sc_idct<N>(cp + bi * 64, qs->q[0], v);
        const uint32_t npix = min((uint32_t)N, ow - x0);
#pragma unroll
        for (int y = 0; y < N; y++) {
            if (y0 + y >= oh) break;
            int ch[C * N];                              // the row's output bytes
#pragma unroll
            for (int x = 0; x < N; x++) {
                if constexpr (GRAY) {
                    ch[x] = v[y * N + x];
                } else {
                    int cb = 128, cr = 128;
                    if (!mono) {
                        const uint32_t coff = ((bx * N + x) >> hs) + ((by * N + y) >> vs) * N;
                        cb = tcb[coff];
                        cr = tcr[coff];
                    }
                    sc_ycc(v[y * N + x], cb, cr, ch + 3 * x);
                }
            }
            uint8_t* dst = img_out + ((uint64_t)(y0 + y) * ow + x0) * C;
            if (N == 4 && npix == 4 && (((uintptr_t)dst) & 3) == 0) {
                uint32_t* o = (uint32_t*)dst;
#pragma unroll
                for (int w = 0; w < C * N / 4; w++)
                    o[w] = (uint32_t)ch[4 * w] | (uint32_t)ch[4 * w + 1] << 8 | (uint32_t)ch[4 * w + 2] << 16 |
                           (uint32_t)ch[4 * w + 3] << 24;
            } else {
#pragma unroll
                for (int i = 0; i < C * N; i++)
                    if ((uint32_t)i < npix * C) dst[i] = (uint8_t)ch[i];
            }
        }
    }
}

template <int N>
static void launch_n(const int16_t* coef, const HjdImageDesc* imgs, const HjdQuantSet* qsets, uint8_t* out,
                     const uint32_t* mcu_prefix, int n_images, uint32_t n_mcus, uint32_t max_mcus, bool gray, cudaStream_t st)
{
    if (gray)
        hjd_launch_per_image(hjd_k_mcu_scaled<N, true, false>, hjd_k_mcu_scaled<N, true, true>, HJD_MCU_THREADS, mcu_prefix,
                             n_images, n_mcus, max_mcus, st, coef, imgs, qsets, out);
    else
        hjd_launch_per_image(hjd_k_mcu_scaled<N, false, false>, hjd_k_mcu_scaled<N, false, true>, HJD_MCU_THREADS, mcu_prefix,
                             n_images, n_mcus, max_mcus, st, coef, imgs, qsets, out);
}

cudaError_t hjd_launch_scaled(const int16_t* coef, const HjdImageDesc* imgs, const HjdQuantSet* qsets, uint8_t* out,
                              const uint32_t* mcu_prefix, int n_images, uint32_t n_mcus, uint32_t max_mcus, int shift,
                              bool gray, cudaStream_t st)
{
    if (n_images <= 0 || n_mcus == 0 || max_mcus == 0) return cudaSuccess;
    switch (shift) {
        case 1: launch_n<4>(coef, imgs, qsets, out, mcu_prefix, n_images, n_mcus, max_mcus, gray, st); break;
        case 2: launch_n<2>(coef, imgs, qsets, out, mcu_prefix, n_images, n_mcus, max_mcus, gray, st); break;
        case 3: launch_n<1>(coef, imgs, qsets, out, mcu_prefix, n_images, n_mcus, max_mcus, gray, st); break;
        default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}
