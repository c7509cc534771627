// csrc/mcu_tc.cuh -- kernels 2+3 fused per MCU with the IDCT on the 5th-generation tensor cores (tcgen05).
// Included at the end of kernels.cu (it shares that file's constants, colour conversion and exact evaluation).
//
// Reference functions replaced: DequantizeBlock 144-152, DeZigZag 156-163, TransformArray 167-180, IDCT_calc
// 105-124, PerformIDCT 126-140, Clamp 83-91, DecodeSingleBlock 184-228, YCrCB_to_RGB24_Block8x8 884-932
// (loadjpg.cpp), bit for bit.
//
// IDCT_calc is a 64 x 64 matrix applied to the 64 de-quantised coefficients of a block, then a truncation.
// Truncation is discontinuous, so the decoder works in two tiers: a fast evaluation with a PROVEN error bound,
// and a re-evaluation in the reference's own order of operations of the few samples that land within that
// bound of an integer.  hjd_idct_block (kernels.cu) runs the fast tier as FP32 FMA chains, 16 per sample, and is
// bound by the FMA pipe (64 % busy; the passes and the de-quantisation are two thirds of its cycles).  Here the fast tier is one tcgen05.mma sequence per 128 blocks:
//
//     D[128 blocks x 128] (TMEM, FP32)  =  V[128 x 64] (FP16, shared memory)  x  [M_hi | M_lo]^T (FP16, shared memory)
//
//   V     the de-quantised coefficients short(coef * q) of 128 blocks (thread t = MCU t = row t = TMEM lane t),
//         in zig-zag order (the matrix rows are permuted instead), as FP16: integers, exact while |v| <= 2047;
//   M     M[k][8y+x] = 0.25 * C(u)C(v) * cos[x][u] * cos[y][v] for zig-zag position k = (u, v): the real-number
//         product of the reference's float constants (PI = 3.14f, C(0)C(0) = 0.49999997), in fixed point:
//         M = (M_hi * 2^11 + M_lo) * 2^-24 + e,  |e| <= 2^-25,  M_hi, M_lo integers, |M_hi| <= 2048, |M_lo| <= 1024.
//         The tile holds M_hi * 2^-13 and M_lo, both exact in FP16.
//   Every product v * M_hi (in units of 2^-13) is an integer below 2^22 and every partial sum an integer below
//   2^24 as long as sum |v| < 8192; FP32 represents them all, so the accumulation inside the tensor core is EXACT
//   whatever its internal alignment and rounding are (measured: tools/exp_umma_idct.cu, 0 mismatches against 64-bit
//   integer sums over 9.7 M sums incl. adversarial blocks).  The same holds for M_lo.  Then
//       h = fma(D_lo, 2^-24, D_hi)
//   differs from the real-number value of 0.25 * sum by at most 1 unit (fixed-point error of M: 2^-25 * sum|v|, and
//   sum|v| <= 2A) + 0.25 unit (the FMA's rounding), one unit being 2^-24 * A with A = sum |C(u)C(v) v|.  The reference's
//   own float evaluation (three roundings per product, 63 additions) is within (3 + 63) / 4 = 16.5 units of it, and the
//   two candidates h - win, h + win of the truncation test cost another 0.25 unit: 18 units in all.  The window is 20
//   units; A is accumulated in FP16 (relative error below 1.6 %, C(0) rounded up) and inflated by 2 %.
//   Measured (tools/exp_umma_idct.cu, 4.8 M samples incl. adversarial blocks): at most 0.79 units from the real value,
//   1.34 units from the reference's float result.
//   Blocks outside the fast tier's preconditions (a quantised coefficient beyond +-511, a de-quantised one beyond
//   +-2047, A >= 4000 -- none of which a picture produces at any quality below ~97) take the exact evaluation for
//   all 64 samples.  DC-only blocks are one multiplication (cos(0) == 1: every sample is trunc(0.25 * fl(C00 * v))).
//
// The exact evaluations are batched per warp: flagged samples go to a per-warp list in shared memory and are
// handed out one per lane (a lane re-reads the block's coefficients from L2), instead of every lane walking its
// own flagged samples while the other 31 wait.
#pragma once
#include <cuda_fp16.h>

#ifndef HJD_TC_WAIT_NS
#define HJD_TC_WAIT_NS 100    // sleep between two looks at an mbarrier that has not completed yet
#endif

// ---- tcgen05 / mbarrier PTX -----------------------------------------------------------------------
__device__ __forceinline__ uint32_t hjd_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void hjd_mbar_init(uint32_t bar, uint32_t count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(bar), "r"(count) : "memory"); }
__device__ __forceinline__ void hjd_mbar_wait(uint32_t bar, uint32_t parity)
{
    uint32_t ok, spins = 0;
    do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
        if (!ok) {
            // not yet: sleep instead of spinning (a failed attempt returns after ~100 cycles; fifteen of them per wait were
            // 9 % of all the instructions this kernel issued, in slots the other warps of the SM could have used)
            __nanosleep(HJD_TC_WAIT_NS);
            if (++spins > (1u << 24)) __trap();         // a lost MMA must end the kernel, not hang the device
        }
    } while (!ok);
}
__device__ __forceinline__ void hjd_tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void hjd_tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void hjd_proxy_fence() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void hjd_umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate)
{
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                 :: "r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void hjd_umma_commit(uint32_t bar) { asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(bar) : "memory"); }
__device__ __forceinline__ void hjd_tmem_ld16(uint32_t taddr, uint32_t* r)
{
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]),
                   "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                 : "r"(taddr));
}
// 16 bytes global -> shared, asynchronously, past the L1 (the shared-memory carve-out leaves it almost no capacity)
__device__ __forceinline__ void hjd_cp_async16(uint32_t dst, const void* src) { asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" :: "r"(dst), "l"(src) : "memory"); }
__device__ __forceinline__ void hjd_cp_async_wait() { asm volatile("cp.async.wait_all;" ::: "memory"); }
__device__ __forceinline__ void hjd_group_barrier(uint32_t id) { asm volatile("bar.sync %0, 128;" :: "r"(id) : "memory"); }
__device__ __forceinline__ void hjd_tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// Shared-memory matrix descriptor: K-major, 128-byte swizzle, rows of 64 FP16 = 128 bytes, 8-row atoms of
// 1024 bytes (stride byte offset), descriptor version 1 (sm_100).  The tile must be 1024-byte aligned.
__device__ __forceinline__ uint64_t hjd_smem_desc_sw128(uint32_t addr)
{
    return (uint64_t)((addr >> 4) & 0x3FFF) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
// Instruction descriptor: FP16 x FP16 -> FP32, A and B K-major, M = 128, N = 128.
#define HJD_IDESC_F16_M128_N128 ((1u << 4) | ((128u >> 3) << 17) | ((128u >> 4) << 24))

#define HJD_TC_TILE_BYTES   16384u
#define HJD_TC_LIST_CAP     64
#define HJD_TC_GROUPS       4                          // 128-thread groups per CTA: one V tile, one accumulator, one barrier each; the matrix is shared
#define HJD_TC_THREADS      (128 * HJD_TC_GROUPS)
// slack for the 1024-byte alignment + M + one V tile per group + four 8x8 tiles per thread
#define HJD_TC_SMEM_BYTES   (1024u + (1u + HJD_TC_GROUPS) * HJD_TC_TILE_BYTES + 4u * 8u * HJD_TC_THREADS * 8u)
#define HJD_TC_TMEM_COLS    512u                       // allocation: a power of two >= 128 * groups
#ifndef HJD_TC_WINDOW_UNITS
#define HJD_TC_WINDOW_UNITS 20.0f
#endif

// [M_hi * 2^-13 | M_lo] as the UMMA tile image (FP16): filled per device by hjd_set_idct_constants.
__device__ uint4 g_idct_mat[HJD_TC_TILE_BYTES / 16];

// natural index of zig-zag position p
__host__ __device__ constexpr int hjd_zz(int p)
{
    int r = 0;
#define HJD_ZF(P, N) if ((P) == p) r = (N);
    HJD_ZZ_LIST(HJD_ZF)
#undef HJD_ZF
    return r;
}
// C(u)C(v) of zig-zag positions 2i (low half) and 2i+1 (high half) as FP16 bit patterns, rounded UP (they weigh
// the error bound A): 1 -> 0x3C00, 1/sqrt(2) -> 0x39A9 (0.70752), the DC position -> 0 (its term is added apart)
__host__ __device__ constexpr uint32_t hjd_cc_bits(int p)
{
    return p == 0 ? 0u : (((hjd_zz(p) & 7) == 0 || (hjd_zz(p) >> 3) == 0) ? 0x39A9u : 0x3C00u);
}
__host__ __device__ constexpr uint32_t hjd_cc_pair_bits(int i) { return hjd_cc_bits(2 * i) | hjd_cc_bits(2 * i + 1) << 16; }

// zig-zag position of natural index n (inverse of HJD_ZZ_LIST); n is a compile-time constant wherever this is used
__host__ __device__ constexpr int hjd_izz(int n)
{
    int r = 0;
#define HJD_IZ(P, N) if ((N) == n) r = (P);
    HJD_ZZ_LIST(HJD_IZ)
#undef HJD_IZ
    return r;
}

__device__ __forceinline__ uint32_t hjd_h2_as_u32(__half2 h) { return *(uint32_t*)&h; }
__device__ __forceinline__ __half2 hjd_u32_as_h2(uint32_t u) { return *(__half2*)&u; }

// One sample (x, y) of one block in the reference's exact order of operations (loadjpg.cpp:112-123), from the
// coefficient slab: blk = the block's 64 int16 (zig-zag order), qp = its component's quantisation table packed for DP2A.
// Same operations as hjd_exact_sum, two terms per packed instruction where the order allows it: the products
// (rounded once each, like the scalar ones) pair up, the 64 additions stay a chain in the reference's order.
__device__ __forceinline__ int hjd_exact_sample_gmem(const uint4* __restrict__ blk, const uint4* __restrict__ qp, const float* s_cos, int x, int y)
{
    uint4 c[8], q[8];
#pragma unroll
    for (int i = 0; i < 4; i++) { hjd_ldg256(blk + 2 * i, c[2 * i], c[2 * i + 1]); hjd_ldg256_nc(qp + 2 * i, q[2 * i], q[2 * i + 1]); }
    const uint32_t* cw = (const uint32_t*)c;
    const uint32_t* qw = (const uint32_t*)q;
    float cx[8], ty[8];
    { const float4 a = *(const float4*)(s_cos + x * 8), b = *(const float4*)(s_cos + x * 8 + 4); cx[0] = a.x; cx[1] = a.y; cx[2] = a.z; cx[3] = a.w; cx[4] = b.x; cx[5] = b.y; cx[6] = b.z; cx[7] = b.w; }
    { const float4 a = *(const float4*)(s_cos + y * 8), b = *(const float4*)(s_cos + y * 8 + 4); ty[0] = a.x; ty[1] = a.y; ty[2] = a.z; ty[3] = a.w; ty[4] = b.x; ty[5] = b.y; ty[6] = b.z; ty[7] = b.w; }
    const float cc0 = c_cc0, cc00 = c_cc00;
    uint32_t m16;
    asm volatile("mov.u32 %0, 0xFFFF;" : "=r"(m16));                  // in a register: (prod & 0xFFFF) ^ K is ONE LOP3
    float sum = 0.f;
#pragma unroll
    for (int u = 0; u < 8; u++) {
#pragma unroll
        for (int vp = 0; vp < 4; vp++) {
            float2 f2;
#pragma unroll
            for (int h = 0; h < 2; h++) {
                const int p = hjd_izz(8 * (2 * vp + h) + u);
                const int prod = (p & 1) ? hjd_dp2a_hi_su(cw[p >> 1], qw[p >> 1]) : hjd_dp2a_lo_su(cw[p >> 1], qw[p >> 1]);   // loadjpg.cpp:150
                // (float)(short)prod without the conversion unit: the low 16 bits, offset binary, under the exponent of
                // 1.5 * 2^23: the float 12582912 + 32768 + s, exactly
                uint32_t fb;
                asm("lop3.b32 %0, %1, %2, 0x4B408000, 0x6A;" : "=r"(fb) : "r"(prod), "r"(m16));
                if (h) f2.y = __uint_as_float(fb); else f2.x = __uint_as_float(fb);
            }
            f2 = __fadd2_rn(f2, make_float2(-12615680.0f, -12615680.0f));
            // (C(u)*C(v)) * block[u][v]; a factor 1.0f is exact
            if (u == 0) f2 = __fmul2_rn(f2, vp == 0 ? make_float2(cc00, cc0) : make_float2(cc0, cc0));
            else if (vp == 0) f2 = __fmul2_rn(f2, make_float2(cc0, 1.0f));
            const float2 t2 = __fmul2_rn(__fmul2_rn(f2, make_float2(cx[u], cx[u])), make_float2(ty[2 * vp], ty[2 * vp + 1]));
            sum = __fadd_rn(__fadd_rn(sum, t2.x), t2.y);
        }
    }
    return hjd_finish_sample(sum);
}

// bit b of the result <=> byte b of d is non-zero
__device__ __forceinline__ uint32_t hjd_nonzero_bytes(uint32_t d)
{
    const uint32_t t = (((d & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | d) & 0x80808080u;
    return (((t >> 7) * 0x00204081u) >> 21) & 0xFu;
}

// Work is handed out in units of 128 MCUs, one per group and round: the four groups of a CTA share the matrix tile and
// nothing else, so each walks its own units (unit = first + k * stride) at its own pace -- one resident CTA per SM for the
// whole launch, no tail of half-idle CTAs, TMEM and the matrix set up once.
//   units_x > 0: images of similar size; unit u = (image u / units_x, MCUs (u % units_x) * 128 ...)   (no look-up)
//   units_x = 0: mixed or tiny sizes; unit u = MCUs u * 128 ... of the whole batch, the image of each thread found by
//                binary search in mcu_prefix[i] = MCUs of the images before i.
template <bool BMP>
__global__ void __launch_bounds__(HJD_TC_THREADS, 1)
hjd_k_mcu_rgb_tc(const int16_t* __restrict__ coef, const HjdImageDesc* __restrict__ imgs,
                 const HjdQuantSet* __restrict__ qsets, uint8_t* __restrict__ rgb,
                 const uint32_t* __restrict__ mcu_prefix, int n_images, uint32_t n_units, uint32_t units_x)
{
    extern __shared__ uint8_t smem_raw[];
    __shared__ float s_cos[64];
    __shared__ uint64_t s_bar[HJD_TC_GROUPS];
    __shared__ uint32_t s_tmem;
    __shared__ int s_nsteps[HJD_TC_GROUPS];
    __shared__ uint32_t s_arrive[HJD_TC_GROUPS];                   // warps of the group that are ready for the next MMA
    __shared__ uint32_t s_cnt[HJD_TC_THREADS / 32];
    __shared__ uint32_t s_list[HJD_TC_THREADS / 32][HJD_TC_LIST_CAP];
    // 1024-byte alignment of the swizzled tiles, by an offset so that the pointers stay in the shared address space (LDS / STS)
    uint8_t* const smem = smem_raw + ((1024u - (hjd_smem_u32(smem_raw) & 1023u)) & 1023u);
    const uint32_t t = threadIdx.x, lane = t & 31u, warp = t >> 5, grp = t >> 7, tg = t & 127u;
    uint8_t* const sM = smem;                                                   // the IDCT matrix, shared by the groups
    uint8_t* const sV = smem + (1u + grp) * HJD_TC_TILE_BYTES;                  // this group's coefficient tile
    uint2* const s_tile = (uint2*)(smem + (1u + HJD_TC_GROUPS) * HJD_TC_TILE_BYTES);   // [4][8 * T]: Y (left), Y (right), Cb, Cr; row r of thread t at [r * T + t]

    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(hjd_smem_u32(&s_tmem)), "r"(HJD_TC_TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (t < HJD_TC_GROUPS) { hjd_mbar_init(hjd_smem_u32(&s_bar[t]), 1); s_nsteps[t] = 0; s_arrive[t] = 0; }
    if (t == 0) asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    if (t < 64) s_cos[t] = c_cos[t];
    if (t < HJD_TC_THREADS / 32) s_cnt[t] = 0;
    for (uint32_t i = t; i < HJD_TC_TILE_BYTES / 16; i += HJD_TC_THREADS) ((uint4*)sM)[i] = g_idct_mat[i];
    hjd_proxy_fence();                                            // the matrix tile was written through the generic proxy
    hjd_tc_fence_before();
    __syncthreads();                                              // barriers, TMEM address, matrix
    hjd_tc_fence_after();

    const uint32_t tmem = s_tmem;
    const uint32_t bar = hjd_smem_u32(&s_bar[grp]);
    const uint32_t arrive_s = hjd_smem_u32(&s_arrive[grp]);
    const uint64_t vdesc0 = hjd_smem_desc_sw128(hjd_smem_u32(sV)), mdesc = hjd_smem_desc_sw128(hjd_smem_u32(sM));
    const uint32_t tacc = tmem + 128u * grp;                      // this group's accumulator: 128 lanes x 128 columns
    const uint32_t taddr = tacc + (((warp & 3u) * 32u) << 16);    // a warp reads the 32 lanes of its quarter
    uint8_t* const vrow0 = sV + tg * 128u;                        // this thread's row of the group's V tile
    const uint32_t vrow0_s = hjd_smem_u32(vrow0);
    constexpr uint32_t kPitch = HJD_TC_THREADS * 8;
    constexpr uint32_t kTile = 8 * kPitch;
    uint8_t* const tile0 = (uint8_t*)&s_tile[t];                  // tile s of this thread: tile0 + s * kTile, row r at + r * kPitch
    uint32_t phase = 0;

#pragma unroll 1
    for (uint32_t unit = blockIdx.x * HJD_TC_GROUPS + grp; unit < n_units; unit += gridDim.x * HJD_TC_GROUPS) {
        // ---- which MCU; nobody leaves: every thread of the group takes part in its barriers
        const HjdImageDesc* d = imgs;
        uint32_t m = 0;
        bool valid = true;
        if (units_x == 0) {
            const uint32_t key = unit * 128u + tg + mcu_prefix[0];
            if (key >= mcu_prefix[n_images]) valid = false;
            else {
                const int i = hjd_image_of(mcu_prefix, n_images, key);
                d = imgs + i;
                m = key - mcu_prefix[i];
            }
        } else {
            const uint32_t img = unit / units_x;
            d = imgs + img;
            m = (unit - img * units_x) * 128u + tg;
        }
        if (valid && (m >= d->n_mcus || d->blocks_per_mcu == 0)) valid = false;
        const uint32_t hf = valid ? d->hf : 1u, vf = valid ? d->vf : 1u, bpm = valid ? d->blocks_per_mcu : 0u;
        const bool gray = valid ? d->ncomp == 1 : true;
        const uint32_t ny = gray ? 1u : hf * vf;
        const uint32_t mcus_x = valid ? d->mcus_x : 1u;
        const uint32_t my = m / mcus_x, mx = m - my * mcus_x;
        const int hs = (int)hf - 1, vs = (int)vf - 1;
        const HjdQuantSet* qs = qsets + (valid ? d->quant_set : 0u);
        const uint4* cp = (const uint4*)(coef + ((valid ? d->block_base : 0ull) + (uint64_t)m * bpm) * 64);

        const uint32_t W = valid ? d->width : 0u, H = valid ? d->height : 0u;
        const uint64_t img_pitch = BMP ? (uint64_t)((W * 3 + 3) & ~3u) : (uint64_t)W * 3;
        uint8_t* img_rgb = rgb + (valid ? d->rgb_off : 0ull) + (BMP ? HJD_BMP_PIXEL_OFF : 0);
        const uint32_t px = mx * hf * 8;                              // left edge of the MCU
        const uint32_t npix = px < W ? min(8u * hf, W - px) : 0u;     // loadjpg.cpp:907
        if (BMP && valid && m == 0) {                                 // the header, by the thread of the first MCU (openjpg.cpp:537-552)
            uint8_t* hp = rgb + d->rgb_off + HJD_BMP_FILE_OFF;
            const uint32_t file_size = (uint32_t)(img_pitch * H) + 54u;
            const uint32_t words[13] = {file_size, 0u, 54u, 40u, W, H, 1u | 24u << 16, 0u, 0u, 0u, 0u, 0u, 0u};
            hp[0] = 'B'; hp[1] = 'M';
#pragma unroll
            for (int k = 0; k < 13; k++)
#pragma unroll
                for (int qq = 0; qq < 4; qq++) hp[2 + 4 * k + qq] = (uint8_t)(words[k] >> (8 * qq));
        }
        const uint32_t n_pre = gray ? 0u : 2u;
        const uint32_t n_mine = valid ? n_pre + ny : 0u;
        // One V tile per group: block it + 1 is loaded and converted in REGISTERS while MMA(it) reads the tile, and stored into
        // it once that MMA has completed.  Its 128-byte line is requested into the L2 two steps ahead (the slab is 6 GB: a
        // cold load would wait for HBM); a lane without a block requests nothing and converts what its row holds.
        auto request = [&](uint32_t step) {
            if (step < n_mine) {
                const uint32_t rbi = step < n_pre ? ny + step : step - n_pre;
                asm volatile("prefetch.global.L2 [%0];" :: "l"(cp + rbi * 8));
            }
        };
        request(0);
        request(1);
        {
            const int wmax = __reduce_max_sync(0xffffffffu, (int)n_mine);
            if (tg == 0) s_nsteps[grp] = 0;
            hjd_group_barrier(1u + grp);
            if (lane == 0 && wmax) atomicMax(&s_nsteps[grp], wmax);
            hjd_group_barrier(1u + grp);
        }
        const int n_steps = s_nsteps[grp];                            // of this group: its barrier and its MMAs are its own

        // One loop, software-pipelined: steps 0,1 = Cb, Cr (colour images), then the Y blocks in decode order; after the last
        // Y block of a block row, that row of the MCU (8 or 16 pixels wide) goes out as RGB.  Iteration `it`:
        //   check-in (the last warp of the group issues MMA(it)) -> block it + 1 loaded and converted in registers (the MMA runs
        //   meanwhile) -> MMA(it) done -> block it + 1 stored into the V tile -> block it + 2 requested into the L2
        //   -> samples, exact re-evaluations, colour of block it.
        // Iteration -1 only converts block 0.
        float win = 0.f, n_win = 0.f;         // re-evaluation window on the 0.25*sum scale (0: no sample can be flagged), of block it / it + 1
        uint32_t fl = 0, n_fl = 0;            // bit 0: outside the fast tier's preconditions (all 64 samples exact); bit 1: DC-only
        uint32_t dcw = 0, n_dcw = 0;          // the sample of a DC-only block, four times
#pragma unroll 1
        for (int it = -1; it < n_steps; it++) {
            if (it >= 0) {
                // No barrier: a warp that has converted its rows of block it and read its part of D of block it - 1 checks in and
                // moves on to the next conversion; the LAST of the group's four warps to check in issues the MMA.  Nobody waits for
                // a slower warp before it has to (the completion of MMA(it), further down).
                __syncwarp();
                if (lane == 0) {
                    uint32_t old;
                    asm volatile("atom.acq_rel.cta.shared.add.u32 %0, [%1], 1;" : "=r"(old) : "r"(arrive_s) : "memory");
                    if (old == 3u) {
                        asm volatile("st.relaxed.cta.shared.u32 [%0], %1;" :: "r"(arrive_s), "r"(0u) : "memory");   // nobody checks in again before this MMA completes
                        hjd_tc_fence_after();
                        const uint64_t vdesc = vdesc0;
#pragma unroll
                        for (int k = 0; k < 4; k++) hjd_umma_f16(tacc, vdesc + 2 * k, mdesc + 2 * k, HJD_IDESC_F16_M128_N128, k > 0);
                        hjd_umma_commit(bar);
                    }
                }
                __syncwarp();
            }
            // ---- coefficients of block it + 1 -> de-quantised FP16 row of the V tile; A, preconditions ----------------
            bool waited = false;
            if (it + 1 < n_steps) {
                const uint32_t pit = (uint32_t)(it + 1);
                const bool pact = pit < n_mine;
                const uint32_t pcomp = pit < n_pre ? 1u + pit : 0u;
                uint8_t* const prow = vrow0;
                bool all_exact = false, dc_only = false;
                float dc_bp = 0.f;         // fl(C(0)C(0) * DC), the only term of a DC-only block
                float win_next_tmp = 0.f;
                {
                // Lanes without a block this step (MCU beyond the image, fewer blocks per MCU than the group's longest) convert
                // whatever their row holds like everybody else (any bit pattern converts to finite values): the rows of V are
                // independent (row t -> TMEM lane t), so what such a lane computes is never looked at; only its flags and stores
                // are switched off.  (They must not all fetch one dummy address either: 67 M requests for one L2 line cost
                // config 5 seven milliseconds.)
                uint4 c[8], q[8];
                const HjdQuantSet* const qsrc = pact ? qs : qsets;
#pragma unroll
                for (int i = 0; i < 4; i++) hjd_ldg256_nc((const uint4*)qsrc->qh[pcomp] + 2 * i, q[2 * i], q[2 * i + 1]);
                if (pact) {
                    const uint32_t pbi = pit < n_pre ? ny + pit : pit - n_pre;
#pragma unroll
                    for (int i = 0; i < 4; i++) hjd_ldg256(cp + pbi * 8 + 2 * i, c[2 * i], c[2 * i + 1]);
                } else {
#pragma unroll
                    for (int i = 0; i < 8; i++) c[i] = *(const uint4*)(prow + ((i ^ (tg & 7u)) << 4));
                }
                uint32_t* cw = (uint32_t*)c;
                const uint32_t* qw = (const uint32_t*)q;
                // DC: un-differenced, up to +-1024 / q, beyond the range of the bit trick below: one conversion per block.
                // |c0| <= 2047 converts exactly, and so does the product while it stays below 2048 (checked through vmax).
                const int c0 = (int)(short)(cw[0] & 0xFFFFu);
                const __half dc_h = __hmul(__int2half_rn(c0), __low2half(hjd_u32_as_h2(q[0].x)));
                const float dc_f = __half2float(dc_h);                                // = (float)(short)(c0 * q0) whenever the block stays in the fast tier
                // bits 15..9 of a half-word differ <=> its value is outside [-512, 511]; and p ^ 2p == 0 <=> p == 0
                uint32_t chk = 0;
                const uint32_t ac1_bits = cw[0] & 0xFFFF0000u;                          // position 1 shares its word with the DC
                const uint32_t ac1_chk = (cw[0] ^ (cw[0] << 1)) & 0xFC000000u;
                __half2 a2[2] = {__float2half2_rn(0.f), __float2half2_rn(0.f)};
                __half2 vmax = __float2half2_rn(0.f);
                const __half2 k1536 = __float2half2_rn(1536.f);
                uint32_t kmask;
                asm volatile("mov.u32 %0, 0x03FF03FF;" : "=r"(kmask));                 // in a register: (p & mask) ^ 0x66006600 is ONE LOP3
#pragma unroll
                for (int i = 0; i < 32; i++) {
                    const uint32_t p = cw[i];
                    if (i) chk |= p ^ (p + p);
                    // (c + 1536) as FP16 bit patterns: 0x6400 | ((c + 512) & 1023) for c in [-512, 511]
                    uint32_t hb;
                    asm("lop3.b32 %0, %1, %2, 0x66006600, 0x6A;" : "=r"(hb) : "r"(p), "r"(kmask));
                    const __half2 x = __hsub2(hjd_u32_as_h2(hb), k1536);
                    __half2 v = __hmul2(x, hjd_u32_as_h2(qw[i]));                      // exact while |c * q| <= 2048
                    if (i == 0) v = __halves2half2(dc_h, __high2half(v));
                    const __half2 av = __habs2(v);
                    vmax = __hmax2(vmax, av);
                    // C(u)C(v) per zig-zag position, rounded up: 1, 0.70752 (0x39A9), 0.5; the DC term is kept apart
                    a2[i & 1] = __hfma2(av, hjd_u32_as_h2(hjd_cc_pair_bits(i)), a2[i & 1]);
                    cw[i] = hjd_h2_as_u32(v);
                }
                if (it >= 0) {                                        // MMA(it) is reading the tile: wait for it (normally long done)
                    hjd_mbar_wait(bar, phase);
                    phase ^= 1u;
                    waited = true;
                }
#pragma unroll
                for (int i = 0; i < 8; i++) *(uint4*)(prow + ((i ^ (tg & 7u)) << 4)) = c[i];
                const __half2 as = __hadd2(a2[0], a2[1]);
                const float a_ac = __low2float(as) + __high2float(as);
                const float a_dc = 0.5f * fabsf(dc_f);
                const float a_tot = (a_ac + a_dc) * 1.02f;
                dc_only = (chk | ac1_bits) == 0u;
                dc_bp = __fmul_rn(c_cc00, dc_f);
                const float vm = fmaxf(__low2float(vmax), __high2float(vmax));
                const bool dc_wide = (uint32_t)(c0 + 2047) > 4094u || !(vm < 2048.f);     // the DC itself outside the exact range
                all_exact = (!dc_only && (((chk | ac1_chk) & 0xFC00FC00u) != 0u || !(a_tot < 4000.f))) || dc_wide;
                if (dc_wide) dc_only = false;
                win_next_tmp = (dc_only || !pact || all_exact) ? 0.f : a_tot * (HJD_TC_WINDOW_UNITS * 5.9604644775390625e-08f);
            }
                hjd_proxy_fence();                                    // generic-proxy writes of the tile -> visible to the tensor core
                n_win = win_next_tmp; n_fl = (all_exact ? 1u : 0u) | (dc_only ? 2u : 0u);
                n_dcw = (uint32_t)hjd_finish_sample(dc_bp) * 0x01010101u;
            }
            if (it < 0) { win = n_win; fl = n_fl; dcw = n_dcw; continue; }

            const bool act = (uint32_t)it < n_mine;
            const bool chroma = (uint32_t)it < n_pre;
            const uint32_t bi = chroma ? ny + it : it - n_pre;        // block index inside the MCU
            const uint32_t bx = chroma ? 0u : bi & (hf - 1u), by = chroma ? 0u : bi >> hs;      // sampling factors are 1 or 2
            const uint32_t slot = chroma ? 2u + it : (bx ? 1u : 0u);
            const bool all_exact = (fl & 1u) != 0u, dc_only = (fl & 2u) != 0u;
            if (!waited) { hjd_mbar_wait(bar, phase); phase ^= 1u; }
            hjd_tc_fence_after();
            request((uint32_t)it + 2u);

            // ---- D -> samples.  h = D_hi + 2^-24 * D_lo is within `win` of the reference's 0.25 * sum, and the reference's sample is
            // sat_u8(trunc(0.25 * sum) + 128) = sat_s8(trunc(.)) ^ 0x80 (|h| <= A / 4 < 1000: neither short wrap of loadjpg.cpp:136-137 can
            // trigger), a monotone function: where it gives the same byte for h - win and for h + win, that byte is the reference's.
            // Everything else -- an integer inside the window, not a saturated one, not zero -- is re-evaluated exactly.
            uint32_t near_lo = 0, near_hi = 0;                        // bit (8y + x)
            uint8_t* const dst = tile0 + slot * kTile;
            const uint32_t dc_word = dcw;
            const float2 wpos = make_float2(win, win), wneg = make_float2(-win, -win);
#pragma unroll
            for (int yp = 0; yp < 4; yp++) {
                uint32_t dh[16], dl[16];
                hjd_tmem_ld16(taddr + 16 * yp, dh);
                hjd_tmem_ld16(taddr + 64 + 16 * yp, dl);
                hjd_tmem_ld_wait();
#pragma unroll
                for (int yy = 0; yy < 2; yy++) {
                    const int y = 2 * yp + yy;
                    int ip[8], im[8];
#pragma unroll
                    for (int xp = 0; xp < 4; xp++) {
                        const float2 hi2 = make_float2(__uint_as_float(dh[8 * yy + 2 * xp]), __uint_as_float(dh[8 * yy + 2 * xp + 1]));
                        const float2 lo2 = make_float2(__uint_as_float(dl[8 * yy + 2 * xp]), __uint_as_float(dl[8 * yy + 2 * xp + 1]));
                        const float2 h2 = __ffma2_rn(lo2, make_float2(5.9604644775390625e-08f, 5.9604644775390625e-08f), hi2);
                        const float2 p2 = __fadd2_rn(h2, wpos), m2 = __fadd2_rn(h2, wneg);
                        ip[2 * xp] = __float2int_rz(p2.x); ip[2 * xp + 1] = __float2int_rz(p2.y);         // (int)(0.25*sum), loadjpg.cpp:123
                        im[2 * xp] = __float2int_rz(m2.x); im[2 * xp + 1] = __float2int_rz(m2.y);
                    }
                    const uint32_t p_lo = hjd_pack_sat_s8(ip[1], ip[0], hjd_pack_sat_s8(ip[3], ip[2], 0u));
                    const uint32_t p_hi = hjd_pack_sat_s8(ip[5], ip[4], hjd_pack_sat_s8(ip[7], ip[6], 0u));
                    const uint32_t m_lo = hjd_pack_sat_s8(im[1], im[0], hjd_pack_sat_s8(im[3], im[2], 0u));
                    const uint32_t m_hi = hjd_pack_sat_s8(im[5], im[4], hjd_pack_sat_s8(im[7], im[6], 0u));
                    const uint32_t d_lo = p_lo ^ m_lo, d_hi = p_hi ^ m_hi;
                    if (d_lo | d_hi) {
                        const uint32_t bits = hjd_nonzero_bytes(d_lo) | hjd_nonzero_bytes(d_hi) << 4;
                        if (y < 4) near_lo |= bits << (8 * y); else near_hi |= bits << (8 * (y - 4));
                    }
                    uint32_t r_lo = p_lo ^ 0x80808080u, r_hi = p_hi ^ 0x80808080u;
                    if (dc_only) { r_lo = dc_word; r_hi = dc_word; }
                    if (act) *(uint2*)(dst + (uint32_t)y * kPitch) = make_uint2(r_lo, r_hi);
                }
            }
            hjd_tc_fence_before();                                    // D has been read: the next step's MMA may overwrite it after the barrier
            if (all_exact) { near_lo = 0xFFFFFFFFu; near_hi = 0xFFFFFFFFu; }
            if (!act) { near_lo = 0; near_hi = 0; }

            // ---- exact re-evaluation, batched per warp -------------------------------------------------------------
            const bool batch_end = act && !chroma && bx + 1 >= hf;
            for (;;) {
                const uint32_t n_pend = (uint32_t)__popc(near_lo) + (uint32_t)__popc(near_hi);
                if (n_pend) {
                    const uint32_t base = atomicAdd(&s_cnt[warp], n_pend);
                    uint32_t room = base < HJD_TC_LIST_CAP ? HJD_TC_LIST_CAP - base : 0u;
                    uint32_t j = base;
                    while (room && (near_lo | near_hi)) {
                        uint32_t pos;
                        if (near_lo) { pos = (uint32_t)__ffs((int)near_lo) - 1u; near_lo &= near_lo - 1u; }
                        else         { pos = 32u + (uint32_t)__ffs((int)near_hi) - 1u; near_hi &= near_hi - 1u; }
                        s_list[warp][j++] = lane | slot << 5 | bi << 7 | pos << 11;
                        room--;
                    }
                }
                __syncwarp();
                const bool more = (near_lo | near_hi) != 0u;
                if (!__any_sync(0xffffffffu, more || batch_end)) break;
                const uint32_t n_list = min(s_cnt[warp], (uint32_t)HJD_TC_LIST_CAP);
                for (uint32_t base = 0; base < n_list; base += 32) {
                    const bool have = base + lane < n_list;
                    const uint32_t e = have ? s_list[warp][base + lane] : lane;
                    const uint32_t owner = e & 31u, eslot = (e >> 5) & 3u, ebi = (e >> 7) & 15u, epos = (e >> 11) & 63u;
                    const uint64_t ocp = __shfl_sync(0xffffffffu, (uint64_t)(uintptr_t)cp, (int)owner);
                    const uint64_t oqs = __shfl_sync(0xffffffffu, (uint64_t)(uintptr_t)qs, (int)owner);
                    if (have) {
                        const uint32_t ecomp = eslot < 2u ? 0u : eslot - 1u;
                        const int val = hjd_exact_sample_gmem((const uint4*)(uintptr_t)ocp + ebi * 8,
                                                              (const uint4*)(((const HjdQuantSet*)(uintptr_t)oqs)->qp[ecomp]), s_cos, (int)(epos & 7u), (int)(epos >> 3));
                        ((uint8_t*)&s_tile[warp * 32u + owner])[eslot * kTile + (epos >> 3) * kPitch + (epos & 7u)] = (uint8_t)val;
                    }
                }
                __syncwarp();
                if (lane == 0) s_cnt[warp] = 0;
                __syncwarp();
                if (!__any_sync(0xffffffffu, more)) break;
            }

            win = n_win; fl = n_fl; dcw = n_dcw;                      // block it + 1 becomes the current one

            // ---- upsample + colour conversion of the finished block row ---------------------------------------------
            if (batch_end && npix != 0) {
                const uint8_t* tY0 = tile0, * tY1 = tile0 + kTile, * tCb = tile0 + 2 * kTile, * tCr = tile0 + 3 * kTile;
                const uint32_t py0 = (my * vf + by) * 8;
#pragma unroll 1
                for (uint32_t r = 0; r < 8; r++) {
                    const uint32_t py = py0 + r;
                    if (py >= H) break;                                   // loadjpg.cpp:908
                    uint32_t cbw[2] = {0x80808080u, 0x80808080u}, crw[2] = {0x80808080u, 0x80808080u};
                    if (!gray) {
                        const uint32_t crow = (by * 8 + r) >> vs;         // nearest neighbour, loadjpg.cpp:911-912
                        const uint2 b8 = *(const uint2*)(tCb + crow * kPitch), r8 = *(const uint2*)(tCr + crow * kPitch);
                        cbw[0] = b8.x; cbw[1] = b8.y; crw[0] = r8.x; crw[1] = r8.y;
                    }
                    uint8_t* o8 = img_rgb + (uint64_t)(BMP ? H - 1 - py : py) * img_pitch + (uint64_t)px * 3;      // loadjpg.cpp:921-925 / openjpg.cpp:555
                    const uint2 ya = *(const uint2*)(tY0 + r * kPitch);
                    if (hs) {                                             // 16 pixels: 48 bytes, three 128-bit stores
                        const uint2 yb = *(const uint2*)(tY1 + r * kPitch);
                        const uint32_t yw[4] = {ya.x, ya.y, yb.x, yb.y};
                        uint32_t out[12];
                        hjd_color_n<1, 16, BMP>(yw, cbw, crw, out);
                        if (npix == 16 && (((uintptr_t)o8) & 15) == 0) {
                            uint4* o = (uint4*)o8;
                            o[0] = make_uint4(out[0], out[1], out[2], out[3]);
                            o[1] = make_uint4(out[4], out[5], out[6], out[7]);
                            o[2] = make_uint4(out[8], out[9], out[10], out[11]);
                        } else {
#pragma unroll
                            for (int i = 0; i < 48; i++)
                                if ((uint32_t)i < npix * 3) o8[i] = (uint8_t)(out[i >> 2] >> (8 * (i & 3)));
                        }
                    } else {                                              // 8 pixels: 24 bytes
                        const uint32_t yw[2] = {ya.x, ya.y};
                        uint32_t out[6];
                        hjd_color_n<0, 8, BMP>(yw, cbw, crw, out);
                        if (npix == 8 && (((uintptr_t)o8) & 7) == 0) {
                            uint2* o = (uint2*)o8;
                            o[0] = make_uint2(out[0], out[1]);
                            o[1] = make_uint2(out[2], out[3]);
                            o[2] = make_uint2(out[4], out[5]);
                        } else {
#pragma unroll
                            for (int i = 0; i < 24; i++)
                                if ((uint32_t)i < npix * 3) o8[i] = (uint8_t)(out[i >> 2] >> (8 * (i & 3)));
                        }
                    }
                    if constexpr (BMP) {
                        if (px + npix == W)                               // row padding, openjpg.cpp:563-567
                            for (uint32_t qq = W * 3; qq < (uint32_t)img_pitch; qq++) o8[qq - px * 3] = 0;
                    }
                }
            }
        }
    }
    hjd_tc_fence_before();
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem), "r"(HJD_TC_TMEM_COLS) : "memory");
}
