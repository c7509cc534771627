// csrc/kernels.cu -- hand-written sm_100a kernels of the baseline-JPEG decode path.
//
// Reference functions replaced (harutel/hls-jpeg-decoder, src/loadjpg.cpp):
//   kernel 0  marker scan      : the byte sniffing of ProcessHuffmanBlock 535-550 (done once, in parallel)
//   kernel 1  entropy decode   : FillNBits 446-484, IsInHuffmanCodes 335-392, DetermineSign 396-409,
//                                ProcessHuffmanBlock 497-863, block order of DecodeMCU 945-997
//   kernel 2  dequant+IDCT     : DequantizeBlock 144-152, DeZigZag 156-163, TransformArray 167-180,
//                                IDCT_calc 105-124, PerformIDCT 126-140, Clamp 83-91, DecodeSingleBlock 184-228
//   kernel 3  upsample+colour  : ConvertYCrCbtoRGB 867-880, YCrCB_to_RGB24_Block8x8 884-932
// The MCU raster loop of JpegDecodeHW (1134-1190) becomes the grid: every restart interval,
// 8x8 block and pixel run of every image of the batch is an independent unit of work.
//
// Integer / byte work plus a small FP32 IDCT.  The IDCT's fast tier exists twice: as FP32 FMA chains on the CUDA cores
// (hjd_idct_block, below) and as tcgen05.mma on the tensor cores (mcu_tc.cuh, included at the end of this file); the host
// picks per chunk (mcu_variant, hjd_api.cu).  Both feed the same exact re-evaluation and give the reference's bytes.
#include "kernels.cuh"
#include "device_common.cuh"
#include <cuda_runtime.h>

// ------------------------------------------------------------------------------------------
// constants
// ------------------------------------------------------------------------------------------
__constant__ float c_cos[64];     // c_cos[p*8+k] = cosf(((2p+1)*k*3.14f)/16)  (host libm, loadjpg.cpp:120)
__constant__ float2 c_cos2[64];  // c_cos2[p*8+k] = (c_cos[p*8+k], c_cos[p*8+k]): FFMA2 operand for two rows at once
__constant__ float c_cosq[64];    // 0.25f * c_cos: the final scaling folded into pass 2 (exact, a power of two)
__constant__ float c_cc0;         // C(0)*C(k>0) = 1/sqrtf(2)                    (loadjpg.cpp:96-102)
__constant__ float c_cc00;        // C(0)*C(0) = fl(0.70710677^2) = 0.49999997

static cudaError_t hjd_set_idct_matrix(const float cos_tab[64], float cc0, float cc00);

cudaError_t hjd_set_idct_constants(const float cos_tab[64], float cc0, float cc00)
{
    cudaError_t e = cudaMemcpyToSymbol(c_cos, cos_tab, 64 * sizeof(float));
    if (e != cudaSuccess) return e;
    float2 dup[64];
    for (int i = 0; i < 64; i++) dup[i] = make_float2(cos_tab[i], cos_tab[i]);
    e = cudaMemcpyToSymbol(c_cos2, dup, sizeof dup);
    if (e != cudaSuccess) return e;
    float quarter[64];
    for (int i = 0; i < 64; i++) quarter[i] = 0.25f * cos_tab[i];
    e = cudaMemcpyToSymbol(c_cosq, quarter, sizeof quarter);
    if (e != cudaSuccess) return e;
    e = cudaMemcpyToSymbol(c_cc0, &cc0, sizeof(float));
    if (e != cudaSuccess) return e;
    e = cudaMemcpyToSymbol(c_cc00, &cc00, sizeof(float));
    if (e != cudaSuccess) return e;
    return hjd_set_idct_matrix(cos_tab, cc0, cc00);
}

// zig-zag position p -> natural (row-major) index n; inverse of the reference's ZigZagArray
// (loadjpg.cpp:56-66).  A macro list so that every index is a compile-time constant and the
// 64 coefficients of a block stay in registers.
#define HJD_ZZ_LIST(X) \
    X(0, 0)   X(1, 1)   X(2, 8)   X(3, 16)  X(4, 9)   X(5, 2)   X(6, 3)   X(7, 10)  \
    X(8, 17)  X(9, 24)  X(10, 32) X(11, 25) X(12, 18) X(13, 11) X(14, 4)  X(15, 5)  \
    X(16, 12) X(17, 19) X(18, 26) X(19, 33) X(20, 40) X(21, 48) X(22, 41) X(23, 34) \
    X(24, 27) X(25, 20) X(26, 13) X(27, 6)  X(28, 7)  X(29, 14) X(30, 21) X(31, 28) \
    X(32, 35) X(33, 42) X(34, 49) X(35, 56) X(36, 57) X(37, 50) X(38, 43) X(39, 36) \
    X(40, 29) X(41, 22) X(42, 15) X(43, 23) X(44, 30) X(45, 37) X(46, 44) X(47, 51) \
    X(48, 58) X(49, 59) X(50, 52) X(51, 45) X(52, 38) X(53, 31) X(54, 39) X(55, 46) \
    X(56, 53) X(57, 60) X(58, 61) X(59, 54) X(60, 47) X(61, 55) X(62, 62) X(63, 63)

// ------------------------------------------------------------------------------------------
// kernel 0: restart-marker scan
// ------------------------------------------------------------------------------------------
// One CTA per image.  Every thread inspects 16 bytes per step; RSTn = FF D0..D7 (an FF inside
// entropy data is always followed by 00, so the pair test is exact).  The marker ordinal comes
// from a block-wide prefix sum; interval j+1 starts two bytes after marker j.
// The markers of bytes [beg, end) of one scan (offsets from the 16-byte aligned origin a0, multiples of the
// 16 KB step), in order: 64 contiguous bytes per thread and step (four 16-byte loads), one barrier per
// step (the per-warp counts are double buffered and every thread keeps the running total itself).
// WRITE: marker number `running`+k starts interval `running`+k+1.  Returns the running total at the end.
template <bool WRITE>
__device__ __forceinline__ uint32_t hjd_marker_range(const uint8_t* a0, uint32_t total, uint32_t lead, uint32_t beg,
                                                     uint32_t end, uint32_t running, uint32_t* out,
                                                     uint32_t n_intervals, uint32_t (*s_warp)[8])
{
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int buf = 0;
    for (uint32_t chunk = beg; chunk < end && chunk < total; chunk += 256 * 64, buf ^= 1) {
        const uint32_t off0 = chunk + tid * 64;
        uint64_t mask = 0;                       // bit p: an RSTn marker starts at byte off0 + p
        uint4 v[4];
#pragma unroll
        for (int q = 0; q < 4; q++)
            v[q] = (off0 + 16u * q < total) ? __ldg((const uint4*)(a0 + off0 + 16u * q)) : make_uint4(0, 0, 0, 0);
        if (off0 < total) {
            const uint32_t nb = (off0 + 64 < total) ? a0[off0 + 64] : 0u;
            // SIMD-within-a-register byte tests (exact per byte, no carries between bytes):
            //   ff: bytes equal to FF;  dn: bytes whose SUCCESSOR is D0..D7 (RSTn)
            uint32_t dd[17];
#pragma unroll
            for (int k = 0; k < 17; k++) {
                const uint32_t wk = k < 16 ? ((const uint32_t*)v)[k] : nb;
                const uint32_t x = (wk ^ 0xD0D0D0D0u) & 0xF8F8F8F8u;                      // zero byte <=> D0..D7
                dd[k] = ~(((x & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | x | 0x7F7F7F7Fu);           // 0x80 in those bytes
            }
#pragma unroll
            for (int k = 0; k < 16; k++) {
                const uint32_t wk = ((const uint32_t*)v)[k];
                const uint32_t ff = ((wk & 0x7F7F7F7Fu) + 0x01010101u) & wk & 0x80808080u;
                uint32_t hit = ff & __funnelshift_r(dd[k], dd[k + 1], 8);                 // FF followed by RSTn
                while (hit) {                                                             // rare: ~1 marker per 365 bytes
                    const int bit = __ffs((int)hit) - 1;
                    hit &= hit - 1;
                    const uint32_t p = 4u * k + ((uint32_t)bit >> 3);
                    if (off0 + p >= lead && off0 + p + 1 < total) mask |= 1ull << p;
                }
            }
        }
        const uint32_t cnt = __popcll(mask);
        uint32_t incl = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        if (lane == 31) s_warp[buf][warp] = incl;
        __syncthreads();
        uint32_t before = running;
        uint32_t block_total = 0;
#pragma unroll
        for (int k = 0; k < 8; k++) {
            const uint32_t c = s_warp[buf][k];
            if (k < warp) before += c;
            block_total += c;
        }
        if (WRITE) {
            uint32_t ord = before + incl - cnt;
            while (mask) {
                const int p = __ffsll((long long)mask) - 1;
                mask &= mask - 1;
                if (ord + 1 < n_intervals) out[ord + 1] = off0 + p + 2 - lead;
                ord++;
            }
        }
        running += block_total;
    }
    return running;
}

// Fewer markers than intervals: the missing intervals become empty (the entropy kernel zero-fills them
// and flags overrun) and the image is flagged.
__device__ __forceinline__ void hjd_marker_finish(const HjdImageDesc& d, int img, uint32_t found, uint32_t* out,
                                                  int32_t* status)
{
    if (found != d.n_intervals - 1) {
        if (threadIdx.x == 0) atomicOr(&status[img], HJD_ST_RESTART);
        for (uint32_t j = found + 1 + threadIdx.x; j < d.n_intervals; j += 256) out[j] = d.scan_len;
    }
}

__global__ void __launch_bounds__(256)
hjd_k_marker_scan(const uint8_t* __restrict__ arena, const HjdImageDesc* __restrict__ imgs,
                  uint32_t* __restrict__ interval_start, int32_t* __restrict__ status, int img_base)
{
    const int img = blockIdx.x + img_base;
    const HjdImageDesc d = imgs[img];
    uint32_t* out = interval_start + d.interval_base;
    if (d.n_intervals == 0) return;
    if (threadIdx.x == 0) out[0] = 0;
    if (d.restart_interval == 0 || d.n_intervals <= 1) return;
    if (d.scan_len > HJD_SCAN_SLICE_MIN) return;            // long scans: hjd_k_marker_slice_*

    __shared__ uint32_t s_warp[2][8];
    const uint8_t* s = arena + d.scan_off;
    const uint32_t lead = (uint32_t)((uintptr_t)s & 15);
    const uint32_t total = d.scan_len + lead;
    const uint32_t found = hjd_marker_range<true>(s - lead, total, lead, 0, total, 0, out, d.n_intervals, s_warp);
    hjd_marker_finish(d, img, found, out, status);
}

// Long scans (one CTA would walk them alone long after the rest of the batch is done: 0.31 ms for a
// 4096x4096 image) are cut into slices of HJD_SCAN_SLICE_BYTES: count per slice, then every slice adds up
// the counts of the slices before it and numbers its markers.
__global__ void __launch_bounds__(256)
hjd_k_marker_slice_count(const uint8_t* __restrict__ arena, const HjdImageDesc* __restrict__ imgs,
                         const HjdScanSlice* __restrict__ slices, uint32_t* __restrict__ slice_cnt)
{
    __shared__ uint32_t s_warp[2][8];
    const HjdScanSlice sl = slices[blockIdx.x];
    const HjdImageDesc d = imgs[sl.image];
    const uint8_t* s = arena + d.scan_off;
    const uint32_t lead = (uint32_t)((uintptr_t)s & 15);
    const uint32_t beg = sl.index * HJD_SCAN_SLICE_BYTES;
    const uint32_t n = hjd_marker_range<false>(s - lead, d.scan_len + lead, lead, beg, beg + HJD_SCAN_SLICE_BYTES, 0,
                                               nullptr, d.n_intervals, s_warp);
    if (threadIdx.x == 0) slice_cnt[blockIdx.x] = n;
}

__global__ void __launch_bounds__(256)
hjd_k_marker_slice_write(const uint8_t* __restrict__ arena, const HjdImageDesc* __restrict__ imgs,
                         const HjdScanSlice* __restrict__ slices, const uint32_t* __restrict__ slice_cnt,
                         uint32_t* __restrict__ interval_start, int32_t* __restrict__ status)
{
    __shared__ uint32_t s_warp[2][8];
    __shared__ uint32_t s_red[8];
    const HjdScanSlice sl = slices[blockIdx.x];
    const HjdImageDesc d = imgs[sl.image];
    uint32_t* out = interval_start + d.interval_base;
    // markers in the slices of this image before this one (the slices of an image are consecutive)
    uint32_t part = 0;
    for (uint32_t k = threadIdx.x; k < sl.index; k += 256) part += slice_cnt[blockIdx.x - sl.index + k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = part;
    __syncthreads();
    uint32_t before = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) before += s_red[k];
    const uint8_t* s = arena + d.scan_off;
    const uint32_t lead = (uint32_t)((uintptr_t)s & 15);
    const uint32_t beg = sl.index * HJD_SCAN_SLICE_BYTES;
    const uint32_t found = hjd_marker_range<true>(s - lead, d.scan_len + lead, lead, beg, beg + HJD_SCAN_SLICE_BYTES,
                                                  before, out, d.n_intervals, s_warp);
    if (sl.index + 1 == sl.n_slices) hjd_marker_finish(d, (int)sl.image, found, out, status);
}

cudaError_t hjd_launch_marker_scan(const uint8_t* arena, const HjdImageDesc* imgs, uint32_t* interval_start,
                                   int32_t* status, int first_image, int n_images, const HjdScanSlice* slices,
                                   int n_slices, uint32_t* slice_cnt, cudaStream_t st)
{
    if (n_images <= 0) return cudaSuccess;
    hjd_k_marker_scan<<<n_images, 256, 0, st>>>(arena, imgs, interval_start, status, first_image);
    if (n_slices > 0) {
        hjd_k_marker_slice_count<<<n_slices, 256, 0, st>>>(arena, imgs, slices, slice_cnt);
        hjd_k_marker_slice_write<<<n_slices, 256, 0, st>>>(arena, imgs, slices, slice_cnt, interval_start, status);
    }
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// kernel 1a: restart-interval-parallel entropy decode
// ------------------------------------------------------------------------------------------
// One thread per restart interval (the unit the bitstream makes independent: byte-aligned start,
// DC predictors reset).  The kernel is instruction-issue bound, and with ~12 symbols per block
// some lane of a warp is in every special case on every step, so a divergent sub-path costs the
// whole warp its full instruction count.  Hence:
//   * one branch-free symbol step shared by DC and AC (predictors and table offsets are rotated
//     through registers when the component changes);
//   * a round = one scheduled bit-buffer top-up for all lanes + HJD_ENT_SYMS symbol steps; a lane
//     that completes its block inside a round idles until the round ends, so block hand-over and
//     flushing are paid once per round instead of once per symbol;
//   * finished blocks are published in a small shared-memory list and flushed four at a time from
//     their slots to HBM with 128-bit accesses (8 lanes x 16 B per block): the coefficient slab is
//     written exactly once, densely, in full 128-byte lines;
//   * shared memory is addressed with 32-bit shared-window addresses (ld/st.shared).
//
// Shared memory: [threads x 128 B] coefficient slots, 16-byte chunks XOR-swizzled by (lane & 7)
// (conflict-free 128-bit flush, spread 2-byte scatter stores); [warps x 32 x 8 B] flush lists;
// the table set of this CTA's images (per component: DC table then AC table, contiguous).
#ifndef HJD_ENT_SYMS
#define HJD_ENT_SYMS 4
#endif
#ifndef HJD_ENT_TOPUP
#define HJD_ENT_TOPUP 32   // second top-up of a round when fewer bits than this are left (B200, config 2: 40: 3.19, 32: 3.12, 16: 3.14 ms)
#endif
// HJD_ENT_SYMS measured on B200 (ms per 1024 x 1080p, 256 threads): 3: 3.25, 4: 3.19, 5: 3.61, 6: 4.19

struct BitReader {
    const uint8_t* base;   // entropy-coded segment of the image
    uint32_t pos, end;     // byte cursor / end of this interval (relative to base)
    uint32_t hi, lo;       // MSB-aligned 64-bit window (hi:lo)
    int nbits;             // valid bits in the window
    int padbits;           // zero bits appended after `end`
    // three aligned words prefetched one round ahead: with seven CTAs of shared memory per SM there
    // is next to no L1 left, so every stream load is an L2 round trip that must not sit on the
    // critical path of the symbol loop
    const uint32_t* wptr;
    uint32_t w0, w1, w2;
};

__device__ __forceinline__ void br_prefetch(BitReader& r)
{
    r.wptr = (const uint32_t*)((uintptr_t)(r.base + r.pos) & ~(uintptr_t)3);
    r.w0 = __ldg(r.wptr);
    r.w1 = __ldg(r.wptr + 1);
    r.w2 = __ldg(r.wptr + 2);
}

// Append up to four bytes (as many as fit and as the interval still has).  FillNBits semantics
// (loadjpg.cpp:446-484): the 00 stuffed after an FF data byte is dropped.  Bytes are taken up to
// and including the first FF of the window so that the stuffed byte can be skipped without a
// branch; a second FF in the same window is picked up by the next call.
// CACHED: take the bytes from the prefetched words when they cover [pos, pos + 4).
template <bool CACHED>
__device__ __forceinline__ void br_refill(BitReader& r)
{
    const uint32_t avail = r.end - r.pos;                       // pos never passes end
    const uintptr_t a = (uintptr_t)(r.base + r.pos);
    const uint32_t* ap = (const uint32_t*)(a & ~(uintptr_t)3);
    uint32_t x0, x1;
    const uint32_t d = (uint32_t)(ap - r.wptr);                 // words between the prefetch origin and pos
    if (CACHED && d <= 1u) { x0 = d ? r.w1 : r.w0; x1 = d ? r.w2 : r.w1; }
    else { x0 = __ldg(ap); x1 = __ldg(ap + 1); }
    const uint32_t x = __funnelshift_r(x0, x1, (uint32_t)(a & 3) * 8);       // 4 bytes, memory order
    const uint32_t ffm = ((~x) - 0x01010101u) & x & 0x80808080u;             // lowest set bit is exact
    const uint32_t j = (uint32_t)(__ffs((int)ffm) - 1) >> 3;                 // first FF byte; >= 4 when none
    const uint32_t room = (uint32_t)(64 - r.nbits) >> 3;
    const uint32_t take = min(min(j + 1u, 4u), min(room, avail));
    const uint32_t skip = (take == j + 1u) ? 1u : 0u;                        // the FF went in: drop its 00
    const uint32_t w = __byte_perm(x, 0, 0x0123) & ~hjd_shr(0xFFFFFFFFu, 8 * take);   // top `take` bytes, big-endian
    // window |= w >> nbits (as a 64-bit quantity whose top word is w)
    const uint32_t n = (uint32_t)r.nbits;
    r.hi |= hjd_shr(w, n);
    r.lo |= (n >= 32u) ? hjd_shr(w, n - 32u) : hjd_shl(w, 32u - n);
    r.nbits += 8 * (int)take;
    r.pos = min(r.pos + take + skip, r.end);
    if (avail == 0 && r.nbits <= 32) { r.nbits += 32; r.padbits += 32; }     // past the interval: zero padding
}

__global__ void __launch_bounds__(HJD_ENT_THREADS, HJD_ENT_MINBLOCKS)
hjd_k_entropy_restart(const uint8_t* __restrict__ arena, const HjdImageDesc* __restrict__ imgs,
                      const HjdTableSet* __restrict__ tsets, const uint32_t* __restrict__ interval_start,
                      const HjdEntropyWork* __restrict__ work, const HjdEntropySeg* __restrict__ segs,
                      int16_t* __restrict__ coef,
                      int32_t* __restrict__ status)
{
    extern __shared__ __align__(16) uint8_t s_raw[];
    constexpr uint32_t kSlotBytes = HJD_ENT_THREADS * 128;
    constexpr uint32_t kListBytes = HJD_ENT_THREADS * 8;
    constexpr uint32_t kTabBytes = (uint32_t)sizeof(HjdHuffTable);
    const uint32_t sh_base = (uint32_t)__cvta_generic_to_shared(s_raw);
    const uint32_t sh_list = sh_base + kSlotBytes;
    const uint32_t sh_tab = sh_list + kListBytes;

    const HjdEntropyWork wk = work[blockIdx.x];
    const int tid = threadIdx.x, lane = tid & 31;
    const HjdTableSet* ts = tsets + wk.table_set;
    {
        // the distinct tables of this table set (normally 4: Cb and Cr share theirs)
        const uint4* src = (const uint4*)ts->tab;
        uint4* dst = (uint4*)(s_raw + kSlotBytes + kListBytes);
        const int n16 = ts->n_tabs * (int)(kTabBytes / 16);
        for (int i = tid; i < n16; i += HJD_ENT_THREADS) dst[i] = __ldg(src + i);
        uint4* z = (uint4*)s_raw;
        for (int i = tid; i < HJD_ENT_THREADS * 8; i += HJD_ENT_THREADS) z[i] = make_uint4(0, 0, 0, 0);
    }
    __syncthreads();

    // ---- per-lane interval setup -----------------------------------------------------------
    const uint32_t sel = (uint32_t)tid;     // (ordering a CTA's intervals by compressed length so that a warp's lanes finish
                                            //  together was measured: no gain, 2.97 vs 2.94 ms -- DESIGN.md 4.6)
    BitReader br;
    br.base = arena; br.pos = br.end = 0; br.hi = br.lo = 0; br.nbits = 0; br.padbits = 0;
    br.wptr = (const uint32_t*)arena; br.w0 = br.w1 = br.w2 = 0;
    uint32_t blocks_left = 0, gblk = 0;
    int img = 0, bpm = 1, ny = 1;
    if (sel < wk.n_intervals) {
        // the segment this interval falls into (tid0 is ascending): binary search
        uint32_t lo = 0, hi = wk.n_segs - 1;
        while (lo < hi) {
            const uint32_t mid = (lo + hi + 1) >> 1;
            if (segs[wk.first_seg + mid].tid0 <= sel) lo = mid; else hi = mid - 1;
        }
        const HjdEntropySeg sg = segs[wk.first_seg + lo];
        const uint32_t g = sg.first_interval + (sel - sg.tid0);
        img = (int)sg.image;
        const HjdImageDesc* d = imgs + img;
        const uint32_t j = g - d->interval_base;
        const uint32_t ri = d->restart_interval;
        const uint32_t first_mcu = ri ? j * ri : 0;
        const uint32_t n_mcu = ri ? min(ri, d->n_mcus - first_mcu) : d->n_mcus;
        bpm = d->blocks_per_mcu;
        ny = d->ncomp == 3 ? d->hf * d->vf : 1;
        br.base = arena + d->scan_off;
        br.pos = interval_start[g];
        br.end = (j + 1 < d->n_intervals) ? interval_start[g + 1] - 2 : d->scan_len;
        if (br.end < br.pos || br.end > d->scan_len) br.end = br.pos;
        blocks_left = n_mcu * (uint32_t)bpm;
        gblk = (uint32_t)(d->block_base + (uint64_t)first_mcu * bpm);
    }
    // byte offsets of the current component's DC (low half) and AC (high half) table; rotated with p0..p2
    uint32_t t0 = ts->dc_of_comp[0] * kTabBytes | (ts->ac_of_comp[0] * kTabBytes) << 16;
    uint32_t t1 = ts->dc_of_comp[1] * kTabBytes | (ts->ac_of_comp[1] * kTabBytes) << 16;
    uint32_t t2 = ts->dc_of_comp[2] * kTabBytes | (ts->ac_of_comp[2] * kTabBytes) << 16;
    int p0 = 0, p1 = 0, p2 = 0;        // DC predictors
    const uint32_t my_slot = sh_base + (uint32_t)tid * 128u;
    const uint32_t swz = (uint32_t)(lane & 7) << 4;      // XOR on the 16-byte chunk index
    const uint32_t warp_slots = sh_base + (uint32_t)(tid & ~31) * 128u;
    const uint32_t warp_list = sh_list + (uint32_t)(tid & ~31) * 8u;
    const uint32_t lt_mask = (1u << lane) - 1u;
    int k = 0, bi = 0;                 // zig-zag index inside the block, block index inside the MCU
    int flags = 0;
    bool dead = false;                 // undecodable code or data exhausted: zero-fill the rest
    br_prefetch(br);

    while (__any_sync(0xffffffffu, blocks_left > 0)) {
        // scheduled top-up, all lanes together, from the words prefetched during the previous round
        br_refill<true>(br);
        if (br.nbits <= HJD_ENT_TOPUP) br_refill<false>(br);        // busy stretch: keep the reserve up
        br_prefetch(br);                                 // in flight while this round's symbols decode
        if (br.padbits > 512) dead = true;
        const bool live = blocks_left > 0;
        bool done_block = !live ? false : dead;
        if (live && !dead) {
#pragma unroll
            for (int rep = 0; rep < HJD_ENT_SYMS; rep++) {
                if (!done_block) {
                    if (br.nbits < 32) {                 // several long symbols since the round's top-up
                        // Refill until a refill would change nothing (the window is full, or no padding is due), at
                        // most four times: four leave at least 32 bits (each adds a byte or more), and stopping at the
                        // first idle one gives the window all four would; the warp runs as many as its neediest lane.
#pragma unroll 1
                        for (int i = 0; i < 4 && (br.pos != br.end ? br.nbits <= 56 : br.nbits <= 32); i++)
                            br_refill<false>(br);
                    }
                    const bool is_ac = k != 0;
                    const uint32_t t = sh_tab + (is_ac ? (t0 >> 16) : (t0 & 0xFFFFu));
                    // the entry says what the symbol means: code length, value bits, zig-zag advance, store or not
                    const uint32_t e = hjd_lookup(t, br.hi);
                    const uint32_t len = e & 31u, size = (e >> 5) & 15u, kadv = (e >> 9) & 127u;
                    // value bits follow the code
                    const uint32_t after = __funnelshift_l(br.lo, br.hi, len);            // window << len, top word
                    const uint32_t v = hjd_shr(after, 32u - size);                         // 0 for size 0
                    // DetermineSign (loadjpg.cpp:396-409): leading 0 bit -> v - (2^size - 1)
                    const int neg = ~((int)after >> 31);                                   // all ones if negative
                    const int val = (int)v + (neg & (int)(hjd_shl(0xFFFFFFFFu, size) + 1u));
                    const uint32_t used = len + size;                                      // <= 31
                    br.hi = __funnelshift_l(br.lo, br.hi, used);
                    br.lo <<= used;
                    br.nbits -= (int)used;
                    const uint32_t kpos = (uint32_t)k + kadv - 1u;                         // loadjpg.cpp:778, 806
                    if (size) {                          // a value follows: DC difference or AC coefficient (slot is pre-zeroed)
                        if (kpos <= 63u) hjd_sts_u16_sync(my_slot + ((kpos << 1) ^ swz), (uint32_t)val);
                        else flags |= HJD_ST_COEF_RANGE;                                   // loadjpg.cpp:780-783
                    }
                    k += (int)kadv;                      // EOB: +63, ZRL: +16 (loadjpg.cpp:771-775)
                    done_block = k >= 64;
                }
            }
        }
        // ---- block hand-over ---------------------------------------------------------------
        uint32_t flush_blk = 0;
        if (done_block) {
            if (k >= 127) { dead = true; flags |= HJD_ST_BAD_CODE; }      // HJD_BAD_ENTRY: no such code, the interval ends here
            if (!dead) {                                  // DCT[0] = data + prevDC in int16 (loadjpg.cpp:664-665)
                p0 = (int)(short)(p0 + (int)(short)hjd_lds_u16_sync(my_slot + swz));
                hjd_sts_u16_sync(my_slot + swz, (uint32_t)p0);
            }
            flush_blk = gblk++;
            blocks_left--;
            k = 0;
            if (++bi == bpm) bi = 0;
            if (bpm > 1 && (bi == 0 || bi >= ny)) {       // component changes: Y -> Cb -> Cr -> Y
                const int tp = p0; p0 = p1; p1 = p2; p2 = tp;
                const uint32_t tt = t0; t0 = t1; t1 = t2; t2 = tt;
            }
            if (blocks_left == 0 && br.nbits < br.padbits) flags |= HJD_ST_OVERRUN;
        }
        // ---- cooperative flush of the finished blocks, four per step --------------------------
        const uint32_t m = __ballot_sync(0xffffffffu, done_block);
        if (m) {
            if (done_block) hjd_sts_v2_sync(warp_list + (uint32_t)__popc(m & lt_mask) * 8u, flush_blk, (uint32_t)lane);
            __syncwarp();
            const int n_done = __popc(m);
            const uint32_t chunk = (uint32_t)lane & 7u;
            for (int base = 0; base < n_done; base += 4) {                                  // warp-uniform trip count
                const int idx = base + (lane >> 3);
                if (idx < n_done) {
                    const uint2 ent = hjd_lds_v2_sync(warp_list + (uint32_t)idx * 8u);      // {block, owner lane}
                    const uint32_t src = warp_slots + ent.y * 128u + ((chunk ^ (ent.y & 7u)) << 4);
                    const uint4 w = hjd_lds_v4_sync(src);
                    hjd_sts_zero16_sync(src);
                    ((uint4*)coef)[(size_t)ent.x * 8u + chunk] = w;      // 64-bit: ent.x * 8 wraps from block 2^29 on
                }
            }
            __syncwarp();
        }
    }
    if (flags) atomicOr(&status[img], flags);
}

// Function attributes are per device: hjd_batch_create calls this after cudaSetDevice, for every batch
// (a process-wide "done once" flag would leave the second GPU of a process without the larger
// shared-memory window, and six distinct Huffman tables need more than the default 48 KB).
cudaError_t hjd_mcu_tc_init_device(void);
cudaError_t hjd_kernels_init_device(void)
{
    cudaError_t e = cudaFuncSetAttribute(hjd_k_entropy_restart, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)(HJD_ENT_THREADS * (128 + 8) + HJD_MAX_TABLES * sizeof(HjdHuffTable)));
    if (e != cudaSuccess) return e;
    return hjd_mcu_tc_init_device();
}

cudaError_t hjd_launch_entropy_restart(const uint8_t* arena, const HjdImageDesc* imgs, const HjdTableSet* tsets,
                                       const uint32_t* interval_start, const HjdEntropyWork* work,
                                       const HjdEntropySeg* segs, int n_work,
                                       int max_tabs, int16_t* coef, int32_t* status, cudaStream_t st)
{
    if (n_work <= 0) return cudaSuccess;
    if (max_tabs < 1) max_tabs = 1;
    if (max_tabs > HJD_MAX_TABLES) max_tabs = HJD_MAX_TABLES;
    const size_t smem = HJD_ENT_THREADS * (128 + 8) + (size_t)max_tabs * sizeof(HjdHuffTable);
    hjd_k_entropy_restart<<<n_work, HJD_ENT_THREADS, smem, st>>>(arena, imgs, tsets, interval_start, work, segs, coef, status);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// kernel 2: dequantise + de-zig-zag + IDCT (+128, clamp) -> planes
// ------------------------------------------------------------------------------------------
// The reference evaluates, for every output sample, a 64-term float sum in a fixed order with
// PI = 3.14f and truncates 0.25*sum toward zero (loadjpg.cpp:105-124).  Truncation is
// discontinuous, so a faster summation order can differ by one level whenever 0.25*sum lands
// next to an integer.  This kernel computes the separable form (16 FMA per sample) and proves,
// per sample, that truncation cannot differ: with A = sum |C(u)C(v)*coef| the two evaluations
// differ by at most (65+14) * 2^-24 * A (standard rounding-error bounds for a 64-term recursive
// sum of doubly-rounded products, and for two 8-term FMA chains; the packed even/odd split of the
// second pass is within the same bound), i.e. < 20 * 2^-24 * A on the
// 0.25*sum scale.  Samples closer than 24 * 2^-24 * A to a non-zero integer (well under 1 %) are
// re-evaluated in the reference's exact order (u outer, v inner, products left to right, no FMA).
// Blocks with only a DC term are exact in both forms (cos(0) = 1) and are never re-evaluated.
// Result: planes identical to the reference's, not merely within 1.

__device__ __forceinline__ int hjd_finish_sample(float sum)
{
    int iv = __float2int_rz(0.25f * sum);      // (int)(0.25*sum), loadjpg.cpp:123
    iv = (int)(short)iv;                       // stored to short, loadjpg.cpp:136
    iv = (int)(short)(iv + 128);               // loadjpg.cpp:137
    return min(max(iv, 0), 255);               // Clamp, loadjpg.cpp:83-91
}

// a = two signed 16-bit lanes, b = four unsigned bytes: lo -> a.lo*b0 + a.hi*b1, hi -> a.lo*b2 + a.hi*b3
__device__ __forceinline__ int hjd_dp2a_lo_su(uint32_t a, uint32_t b) { int d; asm("dp2a.lo.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(0)); return d; }
__device__ __forceinline__ int hjd_dp2a_hi_su(uint32_t a, uint32_t b) { int d; asm("dp2a.hi.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(0)); return d; }

// Short blocks.  Most blocks end, in zig-zag order, long before index 63 (at 20 on average for the q85
// workload) and everything behind the end is zero.  Skipping a zero term is exact -- x + 0*c == x, and
// fl() of an unchanged sum is unchanged -- so an IDCT variant that leaves out the frequencies beyond index
// KM computes, instruction for instruction, the same sums as the full one on any block that ends at or
// before KM: the error window, the exact re-evaluation and with them bit-exactness carry over.
// A variant ends on a whole anti-diagonal of the zig-zag scan: KM = 20 <=> u + v <= 5 (21 coefficients).
// hjd_live_mask(KM): bit n set <=> natural position n (8 * row + column) can be non-zero.
__host__ __device__ constexpr uint64_t hjd_live_mask(int km)
{
    uint64_t m = 0;
#define HJD_LM(P, N) if ((P) <= km) m |= 1ull << (N);
    HJD_ZZ_LIST(HJD_LM)
#undef HJD_LM
    return m;
}

// q: HjdQuantSet::qp (byte-packed pairs).  Dequantise one block held as 8 x uint4 (zig-zag order) into
// bp[natural] = fl(C(u)C(v) * (float)(short)(coef*q)), stored as row pairs: bp2[(v>>1)*8+u] = (bp[8v+u], bp[8(v+1)+u]), v even.
// Only zig-zag positions <= KM are computed; the others are zero by the block's length and are set to zero.
// Returns A_ac = sum over AC terms of |bp| ; *a_dc = |bp[0]|.
template <int KM>
__device__ __forceinline__ float hjd_dequant_block(const uint4 c[8], const uint4 q[8], float2 bp2[32], float* a_dc)
{
    const float cc0 = c_cc0, cc00 = c_cc00;
    const uint32_t* cw = (const uint32_t*)c;
    const uint32_t* qw = (const uint32_t*)q;
    float a_ac = 0.f;
#define HJD_DQ(P, N)                                                                           \
    if ((P) > KM) {                                                                            \
        if (((N) >> 3) & 1) bp2[((N) >> 4) * 8 + ((N) & 7)].y = 0.f;                            \
        else                bp2[((N) >> 4) * 8 + ((N) & 7)].x = 0.f;                            \
    } else {                                                                                   \
        /* coef*q straight from the packed pair (loadjpg.cpp:150; the product is exact) */      \
        const int prod = ((P) & 1) ? hjd_dp2a_hi_su(cw[(P) >> 1], qw[(P) >> 1])                \
                                   : hjd_dp2a_lo_su(cw[(P) >> 1], qw[(P) >> 1]);               \
        const float f = (float)(int)(short)prod;            /* stored to short */              \
        const float ccw = ((N) == 0) ? cc00 : ((((N) & 7) == 0 || ((N) >> 3) == 0) ? cc0 : 1.0f); \
        const float b = __fmul_rn(ccw, f);                  /* (C(u)*C(v)) * block[u][v] */    \
        if (((N) >> 3) & 1) bp2[((N) >> 4) * 8 + ((N) & 7)].y = b;                              \
        else                bp2[((N) >> 4) * 8 + ((N) & 7)].x = b;                              \
        if ((N) == 0) *a_dc = fabsf(b); else a_ac += fabsf(b);                                 \
    }
    HJD_ZZ_LIST(HJD_DQ)
#undef HJD_DQ
    return a_ac;
}

// d = {sat_s8(a), sat_s8(b)} in the low half-word, c's low half-word in the high one.  Flipping the top
// bit of each byte afterwards adds 128: sat_u8(v + 128) == sat_s8(v) ^ 0x80, once per word instead of
// once per sample.
__device__ __forceinline__ uint32_t hjd_pack_sat_s8(int a, int b, uint32_t c)
{
    uint32_t d;
    asm("cvt.pack.sat.s8.s32.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}

// d = {sat_u8(a), sat_u8(b)} in the low half-word, c's low half-word in the high one: clamp + pack.
__device__ __forceinline__ uint32_t hjd_pack_sat_u8(int a, int b, uint32_t c)
{
    uint32_t d;
    asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}

// Exact re-evaluation of sample (x, y) in the reference's order.  tx/ty: rows of the cos table.
__device__ __forceinline__ float hjd_exact_sum(const float2 bp2[32], const float* tx, const float* ty)
{
    float sum = 0.f;
#pragma unroll
    for (int u = 0; u < 8; u++) {
        const float cxu = tx[u];
#pragma unroll
        for (int v = 0; v < 8; v++)
            sum = __fadd_rn(sum, __fmul_rn(__fmul_rn((v & 1) ? bp2[(v >> 1) * 8 + u].y : bp2[(v >> 1) * 8 + u].x, cxu), ty[v]));
    }
    return sum;
}

__device__ __forceinline__ void hjd_ldg256(const uint4* p, uint4& a, uint4& b)
{
    asm volatile("ld.global.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(a.x), "=r"(a.y), "=r"(a.z), "=r"(a.w), "=r"(b.x), "=r"(b.y), "=r"(b.z), "=r"(b.w) : "l"(p));
}
__device__ __forceinline__ void hjd_ldg256_nc(const uint4* p, uint4& a, uint4& b)
{
    asm volatile("ld.global.nc.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(a.x), "=r"(a.y), "=r"(a.z), "=r"(a.w), "=r"(b.x), "=r"(b.y), "=r"(b.z), "=r"(b.w) : "l"(p));
}

// Pass 1 of one output column x for the frequencies that variant KM keeps:
//   r[vp] = (r[2vp][x], r[2vp+1][x]),  r[v][x] = sum_u bp[8v+u] * cos[x][u],  u over the live columns of row pair vp.
// The dead entries of bp2 hold zeros (the dequantisation step cleared them), so leaving them out changes nothing.
template <int KM, int X>
__device__ __forceinline__ void hjd_pass1_column(const float2 bp2[32], float2 r[4])
{
    constexpr uint64_t L = hjd_live_mask(KM);
#pragma unroll
    for (int vp = 0; vp < 4; vp++) {
        float2 acc = bp2[vp * 8];                  // cos[x][0] == 1
#pragma unroll
        for (int u = 1; u < 8; u++)
            if (((L >> (16 * vp + u)) | (L >> (16 * vp + 8 + u))) & 1)
                acc = __ffma2_rn(bp2[vp * 8 + u], c_cos2[X * 8 + u], acc);
        r[vp] = acc;
    }
}

// One 8x8 block: dequantise, IDCT, +128, clamp; rows go to dst[y*pitch + 0..7] (planes in HBM for the
// unfused kernel, a shared-memory tile for the fused one).  s_cos: the cos table in shared memory (the
// exact re-evaluation indexes it dynamically).
// Short blocks: when NONE of the lanes that are here together holds a coefficient beyond zig-zag index 20
// (u + v <= 5: the usual case for the chroma blocks of a warp, 79 % on the q85 workload; a warp's 32 luma
// blocks practically never qualify), the dequantisation and pass 1 leave those frequencies out.  The two
// variants are arms of small warp-uniform switches inside ONE body -- pass 2, the epilogue and the exact path
// are shared -- because the kernel has to stay around the 32 KB of the instruction cache (see DESIGN 4.6:
// complete copies of this routine per length class executed 17 % fewer instructions and ran 45 % slower).
__device__ __forceinline__ void hjd_idct_block(const uint4* __restrict__ cp, const uint4* __restrict__ qp,
                                               const float* s_cos, uint8_t* dst, uint32_t pitch)
{
    // 256-bit loads (sm_100 LDG.256): a lane owns a whole 128-byte line, and every instruction of the
    // warp touches 32 different lines, so wider loads halve the L1 wavefronts of this kernel
    uint4 c[8], q[8];
#pragma unroll
    for (int i = 0; i < 4; i++) { hjd_ldg256(cp + 2 * i, c[2 * i], c[2 * i + 1]); hjd_ldg256_nc(qp + 2 * i, q[2 * i], q[2 * i + 1]); }
    int cls;
    {
        // any coefficient at zig-zag index 21..63?  (the odd half of word 10, words 11..31)
        const uint32_t* cw = (const uint32_t*)c;
        uint32_t tail = cw[10] >> 16;
#pragma unroll
        for (int k = 11; k < 32; k++) tail |= cw[k];
        cls = __any_sync(__activemask(), tail != 0u) ? 3 : 1;
    }

    float2 bp2[32];
    float a_dc, a_ac;
#ifndef HJD_IDCT_VARIANTS
#define HJD_IDCT_VARIANTS 2
#endif
    if (HJD_IDCT_VARIANTS == 1) cls = 3;
    if (cls <= 1) {
        a_ac = hjd_dequant_block<20>(c, q, bp2, &a_dc);
    } else {
        a_ac = hjd_dequant_block<63>(c, q, bp2, &a_dc);
    }
    // re-evaluation window on the 0.25*sum scale: 24 * 2^-24 * A; DC-only blocks are exact (no window)
    const float win = (a_ac == 0.f) ? -1.f : (a_ac + a_dc) * 1.430511474609375e-06f;

    const float2* cosp = (const float2*)c_cosq;    // cosp[y*4+vp] = 0.25 * (cos[y][2vp], cos[y][2vp+1])
    // Packed FP32x2 FMAs (Blackwell FFMA2) halve the issue slots of this issue-bound kernel.  Column by column:
    // pass 1 (horizontal frequency u -> position x) for two coefficient rows per instruction, then
    // pass 2 (vertical frequency v -> position y), pack rows, collect near-integer samples:
    // |h - rint(h)| <= win  <=  an integer (truncation boundary) lies within the error window of h;
    // everywhere else trunc(h) is provably the reference's value.
    // With A < 1e5 neither short wrap of the reference (loadjpg.cpp:136-137) can trigger (|h| <= A/4), so
    // the sample is sat_u8(trunc(h) + 128), and the clamp comes free with the byte packing
    // (cvt.pack.sat.u8.s32).  Absurd blocks (A >= 1e5) take the exact path for every sample.
    uint32_t row_lo[8], row_hi[8];
#pragma unroll
    for (int y = 0; y < 8; y++) { row_lo[y] = 0; row_hi[y] = 0; }
    uint32_t near_lo = 0, near_hi = 0;             // bit (8y + x)
#define HJD_COLUMN_PAIR(X)                                                                                     \
    {                                                                                                          \
        float2 ra[4], rb[4];                                                                                   \
        if (cls <= 1) { hjd_pass1_column<20, X>(bp2, ra); hjd_pass1_column<20, (X) + 1>(bp2, rb); }            \
        else          { hjd_pass1_column<63, X>(bp2, ra); hjd_pass1_column<63, (X) + 1>(bp2, rb); }            \
        _Pragma("unroll")                                                                                      \
        for (int y = 0; y < 8; y++) {                                                                          \
            /* pass 2: even and odd vertical frequencies accumulate in the two halves; the table carries the */ \
            /* 0.25 (0.25 * fl(s) == fl(0.25 * s): scaling by a power of two commutes with rounding)         */ \
            float2 a2 = __fmul2_rn(ra[0], cosp[y * 4]), b2 = __fmul2_rn(rb[0], cosp[y * 4]);                   \
            _Pragma("unroll")                                                                                  \
            for (int vp = 1; vp < 4; vp++) {                                                                   \
                a2 = __ffma2_rn(ra[vp], cosp[y * 4 + vp], a2);                                                 \
                b2 = __ffma2_rn(rb[vp], cosp[y * 4 + vp], b2);                                                 \
            }                                                                                                  \
            const float2 h2 = make_float2(a2.x + a2.y, b2.x + b2.y);                                           \
            /* rint(h) as (h + 1.5*2^23) - 1.5*2^23 (|h| < 2^22 whenever the window is in use), for the two  */ \
            /* columns at once with packed adds: no FRND on the conversion unit, half the issue slots        */ \
            const float2 hr2 = __fadd2_rn(__fadd2_rn(h2, make_float2(12582912.0f, 12582912.0f)),               \
                                          make_float2(-12582912.0f, -12582912.0f));                            \
            const float2 d2 = __fadd2_rn(h2, make_float2(-hr2.x, -hr2.y));                                     \
            const bool near_a = fabsf(d2.x) <= win, near_b = fabsf(d2.y) <= win;                               \
            const int ia = __float2int_rz(h2.x), ib = __float2int_rz(h2.y);   /* (int)(0.25*sum), loadjpg.cpp:123 */ \
            if (y < 4) { if (near_a) near_lo |= 1u << (8 * y + (X)); if (near_b) near_lo |= 1u << (8 * y + (X) + 1); }             \
            else       { if (near_a) near_hi |= 1u << (8 * (y - 4) + (X)); if (near_b) near_hi |= 1u << (8 * (y - 4) + (X) + 1); } \
            if ((X) < 4) row_lo[y] = hjd_pack_sat_s8(ib, ia, row_lo[y]);                                       \
            else         row_hi[y] = hjd_pack_sat_s8(ib, ia, row_hi[y]);                                       \
        }                                                                                                      \
    }
    // pairs (2,3) (0,1) (6,7) (4,5): high half-word first
    HJD_COLUMN_PAIR(2) HJD_COLUMN_PAIR(0) HJD_COLUMN_PAIR(6) HJD_COLUMN_PAIR(4)
#undef HJD_COLUMN_PAIR
    if (a_ac + a_dc >= 1.0e5f) { near_lo = 0xFFFFFFFFu; near_hi = 0xFFFFFFFFu; }

#pragma unroll
    for (int y = 0; y < 8; y++)
        *(uint2*)(dst + (size_t)y * pitch) = make_uint2(row_lo[y] ^ 0x80808080u, row_hi[y] ^ 0x80808080u);

    // exact re-evaluation of the flagged samples (same thread, later store wins)
    while (near_lo | near_hi) {
        int pos;
        if (near_lo) { pos = __ffs(near_lo) - 1; near_lo &= near_lo - 1; }
        else         { pos = 32 + __ffs(near_hi) - 1; near_hi &= near_hi - 1; }
        const int y = pos >> 3, x = pos & 7;
        const float sum = hjd_exact_sum(bp2, s_cos + x * 8, s_cos + y * 8);
        dst[(size_t)y * pitch + x] = (uint8_t)hjd_finish_sample(sum);
    }
}

__global__ void __launch_bounds__(HJD_IDCT_THREADS, 4)
hjd_k_idct_planes(const int16_t* __restrict__ coef, const HjdImageDesc* __restrict__ imgs,
                  const HjdQuantSet* __restrict__ qsets, uint8_t* __restrict__ planes, int img_base)
{
    __shared__ float s_cos[64];
    if (threadIdx.x < 64) s_cos[threadIdx.x] = c_cos[threadIdx.x];
    __syncthreads();

    const HjdImageDesc* d = imgs + (blockIdx.y + img_base);
    const uint64_t b = (uint64_t)blockIdx.x * HJD_IDCT_THREADS + threadIdx.x;
    if (b >= d->n_blocks) return;
    const uint32_t bpm = d->blocks_per_mcu;
    const uint32_t mcu = (uint32_t)(b / bpm), bi = (uint32_t)(b - (uint64_t)mcu * bpm);
    const uint32_t my = mcu / d->mcus_x, mx = mcu - my * d->mcus_x;
    const uint32_t ny = d->ncomp == 3 ? (uint32_t)d->hf * d->vf : 1u;
    int comp; uint32_t bx, by, pitch; uint64_t poff;
    if (bi < ny) {                     // Y blocks, row-major inside the MCU (loadjpg.cpp:949-959)
        comp = 0; pitch = d->y_pitch; poff = d->y_off;
        bx = mx * d->hf + bi % d->hf; by = my * d->vf + bi / d->hf;
    } else {
        comp = (bi == ny) ? 1 : 2; pitch = d->c_pitch; poff = comp == 1 ? d->cb_off : d->cr_off;
        bx = mx; by = my;
    }
    hjd_idct_block((const uint4*)(coef + (d->block_base + b) * 64), (const uint4*)(qsets[d->quant_set].qp[comp]),
                   s_cos, planes + poff + (uint64_t)by * 8 * pitch + (uint64_t)bx * 8, pitch);
}

cudaError_t hjd_launch_idct_planes(const int16_t* coef, const HjdImageDesc* imgs, const HjdQuantSet* qsets,
                                   uint8_t* planes, int n_images, uint32_t max_blocks, cudaStream_t st)
{
    if (n_images <= 0 || max_blocks == 0) return cudaSuccess;
    const unsigned gx = (max_blocks + HJD_IDCT_THREADS - 1) / HJD_IDCT_THREADS;
    for (int base = 0; base < n_images; base += 65535) {
        const int n = min(65535, n_images - base);
        hjd_k_idct_planes<<<dim3(gx, n), HJD_IDCT_THREADS, 0, st>>>(coef, imgs, qsets, planes, base);
    }
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// kernel 3: chroma upsample + YCbCr -> RGB + clamp
// ------------------------------------------------------------------------------------------
// One thread = 16 pixels of one row = 48 output bytes = three 128-bit stores.  Float arithmetic
// is the reference's, operation for operation (no FMA contraction, truncation toward zero):
//   R = Y + 1.402f*(Cr-128);  G = (Y - 0.34414f*(Cb-128)) - 0.71414f*(Cr-128);  B = Y + 1.772f*(Cb-128)
// (loadjpg.cpp:873-879 with the swapped argument names of the call at 918 resolved).
// Chroma is replicated, nearest neighbour (loadjpg.cpp:911-912).

// The kernel is issue-bound before it is HBM-bound, so every pixel uses the fewest instructions
// that still reproduce the reference bit for bit: byte -> float is one I2F with a byte selector,
// truncation toward zero is one F2I.TRUNC, and the clamp to [0, 255] comes free with the byte
// packing (cvt.pack.sat.u8.s32 packs and saturates two values per instruction).
template <int SEL>
__device__ __forceinline__ float hjd_byte_to_float(uint32_t word)
{
    return (float)((word >> (8 * SEL)) & 255u);
}

// Chroma terms of NC chroma samples: (1.402*(Cr-128), 0.34414*(Cb-128), 0.71414*(Cr-128), 1.772*(Cb-128)),
// each product rounded once as in loadjpg.cpp:873-879.  Shared by every luma sample that maps to the
// chroma sample (2x1, 1x2 or 2x2 of them): nearest-neighbour upsampling, loadjpg.cpp:911-912.
template <int NC>
__device__ __forceinline__ void hjd_chroma_terms(const uint32_t* cbw, const uint32_t* crw, float4* terms)
{
#pragma unroll
    for (int ci = 0; ci < NC; ci++) {
        float cb, cr;
        switch (ci & 3) {
            case 0: cb = hjd_byte_to_float<0>(cbw[ci >> 2]); cr = hjd_byte_to_float<0>(crw[ci >> 2]); break;
            case 1: cb = hjd_byte_to_float<1>(cbw[ci >> 2]); cr = hjd_byte_to_float<1>(crw[ci >> 2]); break;
            case 2: cb = hjd_byte_to_float<2>(cbw[ci >> 2]); cr = hjd_byte_to_float<2>(crw[ci >> 2]); break;
            default: cb = hjd_byte_to_float<3>(cbw[ci >> 2]); cr = hjd_byte_to_float<3>(crw[ci >> 2]); break;
        }
        cb = __fadd_rn(cb, -128.0f);      // (float)(Cb - 128), exact
        cr = __fadd_rn(cr, -128.0f);
        terms[ci] = make_float4(__fmul_rn(1.402f, cr), __fmul_rn(0.34414f, cb), __fmul_rn(0.71414f, cr), __fmul_rn(1.772f, cb));
    }
}

// NP luma samples (8 or 16) + their chroma terms -> 3*NP packed bytes.  HS = log2(horizontal luma factor).
template <int HS, int NP>
__device__ __forceinline__ void hjd_color_apply(const uint32_t* yw, const float4* terms, uint32_t* out)
{
    int ch[3 * NP];                       // R, G, B before clamping
#pragma unroll
    for (int i = 0; i < NP; i++) {
        const float4 t = terms[i >> HS];
        float fy;
        switch (i & 3) {
            case 0: fy = hjd_byte_to_float<0>(yw[i >> 2]); break;
            case 1: fy = hjd_byte_to_float<1>(yw[i >> 2]); break;
            case 2: fy = hjd_byte_to_float<2>(yw[i >> 2]); break;
            default: fy = hjd_byte_to_float<3>(yw[i >> 2]); break;
        }
        // loadjpg.cpp:873-879 with the argument swap of the call at 918 resolved; (int) truncates
        ch[3 * i]     = __float2int_rz(__fadd_rn(fy, t.x));
        ch[3 * i + 1] = __float2int_rz(__fsub_rn(__fsub_rn(fy, t.y), t.z));
        ch[3 * i + 2] = __float2int_rz(__fadd_rn(fy, t.w));
    }
#pragma unroll
    for (int w = 0; w < 3 * NP / 4; w++)  // Clamp (loadjpg.cpp:83-91) + pack, two values per instruction
        out[w] = hjd_pack_sat_u8(ch[4 * w + 1], ch[4 * w], hjd_pack_sat_u8(ch[4 * w + 3], ch[4 * w + 2], 0u));
}

// Byte idx of a word array as float (idx is a compile-time constant after unrolling: one I2F.U8 with a byte selector).
__device__ __forceinline__ float hjd_byte_f(const uint32_t* w, int idx)
{
    return (float)((w[idx >> 2] >> (8 * (idx & 3))) & 255u);
}
// The same byte under the exponent of 2^23: the float 8388608 + byte, exactly, with one PRMT on the ALU pipe instead of
// a conversion on the quarter-rate XU pipe; the caller subtracts 8388608 (+ 128 for chroma) in the packed add it does anyway.
__device__ __forceinline__ float hjd_byte_m(const uint32_t* w, int idx)
{
    return __uint_as_float(__byte_perm(w[idx >> 2], 0x4B000000u, 0x7540u | (uint32_t)(idx & 3)));
}

#ifdef HJD_COLOR_SCALAR
template <int HS, int NP>
__device__ __forceinline__ void hjd_color_n(const uint32_t* yw, const uint32_t* cbw, const uint32_t* crw, uint32_t* out)
{
    float4 terms[NP >> HS];
    hjd_chroma_terms<(NP >> HS)>(cbw, crw, terms);
    hjd_color_apply<HS, NP>(yw, terms, out);
}
#else
// The same arithmetic as hjd_chroma_terms + hjd_color_apply with packed FP32x2 instructions: chroma
// samples (2p, 2p+1) share a register pair, and so do the two pixels that use them -- neighbours for
// 4:4:4, two apart for 2:1 horizontal sampling.  Every lane of a packed add / multiply is the IEEE
// operation of the scalar code (rounded once, never fused), and -(a*b) == (-a)*b exactly, so
// G = (y - 0.34414 cb) - 0.71414 cr keeps its two roundings.  A third fewer issue slots than scalar.
template <int HS, int NP, bool BGR = false>      // BGR: byte order of the reference's BMP writer (openjpg.cpp:559-561)
__device__ __forceinline__ void hjd_color_n(const uint32_t* yw, const uint32_t* cbw, const uint32_t* crw, uint32_t* out)
{
    constexpr int NC = NP >> HS, D = 1 << HS;
    static_assert(NC % 2 == 0, "chroma samples are processed in pairs");
    float2 tx[NC / 2], tyn[NC / 2], tzn[NC / 2], tw[NC / 2];
    const float2 m128 = make_float2(-8388736.0f, -8388736.0f);      // -(2^23 + 128)
    const float2 m0 = make_float2(-8388608.0f, -8388608.0f);
#pragma unroll
    for (int p = 0; p < NC / 2; p++) {
        const float2 cb = __fadd2_rn(make_float2(hjd_byte_m(cbw, 2 * p), hjd_byte_m(cbw, 2 * p + 1)), m128);   // (float)(Cb - 128), exact
        const float2 cr = __fadd2_rn(make_float2(hjd_byte_m(crw, 2 * p), hjd_byte_m(crw, 2 * p + 1)), m128);
        tx[p]  = __fmul2_rn(make_float2(1.402f, 1.402f), cr);
        tyn[p] = __fmul2_rn(make_float2(-0.34414f, -0.34414f), cb);
        tzn[p] = __fmul2_rn(make_float2(-0.71414f, -0.71414f), cr);
        tw[p]  = __fmul2_rn(make_float2(1.772f, 1.772f), cb);
    }
    int ch[3 * NP];                       // R, G, B before clamping
#pragma unroll
    for (int i = 0; i < NP; i++) {
        if (((i >> HS) & 1) != 0) continue;                  // second pixel of a pair
        const int j = i + D, p = (i >> HS) >> 1;
        const float2 y2 = __fadd2_rn(make_float2(hjd_byte_m(yw, i), hjd_byte_m(yw, j)), m0);      // (float)Y, exact
        // loadjpg.cpp:873-879 with the argument swap of the call at 918 resolved; (int) truncates
        const float2 r2 = __fadd2_rn(y2, tx[p]);
        const float2 g2 = __fadd2_rn(__fadd2_rn(y2, tyn[p]), tzn[p]);
        const float2 b2 = __fadd2_rn(y2, tw[p]);
        ch[3 * i + (BGR ? 2 : 0)] = __float2int_rz(r2.x); ch[3 * i + 1] = __float2int_rz(g2.x); ch[3 * i + (BGR ? 0 : 2)] = __float2int_rz(b2.x);
        ch[3 * j + (BGR ? 2 : 0)] = __float2int_rz(r2.y); ch[3 * j + 1] = __float2int_rz(g2.y); ch[3 * j + (BGR ? 0 : 2)] = __float2int_rz(b2.y);
    }
#pragma unroll
    for (int w = 0; w < 3 * NP / 4; w++)  // Clamp (loadjpg.cpp:83-91) + pack, two values per instruction
        out[w] = hjd_pack_sat_u8(ch[4 * w + 1], ch[4 * w], hjd_pack_sat_u8(ch[4 * w + 3], ch[4 * w + 2], 0u));
}
#endif

template <int HS>
__device__ __forceinline__ void hjd_color_16(const uint32_t yw[4], const uint32_t cbw[4], const uint32_t crw[4],
                                             uint32_t out[12])
{
    hjd_color_n<HS, 16>(yw, cbw, crw, out);
}

__global__ void __launch_bounds__(HJD_COLOR_THREADS)
hjd_k_color(const uint8_t* __restrict__ planes, const HjdImageDesc* __restrict__ imgs,
            uint8_t* __restrict__ rgb, int img_base)
{
    const HjdImageDesc* d = imgs + (blockIdx.y + img_base);
    const uint32_t W = d->width, H = d->height;
    const uint32_t segs = (W + 15) >> 4;
    const uint64_t t = (uint64_t)blockIdx.x * HJD_COLOR_THREADS + threadIdx.x;
    if (t >= (uint64_t)segs * H) return;
    const uint32_t row = (uint32_t)(t / segs), seg = (uint32_t)(t - (uint64_t)row * segs);
    const uint32_t x0 = seg * 16;
    const int hs = d->hf - 1, vs = d->vf - 1;      // shifts (factors are 1 or 2)
    const bool gray = d->ncomp == 1;

    const uint8_t* yp = planes + d->y_off + (uint64_t)row * d->y_pitch + x0;
    uint32_t yw[4];
    { const uint2 a = *(const uint2*)yp, b = *(const uint2*)(yp + 8); yw[0] = a.x; yw[1] = a.y; yw[2] = b.x; yw[3] = b.y; }
    uint32_t cbw[4] = {0x80808080u, 0x80808080u, 0x80808080u, 0x80808080u};
    uint32_t crw[4] = {0x80808080u, 0x80808080u, 0x80808080u, 0x80808080u};
    if (!gray) {
        const uint64_t coff = (uint64_t)(row >> vs) * d->c_pitch + (x0 >> hs);
        const uint8_t* bp = planes + d->cb_off + coff;
        const uint8_t* rp = planes + d->cr_off + coff;
        { const uint2 a = *(const uint2*)bp; cbw[0] = a.x; cbw[1] = a.y; }
        { const uint2 a = *(const uint2*)rp; crw[0] = a.x; crw[1] = a.y; }
        if (hs == 0) {
            { const uint2 a = *(const uint2*)(bp + 8); cbw[2] = a.x; cbw[3] = a.y; }
            { const uint2 a = *(const uint2*)(rp + 8); crw[2] = a.x; crw[3] = a.y; }
        }
    }

    uint32_t out[12];
    if (hs) hjd_color_16<1>(yw, cbw, crw, out); else hjd_color_16<0>(yw, cbw, crw, out);

    uint8_t* dst = rgb + d->rgb_off + ((uint64_t)row * W + x0) * 3;    // loadjpg.cpp:921-925
    const uint32_t npix = min(16u, W - x0);
    if (npix == 16 && (((uintptr_t)dst) & 15) == 0) {
        uint4* o = (uint4*)dst;
        o[0] = make_uint4(out[0], out[1], out[2], out[3]);
        o[1] = make_uint4(out[4], out[5], out[6], out[7]);
        o[2] = make_uint4(out[8], out[9], out[10], out[11]);
    } else {
        const uint32_t nbytes = npix * 3;
#pragma unroll
        for (int i = 0; i < 48; i++)
            if ((uint32_t)i < nbytes) dst[i] = (uint8_t)(out[i >> 2] >> (8 * (i & 3)));
    }
}

cudaError_t hjd_launch_color(const uint8_t* planes, const HjdImageDesc* imgs, uint8_t* rgb, int n_images,
                             uint32_t max_width, uint32_t max_height, cudaStream_t st)
{
    if (n_images <= 0 || max_width == 0) return cudaSuccess;
    const uint64_t threads = (uint64_t)((max_width + 15) >> 4) * max_height;
    const unsigned gx = (unsigned)((threads + HJD_COLOR_THREADS - 1) / HJD_COLOR_THREADS);
    for (int base = 0; base < n_images; base += 65535) {
        const int n = min(65535, n_images - base);
        hjd_k_color<<<dim3(gx, n), HJD_COLOR_THREADS, 0, st>>>(planes, imgs, rgb, base);
    }
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// kernels 2+3 fused per MCU (the default path): one thread decodes a whole MCU to RGB
// ------------------------------------------------------------------------------------------
// The reference couples DecodeMCU and YCrCB_to_RGB24_Block8x8 per MCU (loadjpg.cpp:1179-1180); so
// does this kernel, with no barrier at all: a thread runs the IDCT of its MCU's Cb and Cr blocks into
// thread-private shared-memory tiles, then, Y block by Y block, the IDCT into a third private tile
// followed at once by upsampling + colour conversion of those 8x8 pixels and 24-byte row stores.
// Planes never reach HBM.  Tiles are interleaved by thread (row r of thread t at [(r*T + t) * 8 B])
// so row stores and loads are bank-conflict free; the exact re-evaluation patches bytes in the tile
// before the colour step reads them.
#ifndef HJD_MCU_MINBLOCKS
#define HJD_MCU_MINBLOCKS 4
#endif
#define HJD_BMP_PIXEL_OFF   64      // pixel array at +64 of an image's slab region, so the 54-byte header starts at +10
#define HJD_BMP_FILE_OFF    10
template <bool FLAT, bool BMP>     // FLAT: exact 1-D grid with an image look-up; BMP: the reference's BMP file layout (see below)
__global__ void __launch_bounds__(HJD_MCU_THREADS, HJD_MCU_MINBLOCKS)
hjd_k_mcu_rgb(const int16_t* __restrict__ coef, const HjdImageDesc* __restrict__ imgs,
              const HjdQuantSet* __restrict__ qsets, uint8_t* __restrict__ rgb,
              const uint32_t* __restrict__ mcu_prefix, int n_images, int img_base)
{
    __shared__ float s_cos[64];
    __shared__ uint2 s_tile[4][8 * HJD_MCU_THREADS];             // Y (left), Y (right), Cb, Cr: 8 rows x T threads x 8 bytes
    const uint32_t t = threadIdx.x;
    if (t < 64) s_cos[t] = c_cos[t];
    __syncthreads();

    // Two grid shapes (device_common.cuh), two instantiations: the kernel sits at the 128-register cap, and a
    // run-time switch cost 2 %.
    const HjdImageDesc* d;
    uint32_t m;
    if (!hjd_locate<FLAT, HJD_MCU_THREADS>(imgs, mcu_prefix, n_images, img_base, d, m)) return;
    if (m >= d->n_mcus || d->blocks_per_mcu == 0) return;
    const uint32_t hf = d->hf, vf = d->vf, bpm = d->blocks_per_mcu;
    const bool gray = d->ncomp == 1;
    const uint32_t ny = gray ? 1u : hf * vf;
    const uint32_t my = m / d->mcus_x, mx = m - my * d->mcus_x;
    const int hs = (int)hf - 1, vs = (int)vf - 1;
    const HjdQuantSet* qs = qsets + d->quant_set;
    const uint4* cp = (const uint4*)(coef + (d->block_base + (uint64_t)m * bpm) * 64);
    constexpr uint32_t kPitch = HJD_MCU_THREADS * 8;
    uint8_t* tY0 = (uint8_t*)&s_tile[0][t];
    uint8_t* tY1 = (uint8_t*)&s_tile[1][t];
    uint8_t* tCb = (uint8_t*)&s_tile[2][t];
    uint8_t* tCr = (uint8_t*)&s_tile[3][t];

    const uint32_t W = d->width, H = d->height;
    // RGB: top-down, stride 3W (loadjpg.cpp:921-925).  BMP: the file WriteBMP24 would write (openjpg.cpp:504-570),
    // laid out in the image's slab region from +HJD_BMP_FILE_OFF: 54-byte header, then rows bottom-up, B G R,
    // each padded with zeros to a multiple of four bytes; the pixel array starts 64-byte aligned.
    const uint64_t img_pitch = BMP ? (uint64_t)((W * 3 + 3) & ~3u) : (uint64_t)W * 3;
    uint8_t* img_rgb = rgb + d->rgb_off + (BMP ? HJD_BMP_PIXEL_OFF : 0);
    const uint32_t px = mx * hf * 8;                              // left edge of the MCU
    const uint32_t npix = px < W ? min(8u * hf, W - px) : 0u;     // loadjpg.cpp:907
    if (BMP && m == 0) {                                          // the header, by the thread of the first MCU
        uint8_t* hp = rgb + d->rgb_off + HJD_BMP_FILE_OFF;
        const uint32_t file_size = (uint32_t)(img_pitch * H) + 54u;                    // openjpg.cpp:541
        const uint32_t words[13] = {file_size, 0u, 54u, 40u, W, H, 1u | 24u << 16, 0u, 0u, 0u, 0u, 0u, 0u};
        hp[0] = 'B'; hp[1] = 'M';
#pragma unroll
        for (int k = 0; k < 13; k++)
#pragma unroll
            for (int qq = 0; qq < 4; qq++) hp[2 + 4 * k + qq] = (uint8_t)(words[k] >> (8 * qq));
    }
    // one loop, one inlined IDCT: iterations 0,1 = Cb, Cr (colour images), then the Y blocks in decode order;
    // after the last Y block of a block row, that row of the MCU (8 or 16 pixels wide) goes out as RGB
    const uint32_t n_pre = gray ? 0u : 2u;
#pragma unroll 1
    for (uint32_t it = 0; it < n_pre + ny; it++) {
        const bool chroma = it < n_pre;
        const uint32_t bi = chroma ? ny + it : it - n_pre;        // block index inside the MCU
        if (it + 1 < n_pre + ny) {                                // next block's 128-byte line -> L1 while this one computes
            const uint32_t nbi = (it + 1 < n_pre) ? ny + it + 1 : it + 1 - n_pre;
            asm volatile("prefetch.global.L1 [%0];" :: "l"(cp + nbi * 8));
        }
        const uint32_t bx = chroma ? 0u : bi % hf, by = chroma ? 0u : bi / hf;
        hjd_idct_block(cp + bi * 8, (const uint4*)qs->qp[chroma ? 1 + it : 0], s_cos,
                       chroma ? (it ? tCr : tCb) : (bx ? tY1 : tY0), kPitch);
        if (chroma || bx + 1 < hf || npix == 0) continue;
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
            uint8_t* dst = img_rgb + (uint64_t)(BMP ? H - 1 - py : py) * img_pitch + (uint64_t)px * 3;      // loadjpg.cpp:921-925 / openjpg.cpp:555
            const uint2 ya = *(const uint2*)(tY0 + r * kPitch);
            if (hs) {                                             // 16 pixels: 48 bytes, three 128-bit stores
                const uint2 yb = *(const uint2*)(tY1 + r * kPitch);
                const uint32_t yw[4] = {ya.x, ya.y, yb.x, yb.y};
                uint32_t out[12];
                hjd_color_n<1, 16, BMP>(yw, cbw, crw, out);
                if (npix == 16 && (((uintptr_t)dst) & 15) == 0) {
                    uint4* o = (uint4*)dst;
                    o[0] = make_uint4(out[0], out[1], out[2], out[3]);
                    o[1] = make_uint4(out[4], out[5], out[6], out[7]);
                    o[2] = make_uint4(out[8], out[9], out[10], out[11]);
                } else {
#pragma unroll
                    for (int i = 0; i < 48; i++)
                        if ((uint32_t)i < npix * 3) dst[i] = (uint8_t)(out[i >> 2] >> (8 * (i & 3)));
                }
            } else {                                              // 8 pixels: 24 bytes
                const uint32_t yw[2] = {ya.x, ya.y};
                uint32_t out[6];
                hjd_color_n<0, 8, BMP>(yw, cbw, crw, out);
                if (npix == 8 && (((uintptr_t)dst) & 7) == 0) {
                    uint2* o = (uint2*)dst;
                    o[0] = make_uint2(out[0], out[1]);
                    o[1] = make_uint2(out[2], out[3]);
                    o[2] = make_uint2(out[4], out[5]);
                } else {
#pragma unroll
                    for (int i = 0; i < 24; i++)
                        if ((uint32_t)i < npix * 3) dst[i] = (uint8_t)(out[i >> 2] >> (8 * (i & 3)));
                }
            }
            if constexpr (BMP) {
                if (px + npix == W)                               // row padding, openjpg.cpp:563-567
                    for (uint32_t qq = W * 3; qq < (uint32_t)img_pitch; qq++) dst[qq - px * 3] = 0;
            }
        }
    }
}

// ------------------------------------------------------------------------------------------
// luma only (HJD_FLAG_GRAY_OUT): one thread decodes one luma block to its W x H crop of the Y plane
// ------------------------------------------------------------------------------------------
// The threads of an image take its luma blocks that hold a pixel, row-major over ceil(W/8) x ceil(H/8), so the
// lanes of a warp own horizontally adjacent blocks and each of the eight row stores of a warp covers up to 256
// contiguous bytes.  Chroma blocks and MCU-padding blocks are not read.  hjd_idct_block, unchanged, writes the
// block into a thread-private shared-memory tile interleaved by thread (as hjd_k_mcu_rgb does), where the exact
// re-evaluation patches its bytes; then the rows go out clipped at W and H, 8 bytes at once where aligned.
// Grids as hjd_k_mcu_rgb, over luma blocks instead of MCUs.
template <bool FLAT>
__global__ void __launch_bounds__(HJD_LUMA_THREADS, HJD_MCU_MINBLOCKS)
hjd_k_luma(const int16_t* __restrict__ coef, const HjdImageDesc* __restrict__ imgs,
           const HjdQuantSet* __restrict__ qsets, uint8_t* __restrict__ out,
           const uint32_t* __restrict__ luma_prefix, int n_images, int img_base)
{
    __shared__ float s_cos[64];
    __shared__ uint2 s_tile[8 * HJD_LUMA_THREADS];               // 8 rows x T threads x 8 bytes
    const uint32_t t = threadIdx.x;
    if (t < 64) s_cos[t] = c_cos[t];
    __syncthreads();

    const HjdImageDesc* d;
    uint32_t k;
    if (!hjd_locate<FLAT, HJD_LUMA_THREADS>(imgs, luma_prefix, n_images, img_base, d, k)) return;
    const uint32_t W = d->width, H = d->height;
    const uint32_t bw = (W + 7) >> 3;
    if (d->blocks_per_mcu == 0 || k >= bw * ((H + 7) >> 3)) return;
    const uint32_t by = k / bw, bx = k - by * bw;                 // block column / row in the Y plane
    const uint32_t hf = d->hf, vf = d->vf;                        // 1 or 2 (1 for one-component files)
    const uint32_t mx = bx / hf, my = by / vf;
    const uint32_t bi = (by - my * vf) * hf + (bx - mx * hf);     // Y blocks row-major inside the MCU (loadjpg.cpp:949-959)
    const uint64_t blk = d->block_base + (uint64_t)(my * d->mcus_x + mx) * d->blocks_per_mcu + bi;
    constexpr uint32_t kPitch = HJD_LUMA_THREADS * 8;
    uint8_t* tile = (uint8_t*)&s_tile[t];
    hjd_idct_block((const uint4*)(coef + blk * 64), (const uint4*)qsets[d->quant_set].qp[0], s_cos, tile, kPitch);

    const uint32_t x0 = bx * 8, y0 = by * 8;
    const uint32_t nx = min(8u, W - x0), nr = min(8u, H - y0);
    uint8_t* dst = out + d->rgb_off + (uint64_t)y0 * W + x0;
#pragma unroll 1
    for (uint32_t r = 0; r < nr; r++) {
        const uint2 v = *(const uint2*)(tile + r * kPitch);
        uint8_t* row = dst + (uint64_t)r * W;
        if (nx == 8 && (((uintptr_t)row) & 7) == 0) {
            *(uint2*)row = v;
        } else {
#pragma unroll
            for (uint32_t i = 0; i < 8; i++)
                if (i < nx) row[i] = (uint8_t)((i < 4 ? v.x : v.y) >> (8 * (i & 3)));
        }
    }
}

cudaError_t hjd_launch_luma(const int16_t* coef, const HjdImageDesc* imgs, const HjdQuantSet* qsets, uint8_t* out,
                            const uint32_t* luma_prefix, int n_images, uint32_t n_luma, uint32_t max_luma, cudaStream_t st)
{
    if (n_images <= 0 || n_luma == 0 || max_luma == 0) return cudaSuccess;
    hjd_launch_per_image(hjd_k_luma<false>, hjd_k_luma<true>, HJD_LUMA_THREADS, luma_prefix, n_images, n_luma, max_luma, st,
                         coef, imgs, qsets, out);
    return cudaGetLastError();
}

#include "mcu_tc.cuh"

// The IDCT matrix of the tensor-core kernel (see mcu_tc.cuh): M[k][8y+x] = 0.25 * C(u)C(v) * cos[x][u] * cos[y][v], the
// real-number product of the reference's float constants, split into M_hi * 2^-13 and M_lo (integers, exact in FP16)
// and laid out as the K-major, 128-byte-swizzled shared-memory tile tcgen05.mma reads: row n (0..63: M_hi of sample
// n = 8y+x; 64..127: M_lo), 64 FP16 per row in zig-zag order, 16-byte chunk j of row n at chunk j ^ (n & 7).
void hjd_build_idct_matrix(const float cos_tab[64], float cc0, float cc00, uint16_t img[8192])
{
    for (int k = 0; k < 64; k++) {
        const int nat = hjd_zz(k), u = nat & 7, v = nat >> 3;
        const double cc = nat == 0 ? (double)cc00 : ((u == 0 || v == 0) ? (double)cc0 : 1.0);
        for (int y = 0; y < 8; y++)
            for (int x = 0; x < 8; x++) {
                const double m = 0.25 * cc * (double)cos_tab[x * 8 + u] * (double)cos_tab[y * 8 + v];
                const double s = ldexp(m, 13);
                const int hi = (int)nearbyint(s);
                const int lo = (int)nearbyint(ldexp(s - hi, 11));
                for (int half = 0; half < 2; half++) {
                    const int row = half * 64 + 8 * y + x;
                    const size_t off = (size_t)(row >> 3) * 1024 + (size_t)(row & 7) * 128 + (size_t)(((k >> 3) ^ (row & 7)) << 4) + (size_t)(k & 7) * 2;
                    const __half h = __float2half(half ? (float)lo : ldexpf((float)hi, -13));
                    img[off / 2] = *(const uint16_t*)&h;
                }
            }
    }
}

static cudaError_t hjd_set_idct_matrix(const float cos_tab[64], float cc0, float cc00)
{
    static uint16_t img[HJD_TC_TILE_BYTES / 2];
    hjd_build_idct_matrix(cos_tab, cc0, cc00, img);
    return cudaMemcpyToSymbol(g_idct_mat, img, sizeof img);
}

static int g_tc_ctas[64];      // resident CTAs of the tensor-core kernel per device (one per SM), set by hjd_mcu_tc_init_device

cudaError_t hjd_launch_mcu_rgb(const int16_t* coef, const HjdImageDesc* imgs, const HjdQuantSet* qsets,
                               uint8_t* rgb, const uint32_t* mcu_prefix, int n_images, uint32_t n_mcus,
                               uint32_t max_mcus, bool bmp, int variant, cudaStream_t st)
{
    if (n_images <= 0 || n_mcus == 0 || max_mcus == 0) return cudaSuccess;
    if (variant == HJD_MCU_TENSOR_CORE) {
        // units of 128 MCUs, walked by the groups of one resident CTA per SM.  Images of similar size: unit = (image, 128 MCUs of it),
        // no look-up; clearly skewed or tiny-image batches: units over all MCUs of the batch, the image found by binary search
        // (an idle thread slot is cheap, a search in front of every unit is not: the rule of the CUDA-core kernel, over units).
        uint32_t units_x = (max_mcus + 127u) / 128u;
        uint64_t n_units = (uint64_t)units_x * (uint64_t)n_images;
        if (!hjd_grid_per_image(max_mcus, n_images, n_mcus, 128u) || n_units > 0xFFFFFFFFull) { units_x = 0; n_units = ((uint64_t)n_mcus + 127u) / 128u; }
        int dev = 0;
        cudaError_t e = cudaGetDevice(&dev);
        if (e != cudaSuccess) return e;
        const int resident = (dev >= 0 && dev < 64 && g_tc_ctas[dev] > 0) ? g_tc_ctas[dev] : 148;
        const unsigned g = (unsigned)min((uint64_t)resident, (n_units + HJD_TC_GROUPS - 1) / HJD_TC_GROUPS);
        if (bmp) hjd_k_mcu_rgb_tc<true><<<g, HJD_TC_THREADS, HJD_TC_SMEM_BYTES, st>>>(coef, imgs, qsets, rgb, mcu_prefix, n_images, (uint32_t)n_units, units_x);
        else hjd_k_mcu_rgb_tc<false><<<g, HJD_TC_THREADS, HJD_TC_SMEM_BYTES, st>>>(coef, imgs, qsets, rgb, mcu_prefix, n_images, (uint32_t)n_units, units_x);
        return cudaGetLastError();
    }
    if (bmp)
        hjd_launch_per_image(hjd_k_mcu_rgb<false, true>, hjd_k_mcu_rgb<true, true>, HJD_MCU_THREADS, mcu_prefix, n_images,
                             n_mcus, max_mcus, st, coef, imgs, qsets, rgb);
    else
        hjd_launch_per_image(hjd_k_mcu_rgb<false, false>, hjd_k_mcu_rgb<true, false>, HJD_MCU_THREADS, mcu_prefix, n_images,
                             n_mcus, max_mcus, st, coef, imgs, qsets, rgb);
    return cudaGetLastError();
}

cudaError_t hjd_mcu_tc_init_device(void)
{
    cudaError_t e = cudaFuncSetAttribute(hjd_k_mcu_rgb_tc<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)HJD_TC_SMEM_BYTES);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(hjd_k_mcu_rgb_tc<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)HJD_TC_SMEM_BYTES);
    int dev = 0, sms = 0;
    if (e == cudaSuccess) e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (e == cudaSuccess && dev >= 0 && dev < 64) g_tc_ctas[dev] = sms;
    return e;
}
