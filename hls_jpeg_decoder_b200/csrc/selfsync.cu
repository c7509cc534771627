// csrc/selfsync.cu -- kernel 1b: entropy decode INSIDE a restart-free scan.
//
// The reference decodes one bitstream strictly serially through a single bit reservoir
// (ProcessHuffmanBlock, loadjpg.cpp:497-863, driven block after block by DecodeMCU 945-997).
// Without restart markers nothing in the stream says where a symbol starts, so this path
// speculates and lets Huffman codes' self-synchronisation do the rest:
//
//   0. de-stuff: FF00 -> FF once, in parallel (count / prefix-sum / scatter), so that bit positions
//      are plain offsets and the decoders carry no marker logic;
//   1. every thread decodes from a fixed bit offset one sub-sequence ahead of its own 128-byte
//      sub-sequence (assuming a block starts there), then its own, and records its exit state
//      (bit position, zig-zag index, block-in-MCU);
//   2. sync rounds: a sub-sequence is decoded again from its left neighbour's exit state whenever that
//      state differs from the one it was last decoded from.  A warp owns a range of sub-sequences,
//      collects the ones to redo in shared memory and decodes them 32 at a time until the range is
//      stable; between ranges the states travel through L2 and ONE persistent kernel repeats the round
//      (grid-wide barrier in between) until one passes with nothing to redo -- the host is not in the
//      loop.  Sub-sequence 0 starts from the true state, so by induction the fixed point is exactly
//      the sequential decode;
//   3. an exclusive prefix sum of, per sub-sequence, the number of blocks that start in it and the sums
//      of their DC differences gives every thread its first output block and its DC predictors
//      (DCT[0] = data + prevDC in int16, loadjpg.cpp:664-665);
//   4. the final pass decodes, from the correct entry states, the blocks that start in each
//      sub-sequence and writes every block once, in full, as one 128-byte line.
// Output: the same dense [block][64] zig-zag int16 layout kernel 1a produces.
#include "selfsync.cuh"
#include "device_common.cuh"
#include <cuda_runtime.h>
#include <stdlib.h>

// ------------------------------------------------------------------------------------------
// device-wide exclusive scan (uint32, wrap-around arithmetic)
// ------------------------------------------------------------------------------------------
#define SCAN_THREADS 256
#define SCAN_ITEMS   8
#define SCAN_TILE    (SCAN_THREADS * SCAN_ITEMS)

__device__ __forceinline__ uint32_t block_exclusive_scan(uint32_t v, uint32_t* s_warp, uint32_t* total)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    uint32_t before = 0, sum = 0;
    for (int k = 0; k < (int)(blockDim.x >> 5); k++) {
        const uint32_t c = s_warp[k];
        if (k < warp) before += c;
        sum += c;
    }
    __syncthreads();
    *total = sum;
    return before + incl - v;
}

__global__ void __launch_bounds__(SCAN_THREADS)
hjd_k_scan_tiles(uint32_t* __restrict__ data, uint32_t n, uint32_t* __restrict__ tile_sums)
{
    __shared__ uint32_t s_warp[SCAN_THREADS / 32];
    const uint32_t base = blockIdx.x * SCAN_TILE + threadIdx.x * SCAN_ITEMS;
    uint32_t v[SCAN_ITEMS], sum = 0;
#pragma unroll
    for (int i = 0; i < SCAN_ITEMS; i++) { v[i] = (base + i < n) ? data[base + i] : 0u; sum += v[i]; }
    uint32_t total;
    uint32_t run = block_exclusive_scan(sum, s_warp, &total);
#pragma unroll
    for (int i = 0; i < SCAN_ITEMS; i++) { if (base + i < n) data[base + i] = run; run += v[i]; }
    if (threadIdx.x == 0) tile_sums[blockIdx.x] = total;
}

__global__ void __launch_bounds__(1024)
hjd_k_scan_sums(uint32_t* __restrict__ tile_sums, uint32_t n_tiles)
{
    __shared__ uint32_t s_warp[32];
    __shared__ uint32_t s_carry;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    for (uint32_t base = 0; base < n_tiles; base += 1024) {
        const uint32_t i = base + threadIdx.x;
        const uint32_t v = (i < n_tiles) ? tile_sums[i] : 0u;
        uint32_t total;
        const uint32_t ex = block_exclusive_scan(v, s_warp, &total);
        const uint32_t carry = s_carry;
        if (i < n_tiles) tile_sums[i] = carry + ex;
        __syncthreads();
        if (threadIdx.x == 0) s_carry = carry + total;
        __syncthreads();
    }
}

__global__ void __launch_bounds__(SCAN_THREADS)
hjd_k_scan_add(uint32_t* __restrict__ data, uint32_t n, const uint32_t* __restrict__ tile_sums)
{
    const uint32_t add = tile_sums[blockIdx.x];
    const uint32_t base = blockIdx.x * SCAN_TILE + threadIdx.x * SCAN_ITEMS;
#pragma unroll
    for (int i = 0; i < SCAN_ITEMS; i++)
        if (base + i < n) data[base + i] += add;
}

cudaError_t hjd_scan_u32(uint32_t* data, uint32_t n, uint32_t* tmp, cudaStream_t st)
{
    if (n == 0) return cudaSuccess;
    const uint32_t tiles = (n + SCAN_TILE - 1) / SCAN_TILE;
    hjd_k_scan_tiles<<<tiles, SCAN_THREADS, 0, st>>>(data, n, tmp);
    if (tiles > 1) {
        hjd_k_scan_sums<<<1, 1024, 0, st>>>(tmp, tiles);
        hjd_k_scan_add<<<tiles, SCAN_THREADS, 0, st>>>(data, n, tmp);
    }
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// helpers
// ------------------------------------------------------------------------------------------
// Index of the HjdSsImage whose [chunk_base, chunk_base + n_chunks) range contains the chunk `key`.
__device__ __forceinline__ int ss_find_chunk(const HjdSsImage* __restrict__ ss, int n_ss, uint32_t key)
{
    int lo = 0, hi = n_ss - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (ss[mid].chunk_base <= key) lo = mid; else hi = mid - 1;
    }
    return lo;
}

// ------------------------------------------------------------------------------------------
// step 0: de-stuffing
// ------------------------------------------------------------------------------------------
// A thread owns one 16-byte aligned chunk of the stuffed scan.  A byte is dropped iff it is 00 and
// its predecessor (inside the scan) is FF.  Returns the keep mask (bit j = keep byte j).
// The byte tests are SIMD-within-a-register (exact per byte, no carries between bytes).
__device__ __forceinline__ uint32_t destuff_mask(const uint8_t* a0, uint32_t lc, uint32_t lead, uint32_t scan_len,
                                                 uint4* out_bytes)
{
    const uint4 v = __ldg((const uint4*)(a0 + (size_t)lc * 16));
    *out_bytes = v;
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
    const uint32_t q0 = lc * 16;                       // position of byte 0 relative to a0
    uint32_t ff_prev = (q0 > lead && a0[(size_t)q0 - 1] == 0xFFu) ? 0x80000000u : 0u;   // FF flag of the byte before
    uint32_t keep = 0;
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const uint32_t x = w[k];
        const uint32_t zero = ~(((x & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | x | 0x7F7F7F7Fu);     // 0x80 in bytes equal to 00
        const uint32_t ff = ((x & 0x7F7F7F7Fu) + 0x01010101u) & x & 0x80808080u;          // 0x80 in bytes equal to FF
        const uint32_t after_ff = __funnelshift_l(ff_prev, ff, 8);                        // 0x80 in bytes whose predecessor is FF
        const uint32_t kept = ~(zero & after_ff) & 0x80808080u;
        keep |= ((((kept >> 7) * 0x01020408u) >> 24) & 15u) << (4 * k);                   // gather the four flags
        ff_prev = ff;
    }
    // only the first and the last chunk of a scan hold bytes outside it
    if (q0 < lead || q0 + 16 > lead + scan_len) {
        uint32_t valid = 0;
#pragma unroll
        for (int j = 0; j < 16; j++) {
            const uint32_t q = q0 + j;
            if (q >= lead && q - lead < scan_len) valid |= 1u << j;
        }
        keep &= valid;
        // the first byte of the scan has no predecessor inside it
        if (q0 <= lead && lead < q0 + 16 && scan_len) keep |= 1u << (lead - q0);
    }
    return keep;
}

// Image of the chunk t: one binary search per CTA (for its first chunk), then a short walk, since
// the chunks of a CTA are consecutive and images are long.
__device__ __forceinline__ int destuff_image_of(const HjdSsImage* __restrict__ ss, int n_ss, uint32_t t, int* s_first)
{
    if (threadIdx.x == 0) *s_first = ss_find_chunk(ss, n_ss, t - threadIdx.x);
    __syncthreads();
    int si = *s_first;
    while (si + 1 < n_ss && ss[si + 1].chunk_base <= t) si++;
    return si;
}

__global__ void __launch_bounds__(256)
hjd_k_destuff_count(const uint8_t* __restrict__ arena, const HjdImageDesc* __restrict__ imgs,
                    const HjdSsImage* __restrict__ ss, int n_ss, uint32_t t0, uint32_t n_chunks_total,
                    uint32_t* __restrict__ counts)
{
    // chunks [t0, n_chunks_total) of the batch-wide chunk numbering belong to the ss[] images given here
    __shared__ int s_first;
    const uint32_t t = t0 + blockIdx.x * 256 + threadIdx.x;
    const int si = destuff_image_of(ss, n_ss, t < n_chunks_total ? t : n_chunks_total - 1, &s_first);
    if (t >= n_chunks_total) { if (t == n_chunks_total) counts[t] = 0; return; }
    const HjdSsImage s = ss[si];
    const HjdImageDesc* d = imgs + s.img;
    const uint8_t* a0 = arena + d->scan_off - s.lead;
    uint4 bytes;
    counts[t] = __popc(destuff_mask(a0, t - s.chunk_base, s.lead, d->scan_len, &bytes));
}

// The kept bytes of a warp's 32 chunks form one contiguous output range of at most 512 bytes.  They are
// compacted in shared memory (at the same alignment modulo 4 as their destination) and leave as
// aligned 32-bit words, adjacent lanes adjacent: sixteen one-byte global stores per thread kept this
// kernel at 260 us per 91 MB.  A warp that straddles two images falls back to byte stores.
__global__ void __launch_bounds__(256)
hjd_k_destuff_scatter(const uint8_t* __restrict__ arena, const HjdImageDesc* __restrict__ imgs,
                      const HjdSsImage* __restrict__ ss, int n_ss, uint32_t t0, uint32_t n_chunks_total,
                      const uint32_t* __restrict__ prefix, uint8_t* __restrict__ dst, uint32_t* __restrict__ dlen)
{
    __shared__ int s_first;
    __shared__ __align__(16) uint8_t s_stage[8][544];
    const uint32_t t = t0 + blockIdx.x * 256 + threadIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int si = destuff_image_of(ss, n_ss, t < n_chunks_total ? t : n_chunks_total - 1, &s_first);
    const bool in = t < n_chunks_total;
    uint32_t keep = 0, cnt = 0;
    uint32_t w[4] = {0, 0, 0, 0};
    uint64_t my_out = 0;                                // byte offset of this chunk's output in dst
    HjdSsImage s = ss[si];
    if (in) {
        const HjdImageDesc* d = imgs + s.img;
        const uint8_t* a0 = arena + d->scan_off - s.lead;
        uint4 bytes;
        keep = destuff_mask(a0, t - s.chunk_base, s.lead, d->scan_len, &bytes);
        w[0] = bytes.x; w[1] = bytes.y; w[2] = bytes.z; w[3] = bytes.w;
        cnt = __popc(keep);
        my_out = s.dst_off + (prefix[t] - prefix[s.chunk_base]);
    }
    const uint64_t next_out = __shfl_down_sync(0xffffffffu, my_out, 1);
    const bool chained = in && (lane == 31 || next_out == my_out + cnt);
    if (__all_sync(0xffffffffu, chained)) {
        const uint64_t base = __shfl_sync(0xffffffffu, my_out, 0);
        const uint32_t total = (uint32_t)(__shfl_sync(0xffffffffu, my_out + cnt, 31) - base);
        const uint32_t al = (uint32_t)base & 3u;          // dst is 256-byte aligned: offset alignment == address alignment
        uint8_t* st = s_stage[warp];
        uint32_t o = (uint32_t)(my_out - base) + al;
#pragma unroll
        for (int j = 0; j < 16; j++)
            if (keep & (1u << j)) st[o++] = (uint8_t)(w[j >> 2] >> (8 * (j & 3)));
        __syncwarp();
        const uint32_t end = al + total;                 // staged bytes are [al, end)
        const uint32_t first_full = al ? 4u : 0u;
        uint8_t* g = dst + (base - al);                   // 4-byte aligned
        if (end <= first_full) {
            if ((uint32_t)lane >= al && (uint32_t)lane < end) g[lane] = st[lane];
        } else {
            const uint32_t end_full = end & ~3u;
            for (uint32_t i = first_full / 4 + lane; i < end_full / 4; i += 32) ((uint32_t*)g)[i] = ((const uint32_t*)st)[i];
            if ((uint32_t)lane >= al && (uint32_t)lane < first_full) g[lane] = st[lane];                 // head bytes
            if (end_full + lane < end) g[end_full + lane] = st[end_full + lane];                         // tail bytes
        }
    } else if (in) {
        uint8_t* out = dst + my_out;
#pragma unroll
        for (int j = 0; j < 16; j++)
            if (keep & (1u << j)) *out++ = (uint8_t)(w[j >> 2] >> (8 * (j & 3)));
    }
    if (in && t == s.chunk_base + s.n_chunks - 1) {    // last chunk of the image: length + zero slack
        const uint32_t len = prefix[t] - prefix[s.chunk_base] + cnt;
        dlen[si] = len;
        uint4* z = (uint4*)(dst + s.dst_off + ((len + 15u) & ~15u));
        for (uint32_t j = len; j < ((len + 15u) & ~15u); j++) dst[s.dst_off + j] = 0;
        for (int j = 0; j < HJD_SS_SLACK / 16; j++) z[j] = make_uint4(0, 0, 0, 0);
    }
}

cudaError_t hjd_launch_destuff(const uint8_t* arena, const HjdImageDesc* imgs, const HjdSsImage* ss, int n_ss,
                               uint32_t first_chunk, uint32_t n_chunks, uint32_t* counts, uint32_t* scan_tmp,
                               uint8_t* dst, uint32_t* dlen, cudaStream_t st)
{
    if (n_ss <= 0 || n_chunks == 0) return cudaSuccess;
    const uint32_t grid = (n_chunks + 1 + 255) / 256;
    const uint32_t end = first_chunk + n_chunks;
    hjd_k_destuff_count<<<grid, 256, 0, st>>>(arena, imgs, ss, n_ss, first_chunk, end, counts);
    cudaError_t e = hjd_scan_u32(counts + first_chunk, n_chunks + 1, scan_tmp, st);
    if (e != cudaSuccess) return e;
    hjd_k_destuff_scatter<<<grid, 256, 0, st>>>(arena, imgs, ss, n_ss, first_chunk, end, counts, dst, dlen);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// the sub-sequence decoder of the synchronisation rounds
// ------------------------------------------------------------------------------------------
// state = bit position (40 bits) | zig-zag index (7 bits) << 40 | block-in-MCU index (4 bits) << 47
#define SS_INVALID 0xFFFFFFFFFFFFFFFFull
__device__ __forceinline__ uint64_t ss_pack(uint64_t p, int k, int c) { return p | ((uint64_t)k << 40) | ((uint64_t)c << 47); }

struct SsCtx {
    const uint8_t* D;       // de-stuffed stream (zero slack after its end)
    uint32_t sh_tab;        // shared-window address of the component tables (DC, AC per component)
    uint32_t bpm, ny;
};

// What a sub-sequence contributes to the output layout: blocks that START inside it (a block belongs
// to the sub-sequence in which its DC symbol begins) and the sums of their DC differences per component.
struct SsCount { uint32_t ns, dc0, dc1, dc2; };

// Bit reader over the de-stuffed stream: a 64-bit window (hi:lo, MSB first, zero beyond nbits) fed by
// aligned big-endian words that are loaded two refills ahead, so that the load latency stays off the
// serial symbol-to-symbol dependence (what the synchronisation rounds, with few warps, are bound by).
struct SsBits {
    uint32_t hi, lo;
    int nbits;
#ifndef HJD_SS_PREFETCH
#define HJD_SS_PREFETCH 2       // words in flight ahead of the window (3 measured slower: 2.95 vs 2.89 ms per 256 restart-free 1080p images)
#endif
    uint32_t wa, wb, wc;        // the next words (wc unused when HJD_SS_PREFETCH == 2)
    const uint32_t* wp;         // the word after them
    __device__ __forceinline__ void init(const uint8_t* D, uint64_t p)
    {
        const uint32_t* w = (const uint32_t*)D + (p >> 5);           // D is 256-byte aligned
        hi = __byte_perm(__ldg(w), 0, 0x0123);
        lo = __byte_perm(__ldg(w + 1), 0, 0x0123);
        wa = __byte_perm(__ldg(w + 2), 0, 0x0123);
        wb = __byte_perm(__ldg(w + 3), 0, 0x0123);
#if HJD_SS_PREFETCH == 3
        wc = __byte_perm(__ldg(w + 4), 0, 0x0123);
        wp = w + 5;
#else
        wc = 0;
        wp = w + 4;
#endif
        const uint32_t sh = (uint32_t)p & 31u;
        hi = __funnelshift_l(lo, hi, sh);
        lo <<= sh;
        nbits = 64 - (int)sh;
    }
    // at least 32 valid bits afterwards (a symbol takes at most 16 + 15)
    __device__ __forceinline__ void ensure()
    {
        if (nbits < 32) {                                            // lo holds no valid bit here
            hi |= wa >> nbits;
            lo = hjd_shl(wa, 32u - (uint32_t)nbits);
            nbits += 32;
            wa = wb;
#if HJD_SS_PREFETCH == 3
            wb = wc;
            wc = __byte_perm(__ldg(wp++), 0, 0x0123);
#else
            wb = __byte_perm(__ldg(wp++), 0, 0x0123);
#endif
        }
    }
    __device__ __forceinline__ void skip(uint32_t n)                 // n <= 31
    {
        hi = __funnelshift_l(lo, hi, n);
        lo <<= n;
        nbits -= (int)n;
    }
};

// One Huffman symbol from the window (hi:lo): the fields of hjd_sym_fields plus the extended value.
// An undecodable code consumes one bit and ends the block (HJD_BAD_ENTRY) so that every path makes progress;
// the synchronisation rounds and the write pass must agree on this rule, which is why they share this code.
struct SsSym { uint32_t used, size, kadv; int val; };

__device__ __forceinline__ SsSym ss_symbol(uint32_t t, uint32_t hi, uint32_t lo, bool is_ac)
{
    SsSym s;
    const uint32_t e = hjd_lookup(t, hi);
    const uint32_t len = e & 31u;
    s.size = (e >> 5) & 15u;
    s.kadv = (e >> 9) & 127u;
    const uint32_t after = __funnelshift_l(lo, hi, len);
    const uint32_t v = hjd_shr(after, 32u - s.size);
    const int neg = ~((int)after >> 31);
    s.val = (int)v + (neg & (int)(hjd_shl(0xFFFFFFFFu, s.size) + 1u));       // DetermineSign, loadjpg.cpp:396-409
    s.used = len + s.size;
    return s;
}

// Decode symbols from `state` until the bit position reaches end_bit; returns the exit state.
// COUNT: also count the blocks that start in [entry, end_bit) and sum their DC differences.
template <bool COUNT>
__device__ __forceinline__ uint64_t ss_scan_decode(const SsCtx& cx, uint64_t state, uint64_t end_bit, SsCount* cnt)
{
    constexpr uint32_t kTabBytes = (uint32_t)sizeof(HjdHuffTable);
    const uint64_t p0 = state & 0xFFFFFFFFFFull;
    int k = (int)((state >> 40) & 127u), c = (int)((state >> 47) & 15u);
    SsBits br;
    br.init(cx.D, p0);
    int rem = (int)(end_bit - p0);                       // bits left in the sub-sequence (entry is at most one behind)
    // The block-end bookkeeping is straight-line code: nearly every iteration of a warp has some lane
    // at a block end, so a branch here costs more than always executing the selects (it was a quarter
    // of the kernel's instructions).  DC sums rotate with the component, slot 0 = current component.
    uint32_t comp = (uint32_t)c < cx.ny ? 0u : (uint32_t)c - cx.ny + 1u;
    uint32_t t0 = cx.sh_tab + comp * 2u * kTabBytes;
    uint32_t ns = 0, d0 = 0, d1 = 0, d2 = 0;

    while (rem > 0) {
        br.ensure();
        const bool is_ac = k != 0;
        const SsSym s = ss_symbol(t0 + (is_ac ? kTabBytes : 0u), br.hi, br.lo, is_ac);
        br.skip(s.used);
        rem -= (int)s.used;
        if (COUNT) {
            ns += is_ac ? 0u : 1u;
            d0 += is_ac ? 0u : (uint32_t)s.val;
        }
        k += (int)s.kadv;
        const bool blk_end = k >= 64;
        k = blk_end ? 0 : k;
        int c1 = c + 1;
        c1 = (uint32_t)c1 == cx.bpm ? 0 : c1;
        c = blk_end ? c1 : c;
        const uint32_t comp_new = (uint32_t)c < cx.ny ? 0u : (uint32_t)c - cx.ny + 1u;
        if (COUNT) {
            const bool chg = comp_new != comp;           // Y -> Cb -> Cr -> Y: always to the next slot
            const uint32_t r0 = chg ? d1 : d0, r1 = chg ? d2 : d1, r2 = chg ? d0 : d2;
            d0 = r0; d1 = r1; d2 = r2;
        }
        comp = comp_new;
        t0 = cx.sh_tab + comp * 2u * kTabBytes;
    }
    if (COUNT) {
        // back to (Y, Cb, Cr): slot 0 holds the component of block c
        cnt->ns = ns;
        cnt->dc0 = comp == 0u ? d0 : (comp == 1u ? d2 : d1);
        cnt->dc1 = comp == 0u ? d1 : (comp == 1u ? d0 : d2);
        cnt->dc2 = comp == 0u ? d2 : (comp == 1u ? d1 : d0);
    }
    return ss_pack(end_bit - (uint64_t)(int64_t)rem, k, c);
}

// Loads the three per-component (DC, AC) table pairs of a table set into shared memory.
__device__ __forceinline__ void ss_load_tables(const HjdTableSet* ts, uint8_t* s_tab)
{
    constexpr int n16 = (int)(sizeof(HjdHuffTable) / 16);
    for (int c = 0; c < 3; c++) {
        const uint4* sdc = (const uint4*)&ts->tab[ts->dc_of_comp[c]];
        const uint4* sac = (const uint4*)&ts->tab[ts->ac_of_comp[c]];
        uint4* ddc = (uint4*)(s_tab + (2 * c) * sizeof(HjdHuffTable));
        uint4* dac = (uint4*)(s_tab + (2 * c + 1) * sizeof(HjdHuffTable));
        for (int i = threadIdx.x; i < n16; i += blockDim.x) { ddc[i] = __ldg(sdc + i); dac[i] = __ldg(sac + i); }
    }
}

// Which sub-sequence a thread of a speculative / write CTA owns: binary search over the CTA's segments
// (tid0 ascending).  A thread beyond the CTA's sub-sequences gets li = 0xFFFFFFFF (owns nothing).
__device__ __forceinline__ void ss_locate(const HjdSsWork& wk, const HjdSsSeg* __restrict__ segs, uint32_t tid,
                                          uint32_t* ssi, uint32_t* li)
{
    uint32_t lo = 0, hi = wk.n_segs - 1;
    while (lo < hi) {
        const uint32_t mid = (lo + hi + 1) >> 1;
        if (segs[wk.first_seg + mid].tid0 <= tid) lo = mid; else hi = mid - 1;
    }
    const HjdSsSeg sg = segs[wk.first_seg + lo];
    *ssi = sg.ss;
    *li = tid < wk.n_subs ? sg.first_sub + (tid - sg.tid0) : 0xFFFFFFFFu;
}

// ------------------------------------------------------------------------------------------
// step 1: speculative decode
// ------------------------------------------------------------------------------------------
// Every thread decodes the sub-sequence BEFORE its own from the fixed bit offset (assuming a block
// starts there) and takes the state it arrives in as the entry state of its own sub-sequence, which
// it then decodes and counts.  About three quarters of the entry states are already right after
// 1024 bits of lead-in (measured on 1080p 4:2:0: 23 % wrong, then 6 %, 1.5 %, ... per further
// sub-sequence; the block-in-MCU index is what takes long to lock).  Sub-sequence 0 starts from the
// true state.
__global__ void __launch_bounds__(HJD_SS_THREADS)
hjd_k_ss_spec(const HjdImageDesc* __restrict__ imgs, const HjdTableSet* __restrict__ tsets,
              const HjdSsImage* __restrict__ ss, const HjdSsWork* __restrict__ work,
              const HjdSsSeg* __restrict__ segs,
              const uint8_t* __restrict__ dst, const uint32_t* __restrict__ dlen, uint32_t n_subs_total,
              uint64_t* __restrict__ e_arr, uint64_t* __restrict__ x_arr, uint32_t* __restrict__ cnt_arr)
{
    extern __shared__ __align__(16) uint8_t s_tab[];
    const HjdSsWork wk = work[blockIdx.x];
    ss_load_tables(tsets + wk.table_set, s_tab);
    __syncthreads();

    uint32_t ssi, li;                                                // image, local sub-sequence index
    ss_locate(wk, segs, threadIdx.x, &ssi, &li);
    const HjdSsImage s = ss[ssi];
    const HjdImageDesc* d = imgs + s.img;
    if (li >= s.n_subs) return;
    const uint32_t L = dlen[ssi];
    const uint32_t gi = s.sub_base + li;
    SsCount cnt = {0, 0, 0, 0};
    uint64_t e = 0, x = SS_INVALID;
    if ((uint64_t)li * HJD_SS_SUB_BYTES < L) {
        SsCtx cx;
        cx.D = dst + s.dst_off;
        cx.sh_tab = (uint32_t)__cvta_generic_to_shared(s_tab);
        cx.bpm = d->blocks_per_mcu;
        cx.ny = d->ncomp == 3 ? (uint32_t)d->hf * d->vf : 1u;
        const uint64_t sub_bits = (uint64_t)HJD_SS_SUB_BYTES * 8;
        x = ss_pack(0, 0, 0);
        if (li != 0) x = ss_scan_decode<false>(cx, ss_pack((uint64_t)(li - 1) * sub_bits, 0, 0), (uint64_t)li * sub_bits, nullptr);
        e = ss_scan_decode<true>(cx, x, (uint64_t)(li + 1) * sub_bits, &cnt);
    }
    e_arr[gi] = e;
    x_arr[gi] = x;
    cnt_arr[gi] = cnt.ns;
    cnt_arr[n_subs_total + gi] = cnt.dc0;
    cnt_arr[2 * n_subs_total + gi] = cnt.dc1;
    cnt_arr[3 * n_subs_total + gi] = cnt.dc2;
}

cudaError_t hjd_launch_ss_spec(const HjdImageDesc* imgs, const HjdTableSet* tsets, const HjdSsImage* ss,
                               const HjdSsWork* work, const HjdSsSeg* segs, int n_work, const uint8_t* dst,
                               const uint32_t* dlen,
                               uint32_t n_subs_total, uint64_t* e, uint64_t* x, uint32_t* cnt, cudaStream_t st)
{
    if (n_work <= 0) return cudaSuccess;
    hjd_k_ss_spec<<<n_work, HJD_SS_THREADS, 6 * sizeof(HjdHuffTable), st>>>(imgs, tsets, ss, work, segs, dst, dlen,
                                                                           n_subs_total, e, x, cnt);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// step 2: synchronisation rounds
// ------------------------------------------------------------------------------------------
// One WARP owns `range` consecutive sub-sequences of one image (a work item = HJD_SS_FIX_WARPS such
// ranges sharing a table set).  A sub-sequence whose left neighbour's exit state differs from the
// entry state it was decoded from goes on the warp's list in shared memory; the list is decoded 32
// entries at a time, so the few sub-sequences still wrong cost a few dense warp passes instead of one
// mostly idle pass per 32 sub-sequences; repeat until the range is consistent.  The states before the
// range come from L2, where the previous warp may still be correcting them: whichever values the
// reads return, the rounds go on until one passes in which no warp had anything to decode.
// Sub-sequence 0 starts from the true state, so the fixed point is the sequential decode.
//
// The rounds run inside ONE persistent kernel (cooperative launch: every CTA is resident), the CTAs
// striding over the work items, with a grid-wide barrier between rounds; the round in which some warp
// last had anything to decode is kept in ctl[1], and everybody leaves after the first round that did
// not raise it.  (The first version launched one kernel per round and had the host read a flag after
// each: a stream synchronisation per round, in the middle of the hot path.)
// ctl[0] barrier arrivals, ctl[1] last round (1-based) with work, ctl[2] rounds executed (bit 31: the
// round limit was hit, which the induction argument above rules out), ctl[3] work-item counter; all zero at launch.
__device__ __forceinline__ uint64_t ss_ld64(const uint64_t* p) { return __ldcg((const unsigned long long*)p); }
__device__ __forceinline__ void ss_st64(uint64_t* p, uint64_t v) { __stcg((unsigned long long*)p, (unsigned long long)v); }

__global__ void __launch_bounds__(HJD_SS_FIX_WARPS * 32)
hjd_k_ss_sync(const HjdImageDesc* __restrict__ imgs, const HjdTableSet* __restrict__ tsets,
              const HjdSsImage* __restrict__ ss, const HjdSsWork* __restrict__ work,
              const HjdSsSeg* __restrict__ segs, int n_work,
              const uint8_t* __restrict__ dst, const uint32_t* __restrict__ dlen, uint32_t n_subs_total,
              uint64_t* e_arr, uint64_t* x_arr, uint32_t* __restrict__ cnt_arr,
              uint32_t* ctl, uint32_t max_rounds)
{
    extern __shared__ __align__(16) uint8_t s_raw[];
    constexpr uint32_t kEntries = HJD_SS_FIX_MAXR + HJD_SS_FIX_OVERLAP;
    constexpr uint32_t kWarpBytes = (kEntries * 18 + 15) & ~15u;
    uint8_t* s_tab = s_raw + HJD_SS_FIX_WARPS * kWarpBytes;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint64_t* sE = (uint64_t*)(s_raw + warp * kWarpBytes);           // exit state per sub-sequence of the window
    uint64_t* sX = sE + kEntries;                                    // entry state it was computed from
    uint16_t* sL = (uint16_t*)(sX + kEntries);                       // sub-sequences to decode again
    const uint64_t sub_bits = (uint64_t)HJD_SS_SUB_BYTES * 8;
    const uint32_t lt_mask = (1u << lane) - 1u;
    uint32_t loaded_set = 0xFFFFFFFFu;                               // table set in s_tab (CTA-uniform)

    __shared__ int s_wi;
    for (uint32_t round = 1;; round++) {
        // Work items are handed out through one counter (ctl[3]) that is never reset: in every round each CTA
        // draws items until its draw is past the end, so a round advances the counter by n_work + gridDim.x
        // exactly.  (Static striding left the CTAs that happened to own the ranges with many wrong entry
        // states working long after the others: the first round is where nearly all the time goes.)
        const uint32_t round_base = (round - 1u) * ((uint32_t)n_work + gridDim.x);
        for (;;) {
            __syncthreads();                                         // s_wi, s_tab and the windows are free
            if (threadIdx.x == 0) s_wi = (int)(atomicAdd(&ctl[3], 1u) - round_base);
            __syncthreads();
            const int wi = s_wi;
            if (wi >= n_work) break;
            const HjdSsWork wk = work[wi];
            const bool has_range = (uint32_t)warp < wk.n_segs;       // this warp's range (possibly of another image than its neighbours')
            const HjdSsSeg sg = segs[wk.first_seg + (has_range ? warp : 0)];
            const HjdSsImage s = ss[sg.ss];
            const HjdImageDesc* d = imgs + s.img;

            const uint32_t L = dlen[sg.ss];
            const uint32_t first = sg.first_sub;                     // local index of the range's first sub-sequence
            uint32_t n_have = (L + HJD_SS_SUB_BYTES - 1) / HJD_SS_SUB_BYTES;   // sub-sequences that hold data
            if (n_have > s.n_subs) n_have = s.n_subs;
            const int n_own = has_range && first < n_have ? (int)min(sg.n, n_have - first) : 0;
            // The window starts HJD_SS_FIX_OVERLAP sub-sequences before the range: they are re-checked (and, if
            // need be, re-decoded) privately, never written back -- they belong to the previous warp, which
            // may be correcting them at this very moment.  So the entry state of the range does not hinge on
            // one exit state of the speculative pass, and the round after this one is normally a pure check.
            const uint32_t lo = first >= HJD_SS_FIX_OVERLAP ? first - HJD_SS_FIX_OVERLAP : 0u;
            const int kov = n_own ? (int)(first - lo) : 0;
            const int n_act = n_own ? kov + n_own : 0;
            const uint32_t g0 = s.sub_base + lo;
            for (int j = lane; j < n_act; j += 32) { sE[j] = ss_ld64(e_arr + g0 + j); sX[j] = ss_ld64(x_arr + g0 + j); }
            uint64_t boundary = ss_pack(0, 0, 0);
            if (n_act && lo != 0) boundary = ss_ld64(e_arr + g0 - 1);
            __syncwarp();
            bool any = false;
            for (int j = lane; j < n_act; j += 32) any |= (j == 0 ? boundary : sE[j - 1]) != sX[j];
            // A warp that has anything to decode again marks the round.  The rounds stop after one in which
            // no warp did: every warp then found its window -- read while nobody was writing --
            // consistent, including the entry of its range against the previous range's last exit state.
            if (__any_sync(0xffffffffu, any) && lane == 0) atomicMax(&ctl[1], round);
            if (!__syncthreads_or(any)) continue;                    // the usual case in the later rounds (CTA-uniform)
            if (loaded_set != wk.table_set) {
                ss_load_tables(tsets + wk.table_set, s_tab);
                loaded_set = wk.table_set;
            }
            __syncthreads();

            SsCtx cx;
            cx.D = dst + s.dst_off;
            cx.sh_tab = (uint32_t)__cvta_generic_to_shared(s_tab);
            cx.bpm = d->blocks_per_mcu;
            cx.ny = d->ncomp == 3 ? (uint32_t)d->hf * d->vf : 1u;
            for (int iter = 0; iter < n_act + 2; iter++) {
                int n = 0;
                for (int j0 = 0; j0 < n_act; j0 += 32) {
                    const int j = j0 + lane;
                    const bool need = j < n_act && (j == 0 ? boundary : sE[j - 1]) != sX[j];
                    const uint32_t bal = __ballot_sync(0xffffffffu, need);
                    if (need) sL[n + __popc(bal & lt_mask)] = (uint16_t)j;
                    n += __popc(bal);
                }
                __syncwarp();
                if (n == 0) break;
                for (int q0 = 0; q0 < n; q0 += 32) {
                    int t = -1;
                    uint64_t txin = 0;
                    if (q0 + lane < n) {
                        t = sL[q0 + lane];
                        txin = t == 0 ? boundary : sE[t - 1];
                    }
                    __syncwarp();                                    // entry states read before any is rewritten
                    if (t >= 0) {
                        SsCount cnt;
                        const uint64_t te = ss_scan_decode<true>(cx, txin, (uint64_t)(lo + t + 1) * sub_bits, &cnt);
                        if (t >= kov) {
                            const uint32_t g = g0 + (uint32_t)t;
                            cnt_arr[g] = cnt.ns;
                            cnt_arr[n_subs_total + g] = cnt.dc0;
                            cnt_arr[2 * n_subs_total + g] = cnt.dc1;
                            cnt_arr[3 * n_subs_total + g] = cnt.dc2;
                        }
                        sE[t] = te;
                        sX[t] = txin;
                    }
                    __syncwarp();
                }
            }
            for (int j = kov + lane; j < n_act; j += 32) { ss_st64(e_arr + g0 + j, sE[j]); ss_st64(x_arr + g0 + j, sX[j]); }
        }
        // ---- grid-wide barrier, then: did anybody have work in this round? ---------------------
        __syncthreads();
        if (threadIdx.x == 0) {
            __threadfence();
            atomicAdd(&ctl[0], 1u);
            const uint32_t want = round * gridDim.x;
            while (*(volatile uint32_t*)&ctl[0] < want) __nanosleep(64);
            __threadfence();
        }
        __syncthreads();
        const uint32_t last = *(volatile uint32_t*)&ctl[1];
        if (last < round || round >= max_rounds) {
            if (blockIdx.x == 0 && threadIdx.x == 0) ctl[2] = round | (last < round ? 0u : 0x80000000u);
            break;
        }
    }
}

static size_t ss_sync_smem(void)
{
    return (size_t)HJD_SS_FIX_WARPS * (((HJD_SS_FIX_MAXR + HJD_SS_FIX_OVERLAP) * 18 + 15) & ~15u) + 6 * sizeof(HjdHuffTable);
}

cudaError_t hjd_launch_ss_sync(const HjdImageDesc* imgs, const HjdTableSet* tsets, const HjdSsImage* ss,
                               const HjdSsWork* work, const HjdSsSeg* segs, int n_work, const uint8_t* dst,
                               const uint32_t* dlen,
                               uint32_t n_subs_total, uint64_t* e, uint64_t* x, uint32_t* cnt,
                               uint32_t* ctl, uint32_t max_rounds, int max_resident_ctas, cudaStream_t st)
{
    if (n_work <= 0) return cudaSuccess;
    int grid = n_work < max_resident_ctas ? n_work : max_resident_ctas;
    if (grid < 1) grid = 1;
    void* args[] = {(void*)&imgs, (void*)&tsets, (void*)&ss, (void*)&work, (void*)&segs, (void*)&n_work, (void*)&dst,
                    (void*)&dlen, (void*)&n_subs_total, (void*)&e, (void*)&x, (void*)&cnt, (void*)&ctl, (void*)&max_rounds};
    return cudaLaunchCooperativeKernel((const void*)hjd_k_ss_sync, dim3((unsigned)grid), dim3(HJD_SS_FIX_WARPS * 32), args,
                                       ss_sync_smem(), st);
}

// ------------------------------------------------------------------------------------------
// step 4: final pass with output
// ------------------------------------------------------------------------------------------
// Every thread decodes the blocks that START in its sub-sequence, each to its end (running into the
// next sub-sequence if need be), after skipping the tail of the block it was entered in the middle of
// (that block belongs to an earlier thread).  So every 8x8 block is produced by exactly one thread, in
// full, and leaves the SM as one 128-byte line through the same slot / list / four-at-a-time flush as
// kernel 1a; the coefficient slab needs no zero-fill.  prefix[] = exclusive scan of the counts of the
// last round: first owned block and, per component, the DC predictor at it
// (DCT[0] = data + prevDC in int16, loadjpg.cpp:664-665).
#define SS_WRITE_SYMS 4
// Bounds of an owned block (a crafted table whose AC symbols never advance the zig-zag index would
// otherwise keep its owner decoding forever, past the stream, the slack and the buffer): at most
// SS_WRITE_MAX_STEPS rounds of SS_WRITE_SYMS symbols per block -- 16 times what a block of 64
// coefficients can need -- and no bit position beyond the zeroed slack.  A thread that hits either
// flags the image and zero-fills the blocks it still owed.
#define SS_WRITE_MAX_STEPS 256

__global__ void __launch_bounds__(HJD_SS_THREADS)
hjd_k_ss_write(const HjdImageDesc* __restrict__ imgs, const HjdTableSet* __restrict__ tsets,
               const HjdSsImage* __restrict__ ss, const HjdSsWork* __restrict__ work,
               const HjdSsSeg* __restrict__ segs,
               const uint8_t* __restrict__ dst, const uint32_t* __restrict__ dlen, uint32_t n_subs_total,
               const uint64_t* __restrict__ x_arr, const uint32_t* __restrict__ prefix,
               int16_t* __restrict__ coef, int32_t* __restrict__ status)
{
    extern __shared__ __align__(16) uint8_t s_raw[];
    constexpr uint32_t kTabBytes = (uint32_t)sizeof(HjdHuffTable);
    constexpr uint32_t kSlotBytes = HJD_SS_THREADS * 128, kListBytes = HJD_SS_THREADS * 8;
    uint8_t* s_tab = s_raw + kSlotBytes + kListBytes;
    const HjdSsWork wk = work[blockIdx.x];
    ss_load_tables(tsets + wk.table_set, s_tab);
    {
        uint4* z = (uint4*)s_raw;
        for (int i = threadIdx.x; i < HJD_SS_THREADS * 8; i += HJD_SS_THREADS) z[i] = make_uint4(0, 0, 0, 0);
    }
    __syncthreads();

    const int tid = threadIdx.x, lane = tid & 31;
    const uint32_t sh_base = (uint32_t)__cvta_generic_to_shared(s_raw);
    const uint32_t sh_list = sh_base + kSlotBytes;
    const uint32_t sh_tab = sh_list + kListBytes;
    const uint32_t my_slot = sh_base + (uint32_t)tid * 128u;
    const uint32_t swz = (uint32_t)(lane & 7) << 4;
    const uint32_t warp_slots = sh_base + (uint32_t)(tid & ~31) * 128u;
    const uint32_t warp_list = sh_list + (uint32_t)(tid & ~31) * 8u;
    const uint32_t lt_mask = (1u << lane) - 1u;

    uint32_t ssi, li;                 // image, local sub-sequence index (0xFFFFFFFF: none)
    ss_locate(wk, segs, (uint32_t)tid, &ssi, &li);
    const HjdSsImage s = ss[ssi];
    const HjdImageDesc* d = imgs + s.img;
    const uint32_t L = dlen[ssi];
    const uint32_t bpm = d->blocks_per_mcu, ny = d->ncomp == 3 ? (uint32_t)d->hf * d->vf : 1u;
    const uint32_t n_blocks = (uint32_t)d->n_blocks;
    const uint32_t blk_base = (uint32_t)d->block_base;
    const uint8_t* D = dst + s.dst_off;
    const uint64_t end_bit = (uint64_t)(li + 1) * HJD_SS_SUB_BYTES * 8;

    bool finished = true;
    bool owned = false;               // false while skipping the tail of a block entered in the middle
    int rem = 0;                      // bits left in the sub-sequence (<= 0: past its end)
    int k = 0, c = 0;
    uint32_t blk = 0;                 // image-local index of the block being decoded (when owned)
    int p0 = 0, p1 = 0, p2 = 0;       // DC predictors, p0 = current component
    uint32_t t0 = sh_tab, t1 = sh_tab + 2 * kTabBytes, t2 = sh_tab + 4 * kTabBytes;
    SsBits br;
    br.hi = br.lo = br.wa = br.wb = br.wc = 0; br.nbits = 64; br.wp = (const uint32_t*)D;
    int flags = 0;
    int steps = 0;                    // rounds spent on the current owned block
    int rem_min = 0;                  // rem below this: the bit position has left the zeroed slack
    uint32_t own_end = 0;             // image-local index one past the last block this thread owns
    if (li < s.n_subs && (uint64_t)li * HJD_SS_SUB_BYTES < L) {
        const uint32_t gi = s.sub_base + li;
        const uint64_t xs = x_arr[gi];
        {
            const long long lim = ((long long)L + HJD_SS_SLACK - 64) * 8 - (long long)end_bit;   // bits past my sub-sequence that exist
            rem_min = lim > (1ll << 30) ? -(1 << 30) : -(int)(lim < 0 ? 0 : lim);
            own_end = min(prefix[gi + 1] - prefix[s.sub_base], n_blocks);
        }
        if (xs == SS_INVALID) flags |= HJD_ST_BAD_CODE;
        else {
            const uint64_t p = xs & 0xFFFFFFFFFFull;
            rem = (int)(end_bit - p);
            k = (int)((xs >> 40) & 127u);
            c = (int)((xs >> 47) & 15u);
            blk = prefix[gi] - prefix[s.sub_base];
            const int dY = (int)(short)(prefix[n_subs_total + gi] - prefix[n_subs_total + s.sub_base]);
            const int dB = (int)(short)(prefix[2 * n_subs_total + gi] - prefix[2 * n_subs_total + s.sub_base]);
            const int dR = (int)(short)(prefix[3 * n_subs_total + gi] - prefix[3 * n_subs_total + s.sub_base]);
            const uint32_t comp = (uint32_t)c < ny ? 0u : ((uint32_t)c == ny ? 1u : 2u);
            // rotate so that (p0, t0) belong to the component of block c
            if (comp == 0) { p0 = dY; p1 = dB; p2 = dR; }
            else if (comp == 1) { p0 = dB; p1 = dR; p2 = dY; t0 = sh_tab + 2 * kTabBytes; t1 = sh_tab + 4 * kTabBytes; t2 = sh_tab; }
            else { p0 = dR; p1 = dY; p2 = dB; t0 = sh_tab + 4 * kTabBytes; t1 = sh_tab; t2 = sh_tab + 2 * kTabBytes; }
            owned = (k == 0);
            finished = (rem <= 0) || (owned && blk >= n_blocks);
            br.init(D, p);
        }
    }
    const bool last_sub = (li + 1 == s.n_subs) || ((uint64_t)(li + 1) * HJD_SS_SUB_BYTES >= L);

    while (__any_sync(0xffffffffu, !finished)) {
        bool done_block = false;
        if (!finished) {
#pragma unroll
            for (int rep = 0; rep < SS_WRITE_SYMS; rep++) {
                if (!done_block && !finished) {
                    br.ensure();
                    const bool is_ac = k != 0;
                    const SsSym sy = ss_symbol(t0 + (is_ac ? kTabBytes : 0u), br.hi, br.lo, is_ac);
                    br.skip(sy.used);
                    rem -= (int)sy.used;
                    const uint32_t kpos = (uint32_t)k + sy.kadv - 1u;
                    if (owned && sy.size) {
                        if (kpos <= 63u) hjd_sts_u16_sync(my_slot + ((kpos << 1) ^ swz), (uint32_t)sy.val);
                        else flags |= HJD_ST_COEF_RANGE;
                    }
                    k += (int)sy.kadv;
                    if (k >= 64) {
                        // k >= 127: HJD_BAD_ENTRY, no such code.  Flagged only inside an owned (real) block: what a
                        // thread skips may be the padding after the last block, decoded as if a block followed,
                        // and every real block has an owner who sees all of it
                        if (k >= 127 && owned) flags |= HJD_ST_BAD_CODE;
                        if (owned) done_block = true;             // hand-over below
                        else {                                    // the foreign block is over: the next one is mine
                            owned = true;
                            k = 0;
                            if ((uint32_t)++c == bpm) c = 0;
                            if (bpm > 1 && (c == 0 || (uint32_t)c >= ny)) {
                                const int tp = p0; p0 = p1; p1 = p2; p2 = tp;
                                const uint32_t tt = t0; t0 = t1; t1 = t2; t2 = tt;
                            }
                            if (rem <= 0 || blk >= n_blocks) finished = true;
                        }
                    } else if (!owned && rem <= 0) {
                        finished = true;                          // one block covers this whole sub-sequence
                    }
                }
            }
        }
        // ---- bounds (see SS_WRITE_MAX_STEPS) ---------------------------------------------------
        if (!finished && !done_block && owned && (++steps > SS_WRITE_MAX_STEPS || rem < rem_min)) {
            flags |= steps > SS_WRITE_MAX_STEPS ? HJD_ST_BAD_CODE : HJD_ST_OVERRUN;
            for (uint32_t bz = blk; bz < own_end; bz++)
                for (int q = 0; q < 8; q++) ((uint4*)coef)[(size_t)(blk_base + bz) * 8u + q] = make_uint4(0, 0, 0, 0);
            blk = own_end;
            finished = true;
        }
        // ---- block hand-over ---------------------------------------------------------------
        uint32_t flush_blk = 0;
        if (done_block) {
            steps = 0;
            p0 = (int)(short)(p0 + (int)(short)hjd_lds_u16_sync(my_slot + swz));
            hjd_sts_u16_sync(my_slot + swz, (uint32_t)p0);
            flush_blk = blk_base + blk;
            blk++;
            k = 0;
            if ((uint32_t)++c == bpm) c = 0;
            if (bpm > 1 && (c == 0 || (uint32_t)c >= ny)) {
                const int tp = p0; p0 = p1; p1 = p2; p2 = tp;
                const uint32_t tt = t0; t0 = t1; t1 = t2; t2 = tt;
            }
            if (rem <= 0 || blk >= n_blocks) finished = true;
        }
        // ---- cooperative flush, four blocks per step (as in kernel 1a) ----------------------
        const uint32_t m = __ballot_sync(0xffffffffu, done_block);
        if (m) {
            if (done_block) hjd_sts_v2_sync(warp_list + (uint32_t)__popc(m & lt_mask) * 8u, flush_blk, (uint32_t)lane);
            __syncwarp();
            const int n_done = __popc(m);
            const uint32_t chunk = (uint32_t)lane & 7u;
            for (int base = 0; base < n_done; base += 4) {
                const int idx = base + (lane >> 3);
                if (idx < n_done) {
                    const uint2 ent = hjd_lds_v2_sync(warp_list + (uint32_t)idx * 8u);
                    const uint32_t src = warp_slots + ent.y * 128u + ((chunk ^ (ent.y & 7u)) << 4);
                    const uint4 w = hjd_lds_v4_sync(src);
                    hjd_sts_zero16_sync(src);
                    ((uint4*)coef)[(size_t)ent.x * 8u + chunk] = w;      // 64-bit: ent.x * 8 wraps from block 2^29 on
                }
            }
            __syncwarp();
        }
    }
    // the last sub-sequence that holds data must have completed the image
    if (last_sub && li < s.n_subs && (uint64_t)li * HJD_SS_SUB_BYTES < L && blk < n_blocks) flags |= HJD_ST_OVERRUN;
    if (flags) atomicOr(&status[s.img], flags);
}

// Per-device function attributes and limits (see hjd_kernels_init_device): the write pass needs more than
// the default 48 KB of shared memory; *max_sync_ctas = CTAs of the synchronisation kernel that can be
// resident together (its cooperative launch must not ask for more).
cudaError_t hjd_selfsync_init_device(int* max_sync_ctas)
{
    cudaError_t e = cudaFuncSetAttribute(hjd_k_ss_write, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)(HJD_SS_THREADS * (128 + 8) + 6 * sizeof(HjdHuffTable)));
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(hjd_k_ss_sync, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ss_sync_smem());
    if (e != cudaSuccess) return e;
    int dev = 0, sms = 0, per_sm = 0;
    if ((e = cudaGetDevice(&dev)) != cudaSuccess) return e;
    if ((e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev)) != cudaSuccess) return e;
    if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, hjd_k_ss_sync, HJD_SS_FIX_WARPS * 32, ss_sync_smem())) != cudaSuccess) return e;
    if (const char* env = getenv("HJD_SS_SYNC_PER_SM")) { const int v = atoi(env); if (v >= 1 && v < per_sm) per_sm = v; }   // tuning
    *max_sync_ctas = sms * (per_sm < 1 ? 1 : per_sm);
    return cudaSuccess;
}

cudaError_t hjd_launch_ss_write(const HjdImageDesc* imgs, const HjdTableSet* tsets, const HjdSsImage* ss,
                                const HjdSsWork* work, const HjdSsSeg* segs, int n_work, const uint8_t* dst,
                                const uint32_t* dlen,
                                uint32_t n_subs_total, const uint64_t* x, const uint32_t* prefix, int16_t* coef,
                                int32_t* status, cudaStream_t st)
{
    if (n_work <= 0) return cudaSuccess;
    const size_t smem = HJD_SS_THREADS * (128 + 8) + 6 * sizeof(HjdHuffTable);
    hjd_k_ss_write<<<n_work, HJD_SS_THREADS, smem, st>>>(imgs, tsets, ss, work, segs, dst, dlen, n_subs_total, x, prefix,
                                                        coef, status);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// truncated scans: blocks that never started
// ------------------------------------------------------------------------------------------
// A scan that ends early starts fewer blocks than the frame header promises (the write pass flags
// HJD_ST_OVERRUN).  The slab is not zero-filled beforehand, so the missing blocks are zeroed here to
// keep the output a function of the input alone.  Nothing to do for a complete scan.
__global__ void __launch_bounds__(256)
hjd_k_ss_fill_tail(const HjdImageDesc* __restrict__ imgs, const HjdSsImage* __restrict__ ss, int n_ss,
                   const uint32_t* __restrict__ prefix, int16_t* __restrict__ coef)
{
    // one warp per image: nothing but two loads for a complete scan
    const int k = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (k >= n_ss) return;
    const HjdSsImage s = ss[k];
    const HjdImageDesc* d = imgs + s.img;
    const uint64_t started = prefix[s.sub_base + s.n_subs] - prefix[s.sub_base];
    const uint64_t n_blocks = d->n_blocks;
    if (started >= n_blocks) return;
    uint4* out = (uint4*)coef + (d->block_base + started) * 8;
    const uint64_t n16 = (n_blocks - started) * 8;
    for (uint64_t i = lane; i < n16; i += 32) out[i] = make_uint4(0, 0, 0, 0);
}

cudaError_t hjd_launch_ss_fill_tail(const HjdImageDesc* imgs, const HjdSsImage* ss, int n_ss, const uint32_t* prefix,
                                    int16_t* coef, cudaStream_t st)
{
    if (n_ss <= 0) return cudaSuccess;
    hjd_k_ss_fill_tail<<<(n_ss + 7) / 8, 256, 0, st>>>(imgs, ss, n_ss, prefix, coef);
    return cudaGetLastError();
}
