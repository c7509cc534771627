// csrc/orient.cu -- EXIF orientation pass (HJD_FLAG_EXIF_ORIENT): a permutation of the bytes the decode kernels wrote.
//
// The decode kernels are unchanged: an oriented image is decoded into a private staging region of the output slab
// (batch_plan.cpp, plan_staging), and this pass writes it turned into the image's place.  It costs one read and one
// write of the oriented images' output only.  Fusing it into the six output kernels' epilogues would turn their row
// stores into column stores for orientations 5-8 and needs registers and shared memory the tensor-core kernel does not
// have (DESIGN §4.5, §4.11).
#include "orient.cuh"

// One CTA per output tile of T x T pixels.  A CTA never spans two images, so the orientation is uniform in it.
//  1. The tile's source rectangle (T x T pixels, transposed for orientations 5-8) is read as whole aligned 4-byte
//     words, one row per warp at a time, consecutive lanes on consecutive words; every load of a thread is issued before
//     the first store to shared memory.  Row r is staged from the word that holds its first byte, so that byte lies at
//     the row's phase, its offset mod 4.
//  2. One thread per output pixel moves its bpp bytes from the staged source tile to a staged output tile, whose rows
//     are laid out as they will be stored (at the output row's phase).  Row pitches are an odd number of words, so the
//     column reads of a transposing orientation fall into distinct banks.
//  3. The output rows are written as whole aligned words, one row per warp, consecutive lanes on consecutive words; the
//     words at the tile's left and right edges, which it shares with the neighbouring tiles, byte by byte, only the bytes
//     that belong to it.
// Every staged byte is read from HBM once and every output byte written once.  Offsets are 64-bit.
template <int BPP>
__global__ void __launch_bounds__(HJD_ORIENT_THREADS)
hjd_k_orient(uint8_t* __restrict__ out, const HjdOrientJob* __restrict__ jobs, const uint32_t* __restrict__ tile_prefix,
             int n_jobs)
{
    constexpr uint32_t T = HJD_ORIENT_TILE;
    constexpr uint32_t NW = (T * BPP + 6) / 4;            // most words one tile row touches (up to 3 bytes of phase each side)
    constexpr uint32_t WORDS = NW | 1u;                   // pitch of a staged row in words: odd
    constexpr uint32_t PITCH = 4 * WORDS;
    constexpr uint32_t WARPS = HJD_ORIENT_THREADS / 32;
    constexpr uint32_t ROWS = T / WARPS;                  // rows per warp
    constexpr uint32_t KW = (NW + 31) / 32;               // words per lane and row
    static_assert(T % WARPS == 0 && T % 32 == 0, "tile rows split evenly over the warps, columns over the lanes");
    __shared__ uint32_t s_in[T * WORDS], s_out[T * WORDS];

    // The job of this tile: the last k with tile_prefix[k] <= key (every job has a tile, so the prefix rises), by a
    // 32-ary search of each warp (lane l tests the l-th of 32 evenly spaced candidates): two dependent loads for
    // 1024 jobs where a binary search takes ten, ahead of every tile.
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t key = blockIdx.x + tile_prefix[0];
    uint32_t lo = 0, n = (uint32_t)n_jobs;                // tile_prefix[lo] <= key; the job is in [lo, lo + n)
    while (n > 1) {
        const uint32_t step = (n + 31) / 32, at = lo + lane * step;
        const unsigned le = __ballot_sync(0xFFFFFFFFu, lane * step < n && tile_prefix[at] <= key);
        const uint32_t l = 31 - __clz(le);                // lane 0 tests lo itself
        lo += l * step;
        n = min(step, n - l * step);
    }
    const HjdOrientJob j = jobs[lo];
    const uint32_t W = j.w, H = j.h, o = j.o;
    // out(x, y) = in(a, b) with a = x or W'-1-x, b = y or H'-1-y (orientations 1-4), and the same with x and y
    // exchanged (5-8): tr = exchange, fx / fy = mirror the output's x / y.
    const bool tr = o >= 5;
    const bool fx = o == 2 || o == 3 || o == 6 || o == 7;
    const bool fy = o == 3 || o == 4 || o == 7 || o == 8;
    const uint32_t OW = tr ? H : W, OH = tr ? W : H;
    const uint32_t t = key - tile_prefix[lo];
    const uint32_t tiles_x = (OW + T - 1) / T;
    const uint32_t ty = t / tiles_x, tx = t - ty * tiles_x;
    const uint32_t ox0 = tx * T, oy0 = ty * T;
    const uint32_t ow = min(T, OW - ox0), oh = min(T, OH - oy0);
    uint32_t sx0, sy0, sw, sh;                            // the tile's source rectangle
    if (!tr) { sw = ow; sh = oh; sx0 = fx ? W - ox0 - ow : ox0; sy0 = fy ? H - oy0 - oh : oy0; }
    else     { sw = oh; sh = ow; sx0 = fy ? W - oy0 - oh : oy0; sy0 = fx ? H - ox0 - ow : ox0; }
    const uint64_t src_stride = (uint64_t)W * BPP, dst_stride = (uint64_t)OW * BPP;
    const uint8_t* __restrict__ src = out + j.src_off;    // both 256-byte aligned
    uint8_t* __restrict__ dst = out + j.dst_off;
    const uint32_t slen = sw * BPP, dlen = ow * BPP;
    // phases (offsets mod 4) of source / output rows: 32-bit arithmetic keeps the low two bits
    const uint32_t sb32 = (uint32_t)src_stride, db32 = (uint32_t)dst_stride, sxb = sx0 * BPP, oxb = ox0 * BPP;

    {
        uint32_t v[ROWS][KW];
#pragma unroll
        for (uint32_t i = 0; i < ROWS; i++) {
            const uint32_t r = warp + WARPS * i;
            const uint64_t a = (uint64_t)(sy0 + r) * src_stride + sxb;
            const uint32_t* p = (const uint32_t*)(src + (a & ~3ull));
            const uint32_t nw = r < sh ? ((uint32_t)(a & 3u) + slen + 3) >> 2 : 0;
#pragma unroll
            for (uint32_t q = 0; q < KW; q++)
                if (lane + 32 * q < nw) v[i][q] = __ldg(p + lane + 32 * q);
        }
#pragma unroll
        for (uint32_t i = 0; i < ROWS; i++) {
            const uint32_t r = warp + WARPS * i;
            const uint32_t nw = r < sh ? ((((sy0 + r) * sb32 + sxb) & 3u) + slen + 3) >> 2 : 0;
#pragma unroll
            for (uint32_t q = 0; q < KW; q++)
                if (lane + 32 * q < nw) s_in[r * WORDS + lane + 32 * q] = v[i][q];
        }
    }
    __syncthreads();

    const uint8_t* si = (const uint8_t*)s_in;
    uint8_t* so = (uint8_t*)s_out;
#pragma unroll 2
    for (uint32_t i = 0; i < ROWS; i++) {
        const uint32_t y = warp + WARPS * i;
        if (y >= oh) break;
        const uint32_t yy = fy ? oh - 1 - y : y;
        const uint32_t drow = y * PITCH + (((oy0 + y) * db32 + oxb) & 3u);
        const uint32_t srow = yy * PITCH + (((sy0 + yy) * sb32 + sxb) & 3u);     // orientations 1-4: source row yy
#pragma unroll
        for (uint32_t q = 0; q < T / 32; q++) {
            const uint32_t u = lane + 32 * q;
            if (u >= ow) break;
            const uint32_t xx = fx ? ow - 1 - u : u;
            // 5-8: source row xx, column yy
            const uint32_t s = tr ? xx * PITCH + (((sy0 + xx) * sb32 + sxb) & 3u) + yy * BPP : srow + xx * BPP;
#pragma unroll
            for (uint32_t c = 0; c < BPP; c++) so[drow + u * BPP + c] = si[s + c];
        }
    }
    __syncthreads();

#pragma unroll 2
    for (uint32_t i = 0; i < ROWS; i++) {
        const uint32_t y = warp + WARPS * i;
        if (y >= oh) break;
        const uint64_t b = (uint64_t)(oy0 + y) * dst_stride + oxb;
        const uint32_t head = (uint32_t)(b & 3u), end = head + dlen;
        uint32_t* p = (uint32_t*)(dst + (b & ~3ull));
#pragma unroll
        for (uint32_t q = 0; q < KW; q++) {
            const uint32_t k = lane + 32 * q;
            if (4 * k >= end) break;
            const uint32_t v = s_out[y * WORDS + k];
            if (4 * k >= head && 4 * k + 4 <= end) {
                p[k] = v;
            } else {
#pragma unroll
                for (uint32_t e = 0; e < 4; e++)
                    if (4 * k + e >= head && 4 * k + e < end) ((uint8_t*)(p + k))[e] = (uint8_t)(v >> (8 * e));
            }
        }
    }
}

cudaError_t hjd_launch_orient(uint8_t* out, const HjdOrientJob* jobs, const uint32_t* tile_prefix, int n_jobs,
                              uint32_t n_tiles, int bpp, cudaStream_t st)
{
    if (n_jobs <= 0 || n_tiles == 0) return cudaSuccess;
    if (bpp == 1) hjd_k_orient<1><<<n_tiles, HJD_ORIENT_THREADS, 0, st>>>(out, jobs, tile_prefix, n_jobs);
    else hjd_k_orient<3><<<n_tiles, HJD_ORIENT_THREADS, 0, st>>>(out, jobs, tile_prefix, n_jobs);
    return cudaGetLastError();
}
