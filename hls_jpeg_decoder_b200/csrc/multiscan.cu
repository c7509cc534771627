// csrc/multiscan.cu -- entropy decode of multi-scan images (HJD_FLAG_MULTI_SCAN): progressive (SOF2) files and
// sequential files whose components come in separate scans.
//
// One thread decodes one work item, a restart interval of one scan (the trade of kernel 1a and of the
// NO_SELFSYNC path: the bitstream makes nothing smaller independent).  It fills the same coefficient slab as
// kernels 1a / 1b (int16 [block][64], zig-zag order, DC un-differenced), so kernels 2+3 run unchanged.
// The five scan kinds of T.81 G.1.2:
//   sequential   the block decode of kernel 1a (hjd_sym_fields semantics, quirks included), DC predictors int16
//   DC first     pred += diff; coef[0] = pred * 2^Al
//   DC refine    one bit per block, OR-ed in at 2^Al
//   AC first     run / size symbols with EOBRUN (EOBn: 2^n + n further bits); values v * 2^Al
//   AC refine    new coefficients of +-2^Al (size 1); a correction bit for every coefficient of the band that is
//                already nonzero and passed over, EOBRUN included, adds 2^Al in its own sign direction
// EOBRUN and the predictors restart at every interval.  Scans of one dependency level write disjoint (component,
// coefficient) positions, so the host launches one grid per level, in order, and a level sees every bit of the
// levels below it.  The Huffman tables (one pool per batch, de-duplicated by content: optimised per-scan tables
// are rarely shared) are read through the read-only path instead of being staged in shared memory.
#include "multiscan.cuh"
#include "device_common.cuh"

#define HJD_MS_THREADS 128

namespace {

struct MsReader {
    const uint8_t* p;      // next byte
    const uint8_t* end;    // end of this interval
    uint64_t win;          // MSB-aligned bit window
    int nbits;             // valid bits in the window
    int padbits;           // zero bits appended past `end`
};

__device__ __noinline__ void ms_fill(MsReader& r)
{
    while (r.nbits <= 56) {
        if (r.p < r.end) {
            const uint32_t b = __ldg(r.p++);
            if (b == 0xFFu && r.p < r.end) r.p++;            // the stuffed byte after FF (FillNBits, loadjpg.cpp:446-484)
            r.win |= (uint64_t)b << (56 - r.nbits);
        } else {
            r.padbits += 8;                                    // past the interval: zero bits
        }
        r.nbits += 8;
    }
}

__device__ __forceinline__ uint32_t ms_bits(MsReader& r, uint32_t n)          // n <= 16
{
    if (n == 0) return 0;
    if (r.nbits < 16) ms_fill(r);
    const uint32_t v = (uint32_t)(r.win >> (64 - n));
    r.win <<= n;
    r.nbits -= (int)n;
    return v;
}

// Entry of the symbol at the head of the window (see HjdHuffTable), read from global memory.
__device__ __forceinline__ uint32_t ms_lookup(MsReader& r, const HjdHuffTable* __restrict__ t)
{
    if (r.nbits < 32) ms_fill(r);
    const uint32_t hi = (uint32_t)(r.win >> 32);
    uint32_t e = __ldg(&t->lut[hi >> (32 - HJD_LUT_BITS)]);
    if ((e & 31u) == 0) {
        const uint32_t idx = ((hi >> 16) & ((1u << (16 - HJD_LUT_BITS)) - 1u)) >> ((e >> 5) & 7u);
        e = __ldg(&t->lut2[(((e >> 8) << 1) + idx) & (HJD_LUT2_SIZE - 1)]);
    }
    const uint32_t len = e & 31u;
    r.win <<= len;
    r.nbits -= (int)len;
    return e;
}

__device__ __forceinline__ int ms_pred(uint32_t ci, int p0, int p1, int p2) { return ci == 0 ? p0 : (ci == 1 ? p1 : p2); }
__device__ __forceinline__ void ms_set_pred(uint32_t ci, int v, int& p0, int& p1, int& p2)
{
    p0 = ci == 0 ? v : p0;
    p1 = ci == 1 ? v : p1;
    p2 = ci == 2 ? v : p2;
}

// DetermineSign (loadjpg.cpp:396-409): v of `size` bits with a leading 0 bit is v - (2^size - 1)
__device__ __forceinline__ int ms_extend(uint32_t v, uint32_t size)
{
    return (size && !(v >> (size - 1))) ? (int)v - (int)((1u << size) - 1u) : (int)v;
}

} // namespace

__global__ void __launch_bounds__(HJD_MS_THREADS)
hjd_k_multiscan(const uint8_t* __restrict__ arena, const HjdImageDesc* __restrict__ imgs,
                const HjdScanDesc* __restrict__ scans, const HjdMsWork* __restrict__ work, int n_work,
                const uint32_t* __restrict__ starts, const HjdHuffTable* __restrict__ tabs,
                int16_t* __restrict__ coef, int32_t* __restrict__ status)
{
    const int item = blockIdx.x * HJD_MS_THREADS + threadIdx.x;
    if (item >= n_work) return;
    const HjdMsWork w = work[item];
    const HjdScanDesc& s = scans[w.scan];     // fields read where used (indexed ones must not become a local copy)
    const HjdImageDesc& d = imgs[s.image];
    const uint32_t j = w.interval;
    const uint32_t total = s.mcus_x * s.mcus_y;
    const uint32_t ri = s.restart_interval;
    const uint32_t first = ri ? j * ri : 0;
    if (first >= total) return;
    const uint32_t n_mcu = ri ? min(ri, total - first) : total;

    const uint8_t* base = arena + s.scan_off;
    uint32_t b0 = starts[s.start_base + j];
    uint32_t b1 = (j + 1 < s.n_intervals) ? starts[s.start_base + j + 1] - 2 : s.scan_len;
    if (b1 < b0 || b1 > s.scan_len) b1 = b0;
    MsReader r{base + b0, base + b1, 0ull, 0, 0};

    const uint32_t hf = d.hf, vf = d.vf, ny = d.ncomp == 3 ? hf * vf : 1, bpm = d.blocks_per_mcu;
    const bool inter = s.ncomp > 1;
    const uint32_t ss = s.ss, se = s.se, al = s.al;
    const int p1 = 1 << al, m1 = -p1;
    int pred0 = 0, pred1 = 0, pred2 = 0;       // DC predictors of the scan's components (registers, not an indexed array)
    uint32_t eobrun = 0;
    int flags = 0;

    for (uint32_t u = 0; u < n_mcu; u++) {
        const uint32_t mcu = first + u;
        const uint32_t by0 = mcu / s.mcus_x, bx0 = mcu - by0 * s.mcus_x;
        const uint32_t nb = inter ? bpm : 1;
        for (uint32_t bi = 0; bi < nb; bi++) {
            // which component this block belongs to, and its slab index
            uint32_t ci, blk;
            if (inter) {
                // interleaved: the frame's MCU; the scan's components in order, luma with hf * vf blocks
                uint32_t c = 0, sub = 0, left = bi;
                for (ci = 0; ci < s.ncomp; ci++) {
                    const uint32_t n = s.comp[ci] == 0 ? ny : 1;
                    if (left < n) { sub = left; break; }
                    left -= n;
                }
                if (ci >= s.ncomp) break;                      // fewer components than the frame: MCU done
                c = s.comp[ci];
                blk = mcu * bpm + (c == 0 ? sub : ny + c - 1);
            } else {
                ci = 0;
                const uint32_t c = s.comp[0];
                if (c == 0) blk = ((by0 / vf) * d.mcus_x + bx0 / hf) * bpm + (by0 % vf) * hf + bx0 % hf;
                else blk = mcu * bpm + ny + c - 1;
            }
            int16_t* cb = coef + (d.block_base + blk) * 64;
            if (r.padbits > 512) { flags |= HJD_ST_OVERRUN; goto done; }      // data exhausted long ago

            if (s.kind == HJD_SCAN_SEQ) {
                const HjdHuffTable* tdc = tabs + s.dc_tab[ci];
                const HjdHuffTable* tac = tabs + s.ac_tab[ci];
                uint32_t k = 0;
                while (k < 64) {
                    const uint32_t e = ms_lookup(r, k ? tac : tdc);
                    const uint32_t size = (e >> 5) & 15u, kadv = (e >> 9) & 127u;
                    const int val = ms_extend(ms_bits(r, size), size);
                    if (kadv == 127u) { flags |= HJD_ST_BAD_CODE; goto done; }
                    const uint32_t kpos = k + kadv - 1u;
                    if (k == 0) {                                                  // DCT[0] = data + prevDC in int16
                        const int p = (int)(short)(ms_pred(ci, pred0, pred1, pred2) + (int)(short)val);
                        ms_set_pred(ci, p, pred0, pred1, pred2);
                        cb[0] = (int16_t)p;
                    } else if (size) {
                        if (kpos <= 63u) cb[kpos] = (int16_t)val;
                        else flags |= HJD_ST_COEF_RANGE;
                    }
                    k += kadv;
                    if (r.padbits > 512) { flags |= HJD_ST_OVERRUN; goto done; }   // ignored symbols on padding
                }
            } else if (s.kind == HJD_SCAN_DC_FIRST) {
                const uint32_t e = ms_lookup(r, tabs + s.dc_tab[ci]);
                const uint32_t size = (e >> 5) & 15u;
                const int val = ms_extend(ms_bits(r, size), size);
                if (((e >> 9) & 127u) == 127u) { flags |= HJD_ST_BAD_CODE; goto done; }
                const int p = ms_pred(ci, pred0, pred1, pred2) + val;
                ms_set_pred(ci, p, pred0, pred1, pred2);
                cb[0] = (int16_t)(p * p1);
            } else if (s.kind == HJD_SCAN_DC_REFINE) {
                if (ms_bits(r, 1)) cb[0] = (int16_t)(cb[0] | p1);
            } else if (s.kind == HJD_SCAN_AC_FIRST) {
                if (eobrun) { eobrun--; continue; }
                const HjdHuffTable* tac = tabs + s.ac_tab[0];
                for (uint32_t k = ss; k <= se;) {
                    const uint32_t e = ms_lookup(r, tac);
                    const uint32_t size = (e >> 5) & 15u, run = (e >> 9) & 127u;
                    if (run == 127u) { flags |= HJD_ST_BAD_CODE; goto done; }
                    if (size) {
                        k += run;
                        const int val = ms_extend(ms_bits(r, size), size);
                        if (k <= se) cb[k] = (int16_t)(val * p1);
                        else flags |= HJD_ST_COEF_RANGE;
                        k++;
                    } else if (run == 15u) {
                        k += 16;                                                   // ZRL
                        if (k > se + 1) flags |= HJD_ST_COEF_RANGE;
                    } else {
                        eobrun = (1u << run) + ms_bits(r, run) - 1u;               // EOBn: this block is the first
                        break;
                    }
                }
            } else {                                                               // HJD_SCAN_AC_REFINE
                const HjdHuffTable* tac = tabs + s.ac_tab[0];
                uint32_t k = ss;
                if (eobrun == 0) {
                    for (; k <= se; k++) {
                        const uint32_t e = ms_lookup(r, tac);
                        uint32_t size = (e >> 5) & 15u;
                        int run = (int)((e >> 9) & 127u);
                        if (run == 127) { flags |= HJD_ST_BAD_CODE; goto done; }
                        int nz = 0;
                        if (size) {
                            if (size != 1u) flags |= HJD_ST_COEF_RANGE;
                            nz = ms_bits(r, 1) ? p1 : m1;
                        } else if (run != 15) {
                            eobrun = (1u << run) + ms_bits(r, (uint32_t)run);      // the rest of this block: below
                            break;
                        }
                        // pass over nonzero coefficients (a correction bit each) and `run` zero ones
                        for (; k <= se; k++) {
                            const int c = cb[k];
                            if (c != 0) {
                                if (ms_bits(r, 1) && (c & p1) == 0) cb[k] = (int16_t)(c >= 0 ? c + p1 : c + m1);
                            } else if (--run < 0) {
                                break;
                            }
                        }
                        if (nz) {
                            if (k <= se) cb[k] = (int16_t)nz;
                            else flags |= HJD_ST_COEF_RANGE;
                        }
                        if (r.padbits > 512) { flags |= HJD_ST_OVERRUN; goto done; }
                    }
                }
                if (eobrun) {
                    for (; k <= se; k++) {
                        const int c = cb[k];
                        if (c != 0 && ms_bits(r, 1) && (c & p1) == 0) cb[k] = (int16_t)(c >= 0 ? c + p1 : c + m1);
                    }
                    eobrun--;
                }
            }
        }
    }
    if (r.nbits < r.padbits) flags |= HJD_ST_OVERRUN;                              // read past the interval
done:
    if (flags) atomicOr(&status[s.image], flags);
}

cudaError_t hjd_launch_multiscan(const uint8_t* arena, const HjdImageDesc* imgs, const HjdScanDesc* scans,
                                 const HjdMsWork* work, int n_work, const uint32_t* starts, const HjdHuffTable* tabs,
                                 int16_t* coef, int32_t* status, cudaStream_t st)
{
    if (n_work <= 0) return cudaSuccess;
    hjd_k_multiscan<<<(n_work + HJD_MS_THREADS - 1) / HJD_MS_THREADS, HJD_MS_THREADS, 0, st>>>(
        arena, imgs, scans, work, n_work, starts, tabs, coef, status);
    return cudaGetLastError();
}
