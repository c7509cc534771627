// csrc/jpeg_parse.cpp -- see jpeg_parse.h.
#include "jpeg_parse.h"
#include "../../include/hjd.h"
#include <string.h>

namespace {

struct Reader {
    const uint8_t* p;
    size_t n, i;
    bool   need(size_t k) const { return i + k <= n; }
    uint8_t  u8()  { return p[i++]; }
    uint16_t u16() { uint16_t v = (uint16_t)((p[i] << 8) | p[i + 1]); i += 2; return v; }
};

uint64_t fnv1a(uint64_t h, const void* data, size_t n)
{
    const uint8_t* d = (const uint8_t*)data;
    for (size_t k = 0; k < n; k++) { h ^= d[k]; h *= 1099511628211ull; }
    return h;
}

int parse_dqt(Reader& r, size_t end, HjdParsed* o)
{
    // openjpg.cpp:120-155: Pq/Tq byte then 64 entries in zig-zag order; several tables per segment.
    while (r.i < end) {
        uint8_t pq_tq = r.u8();
        int pq = pq_tq >> 4, tq = pq_tq & 15;
        if (pq != 0 || tq > 3) return HJD_IMG_ERR_UNSUPPORTED;   // reference: prints, reads 64 bytes anyway (136-148)
        if (r.i + 64 > end) return HJD_IMG_ERR_TRUNCATED;
        memcpy(o->qt[tq], r.p + r.i, 64);
        o->qt_present[tq] = 1;
        r.i += 64;
    }
    return HJD_IMG_OK;
}

int parse_dht(Reader& r, size_t end, HjdParsed* o)
{
    // openjpg.cpp:234-305: Tc/Th byte, 16 counts, then the symbols; several tables per segment.
    while (r.i < end) {
        if (r.i + 17 > end) return HJD_IMG_ERR_TRUNCATED;
        uint8_t tc_th = r.u8();
        int tc = tc_th >> 4, th = tc_th & 15;
        if (tc > 1 || th > 3) return HJD_IMG_ERR_UNSUPPORTED;
        HjdRawHuff* h = tc ? &o->ac[th] : &o->dc[th];
        int total = 0;
        for (int k = 0; k < 16; k++) { h->bits[k] = r.u8(); total += h->bits[k]; }
        if (total > 256) return HJD_IMG_ERR_BAD_TABLE;
        if (r.i + (size_t)total > end) return HJD_IMG_ERR_TRUNCATED;
        memset(h->vals, 0, sizeof h->vals);
        memcpy(h->vals, r.p + r.i, (size_t)total);
        h->nvals = total;
        h->present = 1;
        r.i += (size_t)total;
    }
    return HJD_IMG_OK;
}

} // namespace

int hjd_exif_orientation(const uint8_t* p, size_t len)
{
    if (len < 6 || memcmp(p, "Exif\0\0", 6) != 0) return 0;
    const uint8_t* t = p + 6;                      // TIFF header; its offsets are relative to here
    const uint64_t n = len - 6;
    if (n < 8) return 1;
    bool le;
    if (t[0] == 'I' && t[1] == 'I' && t[2] == 0x2A && t[3] == 0) le = true;
    else if (t[0] == 'M' && t[1] == 'M' && t[2] == 0 && t[3] == 0x2A) le = false;
    else return 1;
    auto u16 = [&](uint64_t at) { return (uint32_t)(le ? t[at] | t[at + 1] << 8 : t[at] << 8 | t[at + 1]); };
    auto u32 = [&](uint64_t at) { return le ? u16(at) | u16(at + 2) << 16 : u16(at) << 16 | u16(at + 2); };
    const uint64_t ifd = u32(4);
    if (ifd + 2 > n) return 1;
    const uint64_t count = u16(ifd);
    if (ifd + 2 + 12 * count > n) return 1;        // 64-bit: no overflow
    for (uint64_t k = 0; k < count; k++) {
        const uint64_t e = ifd + 2 + 12 * k;
        if (u16(e) != 0x0112) continue;
        if (u16(e + 2) != 3 || u32(e + 4) != 1) return 1;    // SHORT, count 1: the value sits in the first two bytes
        const uint32_t v = u16(e + 8);
        return v >= 1 && v <= 8 ? (int)v : 1;
    }
    return 1;
}

size_t hjd_scan_length(const uint8_t* scan, size_t avail)
{
    // Large file that ends with EOI: taken as "nothing follows the scan" without walking it (a memchr walk
    // over 1024 x 0.36 MB would cost the host tens of milliseconds per batch, on the critical path of the
    // host-buffer decode).  A large file with a second image appended after its EOI (MPF) is therefore sized
    // as before: decoded correctly, its trailer merely counted as scan bytes.
    if (avail >= HJD_SCAN_WALK_MAX && scan[avail - 2] == 0xFF && scan[avail - 1] == 0xD9) return avail - 2;
    // Otherwise (small files; trailer, padding, a caller's oversized buffer): the scan ends at the first
    // marker that is neither a stuffed FF00 nor RSTn, so that what follows EOI is neither counted as
    // restart markers nor sized and decoded as entropy data.
    const uint8_t* p = scan;
    const uint8_t* e = scan + avail;
    while (p + 1 < e) {
        p = (const uint8_t*)memchr(p, 0xFF, (size_t)(e - 1 - p));
        if (!p) break;
        const uint8_t m = p[1];
        if (m == 0x00 || (m & 0xF8) == 0xD0) p += 2;
        else if (m == 0xFF) p += 1;                                  // fill byte
        else return (size_t)(p - scan);
    }
    return avail;
}

int hjd_parse_jpeg(const uint8_t* buf, size_t size, HjdParsed* o)
{
    memset(o, 0, sizeof *o);
    o->status = HJD_IMG_ERR_NOT_JPEG;
    o->orientation = 1;
    if (!buf || size < 4 || buf[0] != 0xFF || buf[1] != 0xD8) return o->status;   // openjpg.cpp:481
    Reader r{buf, size, 2};
    bool have_frame = false, have_exif = false;
    int cid[3] = {0, 0, 0};
    int chf[3] = {1, 1, 1}, cvf[3] = {1, 1, 1};

    for (;;) {
        if (!r.need(2)) return o->status = HJD_IMG_ERR_TRUNCATED;
        if (r.u8() != 0xFF) return o->status = HJD_IMG_ERR_NOT_JPEG;              // openjpg.cpp:383-386
        uint8_t m = r.u8();
        while (m == 0xFF) {                                                       // fill bytes, 389-392
            if (!r.need(1)) return o->status = HJD_IMG_ERR_TRUNCATED;
            m = r.u8();
        }
        if (m == 0xD8 || m == 0x01 || (m >= 0xD0 && m <= 0xD7)) continue;         // stand-alone markers
        if (m == 0xD9) return o->status = HJD_IMG_ERR_TRUNCATED;                  // EOI before SOS
        if (!r.need(2)) return o->status = HJD_IMG_ERR_TRUNCATED;
        size_t seg = r.i;
        uint16_t len = r.u16();
        if (len < 2 || seg + len > size) return o->status = HJD_IMG_ERR_TRUNCATED;
        size_t end = seg + len;

        if (m == 0xDB) {
            int rc = parse_dqt(r, end, o);
            if (rc) return o->status = rc;
        } else if (m == 0xC4) {
            int rc = parse_dht(r, end, o);
            if (rc) return o->status = rc;
        } else if (m == 0xC0 || m == 0xC1) {
            // SOF0 (baseline) and SOF1 restricted to 8 bits: same sequential Huffman decode.
            if (len < 8) return o->status = HJD_IMG_ERR_TRUNCATED;
            uint8_t prec = r.u8();
            o->height = r.u16();
            o->width  = r.u16();
            o->ncomp  = r.u8();
            if (prec != 8 || (o->ncomp != 1 && o->ncomp != 3)) return o->status = HJD_IMG_ERR_UNSUPPORTED;
            if (len < 8 + 3 * o->ncomp) return o->status = HJD_IMG_ERR_TRUNCATED;
            if (o->width == 0 || o->height == 0) return o->status = HJD_IMG_ERR_UNSUPPORTED;
            if ((uint64_t)o->width * o->height > HJD_MAX_PIXELS) return o->status = HJD_IMG_ERR_UNSUPPORTED;
            for (int c = 0; c < o->ncomp; c++) {
                cid[c] = r.u8();
                uint8_t s = r.u8();
                chf[c] = s >> 4;                                                  // openjpg.cpp:344-345
                cvf[c] = s & 15;
                o->tq[c] = r.u8();
                if (o->tq[c] > 3) return o->status = HJD_IMG_ERR_UNSUPPORTED;
            }
            have_frame = true;
        } else if (m >= 0xC2 && m <= 0xCF && m != 0xC8 && m != 0xCC) {
            return o->status = HJD_IMG_ERR_UNSUPPORTED;                           // progressive / lossless / arithmetic
        } else if (m == 0xDD) {
            if (len < 4) return o->status = HJD_IMG_ERR_TRUNCATED;
            o->restart_interval = r.u16();                                        // Ri (the reference reads Lr here)
        } else if (m == 0xDA) {
            if (!have_frame) return o->status = HJD_IMG_ERR_UNSUPPORTED;
            if (len < 6) return o->status = HJD_IMG_ERR_TRUNCATED;
            int ns = r.u8();
            if (ns != o->ncomp) return o->status = HJD_IMG_ERR_UNSUPPORTED;       // one interleaved scan only
            if (len < 6 + 2 * ns) return o->status = HJD_IMG_ERR_TRUNCATED;
            for (int k = 0; k < ns; k++) {
                int cs = r.u8();
                uint8_t t = r.u8();
                int c = -1;
                for (int j = 0; j < o->ncomp; j++) if (cid[j] == cs) c = j;
                if (c < 0 || (t >> 4) > 3 || (t & 15) > 3) return o->status = HJD_IMG_ERR_UNSUPPORTED;
                o->td[c] = t >> 4;                                                // openjpg.cpp:212-213
                o->ta[c] = t & 15;
            }
            uint8_t ss = r.u8(), se = r.u8(), ahal = r.u8();
            if (ss != 0 || se != 63 || ahal != 0) return o->status = HJD_IMG_ERR_UNSUPPORTED;
            o->scan_off = end;
            o->scan_len = hjd_scan_length(buf + end, size - end);
            break;
        } else if (m == 0xE1 && !have_exif) {
            const int v = hjd_exif_orientation(buf + r.i, end - r.i);
            if (v) { o->orientation = v; have_exif = true; }
        }
        // APPn, COM and anything else with a length: skipped (openjpg.cpp:448-461)
        r.i = end;
    }

    if (o->ncomp == 3) {
        // The reference's MCU walk assumes chroma 1x1 and luma in {1,2}^2 (loadjpg.cpp:945-997, 884-932).
        if (chf[1] != 1 || cvf[1] != 1 || chf[2] != 1 || cvf[2] != 1) return o->status = HJD_IMG_ERR_UNSUPPORTED;
        if (chf[0] < 1 || chf[0] > 2 || cvf[0] < 1 || cvf[0] > 2) return o->status = HJD_IMG_ERR_UNSUPPORTED;
        o->hf = chf[0];
        o->vf = cvf[0];
    } else {
        o->hf = o->vf = 1;   // a single-component scan is not interleaved: one block per MCU
    }
    for (int c = 0; c < o->ncomp; c++) {
        if (!o->qt_present[o->tq[c]]) return o->status = HJD_IMG_ERR_BAD_TABLE;
        if (!o->dc[o->td[c]].present || !o->ac[o->ta[c]].present) return o->status = HJD_IMG_ERR_BAD_TABLE;
    }
    return o->status = HJD_IMG_OK;
}

// One entropy-coded segment: its length (up to the first marker that is neither FF00 nor RSTn, as
// hjd_scan_length) and, appended to `starts`, the start of each of its RSTn-delimited intervals (relative to
// the segment), in the same pass.
static size_t walk_segment(const uint8_t* scan, size_t avail, std::vector<uint32_t>& starts)
{
    starts.push_back(0);
    const uint8_t* p = scan;
    const uint8_t* e = scan + avail;
    while (p + 1 < e) {
        p = (const uint8_t*)memchr(p, 0xFF, (size_t)(e - 1 - p));
        if (!p) break;
        const uint8_t m = p[1];
        if (m == 0x00) p += 2;
        else if ((m & 0xF8) == 0xD0) { starts.push_back((uint32_t)(p + 2 - scan)); p += 2; }
        else if (m == 0xFF) p += 1;                                  // fill byte
        else return (size_t)(p - scan);
    }
    return avail;
}

int hjd_parse_jpeg_multi(const uint8_t* buf, size_t size, HjdMultiParsed* mp)
{
    HjdParsed* o = &mp->frame;
    memset(o, 0, sizeof *o);
    mp->scans.clear();
    mp->starts.clear();
    o->status = HJD_IMG_ERR_NOT_JPEG;
    o->orientation = 1;
    if (!buf || size < 4 || buf[0] != 0xFF || buf[1] != 0xD8) return o->status;
    Reader r{buf, size, 2};
    bool have_frame = false, progressive = false, have_exif = false;
    int cid[3] = {0, 0, 0};
    int chf[3] = {1, 1, 1}, cvf[3] = {1, 1, 1};
    uint32_t dri = 0;
    // per (component, coefficient): Al of the last scan that coded it (-1: none yet), level of that scan
    int al_of[3][64], level_of[3][64];
    bool seq_done[3] = {false, false, false};
    for (int c = 0; c < 3; c++)
        for (int k = 0; k < 64; k++) al_of[c][k] = level_of[c][k] = -1;
    HjdParsed later;                        // DQT after the first scan: parsed (bounds, errors) but not used
    // The file ends before EOI: the scans so far are decoded (a missing scan leaves its coefficients 0).
#define HJD_END_EARLY() do { if (mp->scans.empty()) return o->status = HJD_IMG_ERR_TRUNCATED; goto frame_checks; } while (0)

    for (;;) {
        if (!r.need(2)) HJD_END_EARLY();
        if (r.u8() != 0xFF) return o->status = HJD_IMG_ERR_NOT_JPEG;
        uint8_t m = r.u8();
        while (m == 0xFF) {
            if (!r.need(1)) HJD_END_EARLY();
            m = r.u8();
        }
        if (m == 0xD8 || m == 0x01 || (m >= 0xD0 && m <= 0xD7)) continue;
        if (m == 0xD9) HJD_END_EARLY();
        if (!r.need(2)) HJD_END_EARLY();
        const size_t seg = r.i;
        const uint16_t len = r.u16();
        if (len < 2 || seg + len > size) HJD_END_EARLY();
        const size_t end = seg + len;

        if (m == 0xDB) {
            const int rc = parse_dqt(r, end, mp->scans.empty() ? o : &later);
            if (rc) return o->status = rc;
        } else if (m == 0xC4) {
            const int rc = parse_dht(r, end, o);
            if (rc) return o->status = rc;
        } else if (m == 0xC0 || m == 0xC1 || m == 0xC2) {
            if (have_frame) return o->status = HJD_IMG_ERR_UNSUPPORTED;
            if (len < 8) return o->status = HJD_IMG_ERR_TRUNCATED;
            const uint8_t prec = r.u8();
            o->height = r.u16();
            o->width  = r.u16();
            o->ncomp  = r.u8();
            if (prec != 8 || (o->ncomp != 1 && o->ncomp != 3)) return o->status = HJD_IMG_ERR_UNSUPPORTED;
            if (len < 8 + 3 * o->ncomp) return o->status = HJD_IMG_ERR_TRUNCATED;
            if (o->width == 0 || o->height == 0) return o->status = HJD_IMG_ERR_UNSUPPORTED;
            if ((uint64_t)o->width * o->height > HJD_MAX_PIXELS) return o->status = HJD_IMG_ERR_UNSUPPORTED;
            for (int c = 0; c < o->ncomp; c++) {
                cid[c] = r.u8();
                const uint8_t s = r.u8();
                chf[c] = s >> 4;
                cvf[c] = s & 15;
                o->tq[c] = r.u8();
                if (o->tq[c] > 3) return o->status = HJD_IMG_ERR_UNSUPPORTED;
            }
            have_frame = true;
            progressive = (m == 0xC2);
        } else if (m >= 0xC3 && m <= 0xCF && m != 0xC4 && m != 0xC8 && m != 0xCC) {
            return o->status = HJD_IMG_ERR_UNSUPPORTED;                           // lossless / arithmetic
        } else if (m == 0xDD) {
            if (len < 4) return o->status = HJD_IMG_ERR_TRUNCATED;
            dri = r.u16();
        } else if (m == 0xDA) {
            if (!have_frame) return o->status = HJD_IMG_ERR_UNSUPPORTED;
            if (mp->scans.size() >= HJD_MAX_SCANS) return o->status = HJD_IMG_ERR_UNSUPPORTED;
            if (len < 6) return o->status = HJD_IMG_ERR_TRUNCATED;
            HjdScanParsed s;
            memset(&s, 0, sizeof s);
            s.ncomp = r.u8();
            if (s.ncomp < 1 || s.ncomp > o->ncomp) return o->status = HJD_IMG_ERR_UNSUPPORTED;
            if (len < 6 + 2 * s.ncomp) return o->status = HJD_IMG_ERR_TRUNCATED;
            int td[3] = {0, 0, 0}, ta[3] = {0, 0, 0};
            for (int k = 0; k < s.ncomp; k++) {
                const int cs = r.u8();
                const uint8_t t = r.u8();
                int c = -1;
                for (int j = 0; j < o->ncomp; j++) if (cid[j] == cs) c = j;
                // components of a scan come in frame order (T.81 B.2.3), so each at most once
                if (c < 0 || (k && c <= s.comp[k - 1]) || (t >> 4) > 3 || (t & 15) > 3) return o->status = HJD_IMG_ERR_UNSUPPORTED;
                s.comp[k] = c;
                td[k] = t >> 4;
                ta[k] = t & 15;
            }
            s.ss = r.u8();
            s.se = r.u8();
            const uint8_t ahal = r.u8();
            s.ah = ahal >> 4;
            s.al = ahal & 15;
            // T.81 G.1.1.1
            if (!progressive) {
                if (s.ss != 0 || s.se != 63 || ahal != 0) return o->status = HJD_IMG_ERR_UNSUPPORTED;
                for (int k = 0; k < s.ncomp; k++) {
                    if (seq_done[s.comp[k]]) return o->status = HJD_IMG_ERR_UNSUPPORTED;   // every component exactly once
                    seq_done[s.comp[k]] = true;
                }
                s.kind = HJD_SCAN_SEQ;
            } else {
                if (s.al > 13 || s.ah > 13) return o->status = HJD_IMG_ERR_UNSUPPORTED;
                if (s.ss == 0) {
                    if (s.se != 0) return o->status = HJD_IMG_ERR_UNSUPPORTED;
                    s.kind = s.ah ? HJD_SCAN_DC_REFINE : HJD_SCAN_DC_FIRST;
                } else {
                    if (s.ncomp != 1 || s.se < s.ss || s.se > 63) return o->status = HJD_IMG_ERR_UNSUPPORTED;
                    s.kind = s.ah ? HJD_SCAN_AC_REFINE : HJD_SCAN_AC_FIRST;
                }
                for (int k = 0; k < s.ncomp; k++)
                    for (int q = s.ss; q <= s.se; q++) {
                        const int prev = al_of[s.comp[k]][q];
                        // a first pass codes a coefficient once; a refinement follows it, one bit at a time
                        if (s.ah == 0 ? prev != -1 : (prev != s.ah || s.al != s.ah - 1)) return o->status = HJD_IMG_ERR_UNSUPPORTED;
                    }
            }
            s.level = 0;
            for (int k = 0; k < s.ncomp; k++)
                for (int q = s.ss; q <= s.se; q++)
                    if (level_of[s.comp[k]][q] + 1 > s.level) s.level = level_of[s.comp[k]][q] + 1;
            for (int k = 0; k < s.ncomp; k++)
                for (int q = s.ss; q <= s.se; q++) { level_of[s.comp[k]][q] = s.level; al_of[s.comp[k]][q] = s.al; }
            // snapshot of the tables this scan decodes with
            const bool need_dc = s.kind == HJD_SCAN_SEQ || s.kind == HJD_SCAN_DC_FIRST;
            const bool need_ac = s.kind == HJD_SCAN_SEQ || s.kind == HJD_SCAN_AC_FIRST || s.kind == HJD_SCAN_AC_REFINE;
            for (int k = 0; k < s.ncomp; k++) {
                if (need_dc) { if (!o->dc[td[k]].present) return o->status = HJD_IMG_ERR_BAD_TABLE; s.dc[k] = o->dc[td[k]]; }
                if (need_ac) { if (!o->ac[ta[k]].present) return o->status = HJD_IMG_ERR_BAD_TABLE; s.ac[k] = o->ac[ta[k]]; }
            }
            s.restart_interval = dri;
            s.off = end;
            s.first_start = (uint32_t)mp->starts.size();
            s.len = walk_segment(buf + end, size - end, mp->starts);
            s.n_starts = (uint32_t)mp->starts.size() - s.first_start;
            if (s.len > 0xFFFFFF00ull) return o->status = HJD_IMG_ERR_UNSUPPORTED;
            mp->scans.push_back(s);
            r.i = end + s.len;
            continue;
        } else if (m == 0xE1 && !have_exif && mp->scans.empty()) {
            const int v = hjd_exif_orientation(buf + r.i, end - r.i);
            if (v) { o->orientation = v; have_exif = true; }
        }
        r.i = end;
    }
#undef HJD_END_EARLY

frame_checks:
    if (o->ncomp == 3) {
        if (chf[1] != 1 || cvf[1] != 1 || chf[2] != 1 || cvf[2] != 1) return o->status = HJD_IMG_ERR_UNSUPPORTED;
        if (chf[0] < 1 || chf[0] > 2 || cvf[0] < 1 || cvf[0] > 2) return o->status = HJD_IMG_ERR_UNSUPPORTED;
        o->hf = chf[0];
        o->vf = cvf[0];
    } else {
        o->hf = o->vf = 1;
    }
    for (int c = 0; c < o->ncomp; c++)
        if (!o->qt_present[o->tq[c]]) return o->status = HJD_IMG_ERR_BAD_TABLE;
    o->restart_interval = mp->scans[0].restart_interval;
    o->scan_off = mp->scans[0].off;
    o->scan_len = 0;
    for (const HjdScanParsed& s : mp->scans) o->scan_len += s.len;
    return o->status = HJD_IMG_OK;
}

void hjd_scan_grid(const HjdParsed& f, const HjdScanParsed& s, uint32_t* mx, uint32_t* my)
{
    const uint32_t hf = (uint32_t)f.hf, vf = (uint32_t)f.vf;
    if (s.ncomp > 1 || s.comp[0] != 0) {          // interleaved, or a chroma component (1x1: its grid is the MCU grid)
        *mx = (f.width + 8 * hf - 1) / (8 * hf);
        *my = (f.height + 8 * vf - 1) / (8 * vf);
    } else {                                       // luma alone: its own block grid
        *mx = (f.width + 7) / 8;
        *my = (f.height + 7) / 8;
    }
}

#define HJD_TAB_DC  0
#define HJD_TAB_AC  1
#define HJD_TAB_RAW 2      // progressive AC: raw run, see hjd_build_huff_table_raw

static uint32_t sym_fields(uint32_t len, uint32_t sym, int mode)
{
    // keep in sync with hjd_sym_fields() in device_common.cuh (ProcessHuffmanBlock's run/size logic)
    const uint32_t size = sym & 15u, run = sym >> 4;
    if (mode == HJD_TAB_RAW) return HJD_SYM_FIELDS(len, size, run);
    if (mode == HJD_TAB_DC) return HJD_SYM_FIELDS(len, size, 1);
    if (size) return HJD_SYM_FIELDS(len, size, run + 1);
    return HJD_SYM_FIELDS(len, 0, run == 0 ? 63 : (run == 15 ? 16 : 0));
}

static bool build_table(const HjdRawHuff& raw, int mode, HjdHuffTable* t);

bool hjd_build_huff_table(const HjdRawHuff& raw, bool is_ac, HjdHuffTable* t)
{
    return build_table(raw, is_ac ? HJD_TAB_AC : HJD_TAB_DC, t);
}

bool hjd_build_huff_table_raw(const HjdRawHuff& raw, HjdHuffTable* t)
{
    return build_table(raw, HJD_TAB_RAW, t);
}

static bool build_table(const HjdRawHuff& raw, int mode, HjdHuffTable* t)
{
    for (int i = 0; i < HJD_LUT_SIZE; i++) t->lut[i] = (uint16_t)HJD_BAD_ENTRY;
    for (int i = 0; i < HJD_LUT2_SIZE; i++) t->lut2[i] = (uint16_t)HJD_BAD_ENTRY;
    // Canonical code assignment (what GenHuffCodes does, openjpg.cpp:48-66): codes of one length
    // are consecutive; the counter doubles when the length grows.
    uint32_t first_code[17];
    {
        uint32_t code = 0;
        for (int L = 1; L <= 16; L++) {
            const uint32_t cnt = raw.bits[L - 1];
            if (code + cnt > (1u << L)) return false;                // over-subscribed
            first_code[L] = code;
            code = (code + cnt) << 1;
        }
    }
    // first level: every code of up to LUT_BITS bits, replicated over the bits that follow it
    int valptr = 0;
    for (int L = 1; L <= HJD_LUT_BITS; L++) {
        for (int k = 0; k < raw.bits[L - 1]; k++) {
            const uint32_t first = (first_code[L] + (uint32_t)k) << (HJD_LUT_BITS - L);
            const uint16_t e = (uint16_t)sym_fields((uint32_t)L, raw.vals[valptr + k], mode);
            for (uint32_t j = 0; j < (1u << (HJD_LUT_BITS - L)); j++) t->lut[first + j] = e;
        }
        valptr += raw.bits[L - 1];
    }
    // second level: per LUT_BITS-bit prefix that starts longer codes, a sub-table indexed by the next
    // nb = (longest code under the prefix) - LUT_BITS bits
    const int valptr_long = valptr;
    uint8_t nb_of[HJD_LUT_SIZE];
    memset(nb_of, 0, sizeof nb_of);
    for (int L = HJD_LUT_BITS + 1; L <= 16; L++)
        for (int k = 0; k < raw.bits[L - 1]; k++) {
            const uint32_t prefix = (first_code[L] + (uint32_t)k) >> (L - HJD_LUT_BITS);
            nb_of[prefix] = (uint8_t)(L - HJD_LUT_BITS);                // lengths ascend: the last one wins
        }
    uint32_t used = 0;
    for (uint32_t p = 0; p < HJD_LUT_SIZE; p++) {
        if (!nb_of[p]) continue;
        if (used + (1u << nb_of[p]) > HJD_LUT2_SIZE) return false;      // cannot happen for canonical codes (see HJD_LUT2_SIZE)
        t->lut[p] = (uint16_t)((uint32_t)((16 - HJD_LUT_BITS) - nb_of[p]) << 5 | (used >> 1) << 8);
        used += 1u << nb_of[p];
    }
    valptr = valptr_long;
    for (int L = HJD_LUT_BITS + 1; L <= 16; L++) {
        for (int k = 0; k < raw.bits[L - 1]; k++) {
            const uint32_t code = first_code[L] + (uint32_t)k;
            const uint32_t prefix = code >> (L - HJD_LUT_BITS);
            const uint32_t nb = nb_of[prefix], off = (uint32_t)(t->lut[prefix] >> 8) << 1;
            const uint32_t rest = code & ((1u << (L - HJD_LUT_BITS)) - 1u);   // the bits after the prefix
            const uint32_t rep = nb - (uint32_t)(L - HJD_LUT_BITS);          // bits that follow the code
            const uint16_t e = (uint16_t)sym_fields((uint32_t)L, raw.vals[valptr + k], mode);
            for (uint32_t j = 0; j < (1u << rep); j++) t->lut2[off + (rest << rep) + j] = e;
        }
        valptr += raw.bits[L - 1];
    }
    return true;
}

uint32_t hjd_host_huff_lookup(const HjdHuffTable* t, uint32_t peek16)
{
    // host mirror of the kernels' symbol lookup (first level, then hjd_long_code in device_common.cuh)
    peek16 &= 0xFFFFu;
    // host mirror of hjd_lookup() in device_common.cuh
    uint32_t e = t->lut[peek16 >> (16 - HJD_LUT_BITS)];
    if ((e & 31u) == 0) {
        const uint32_t idx = (peek16 & ((1u << (16 - HJD_LUT_BITS)) - 1u)) >> ((e >> 5) & 7u);
        e = t->lut2[(((e >> 8) << 1) + idx) & (HJD_LUT2_SIZE - 1)];
    }
    return e;
}

int hjd_build_table_set(const HjdParsed& p, HjdTableSet* out)
{
    memset(out, 0, sizeof *out);
    // De-duplicate by (class, table id): Cb and Cr normally share one DC and one AC table.
    int slot_dc[4] = {-1, -1, -1, -1}, slot_ac[4] = {-1, -1, -1, -1};
    int n = 0;
    for (int c = 0; c < p.ncomp; c++) {
        if (slot_dc[p.td[c]] < 0) {
            if (!hjd_build_huff_table(p.dc[p.td[c]], false, &out->tab[n])) return HJD_IMG_ERR_BAD_TABLE;
            slot_dc[p.td[c]] = n++;
        }
        if (slot_ac[p.ta[c]] < 0) {
            if (!hjd_build_huff_table(p.ac[p.ta[c]], true, &out->tab[n])) return HJD_IMG_ERR_BAD_TABLE;
            slot_ac[p.ta[c]] = n++;
        }
        out->dc_of_comp[c] = (uint8_t)slot_dc[p.td[c]];
        out->ac_of_comp[c] = (uint8_t)slot_ac[p.ta[c]];
    }
    out->n_tabs = n;
    return HJD_IMG_OK;
}

// FP16 bit pattern of an integer 0 <= v < 2048 (exactly representable)
static uint32_t half_bits_of_small_int(uint32_t v)
{
    if (v == 0) return 0;
    if (v > 2047) v = 2047;     // 16-bit tables are rejected by the parser; never reached
    int e = 0;
    while ((v >> (e + 1)) != 0) e++;
    return ((uint32_t)(e + 15) << 10) | ((v << (10 - e)) & 0x3FFu);
}

void hjd_build_quant_set(const HjdParsed& p, HjdQuantSet* out)
{
    memset(out, 0, sizeof *out);
    for (int c = 0; c < p.ncomp; c++) {
        // loadjpg.cpp:984 dequantises Cb with Cr's table; identical whenever both name one table.
        int src = (p.ncomp == 3 && c == 1) ? 2 : c;
        for (int k = 0; k < 64; k++) out->q[c][k] = p.qt[p.tq[src]][k];
        for (int k = 0; k < 32; k++)
            out->qp[c][k] = (uint32_t)p.qt[p.tq[src]][2 * k] | ((uint32_t)p.qt[p.tq[src]][2 * k + 1] << 24);
        for (int k = 0; k < 32; k++)
            out->qh[c][k] = half_bits_of_small_int(p.qt[p.tq[src]][2 * k]) | (half_bits_of_small_int(p.qt[p.tq[src]][2 * k + 1]) << 16);
    }
}

void hjd_raw_tables(const HjdParsed& p, HjdRawTables* out)
{
    memset(out, 0, sizeof *out);
    out->huff[0] = out->quant[0] = (uint8_t)p.ncomp;
    for (int c = 0; c < p.ncomp; c++) {
        uint8_t* h = out->huff + 4 + c * 2 * (16 + 256);
        const HjdRawHuff* t[2] = {&p.dc[p.td[c]], &p.ac[p.ta[c]]};
        for (int k = 0; k < 2; k++, h += 16 + 256) {
            memcpy(h, t[k]->bits, 16);
            memcpy(h + 16, t[k]->vals, (size_t)(t[k]->nvals < 256 ? t[k]->nvals : 256));
        }
        const int src = (p.ncomp == 3 && c == 1) ? 2 : c;           // Cb is de-quantised with Cr's table (loadjpg.cpp:984)
        memcpy(out->quant + 4 + c * 64, p.qt[p.tq[src]], 64);
    }
}

uint64_t hjd_table_key(const HjdParsed& p)
{
    uint64_t h = 1469598103934665603ull;
    h = fnv1a(h, &p.ncomp, sizeof p.ncomp);
    for (int c = 0; c < p.ncomp; c++) {
        const HjdRawHuff& d = p.dc[p.td[c]];
        const HjdRawHuff& a = p.ac[p.ta[c]];
        h = fnv1a(h, d.bits, 16); h = fnv1a(h, d.vals, (size_t)d.nvals);
        h = fnv1a(h, a.bits, 16); h = fnv1a(h, a.vals, (size_t)a.nvals);
        h = fnv1a(h, "|", 1);
    }
    return h;
}

uint64_t hjd_quant_key(const HjdParsed& p)
{
    uint64_t h = 1469598103934665603ull;
    h = fnv1a(h, &p.ncomp, sizeof p.ncomp);
    for (int c = 0; c < p.ncomp; c++) {
        int src = (p.ncomp == 3 && c == 1) ? 2 : c;
        h = fnv1a(h, p.qt[p.tq[src]], 64);
    }
    return h;
}

uint32_t hjd_host_find_intervals(const uint8_t* scan, size_t scan_len, uint32_t* starts, uint32_t max_out)
{
    uint32_t n = 0;
    if (max_out) starts[n++] = 0;
    const uint8_t* p = scan;
    const uint8_t* e = scan + scan_len;
    while (p + 1 < e) {
        p = (const uint8_t*)memchr(p, 0xFF, (size_t)(e - 1 - p));
        if (!p) break;
        if ((p[1] & 0xF8) == 0xD0) {
            if (n < max_out) starts[n] = (uint32_t)(p + 2 - scan);
            n++;
            p += 2;
        } else {
            p += 1;
        }
    }
    return n;
}
