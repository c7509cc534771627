// csrc/batch_plan.cpp -- host planning of one batch upload (see batch_plan.h).  Stages, in order: parse the headers,
// lay out the images in the slabs, plan the chunks, build each chunk's work lists, plan kernel 1b.  Each index-limit
// guard sits in the stage that computes its quantity.
#include "batch_plan.h"

#include <string.h>
#include <algorithm>
#include <memory>
#include <thread>

uint32_t ms_scan_items(const HjdParsed& frame, const HjdScanParsed& p, uint32_t* mcus_x, uint32_t* mcus_y, bool want_all)
{
    uint32_t mx, my;
    hjd_scan_grid(frame, p, &mx, &my);
    if (mcus_x) { *mcus_x = mx; *mcus_y = my; }
    const uint64_t total = (uint64_t)mx * my;
    const uint64_t want = p.restart_interval ? (total + p.restart_interval - 1) / p.restart_interval : 1;
    return (uint32_t)(want_all || want < p.n_starts ? want : p.n_starts);
}

FrameGeometry frame_geometry(uint32_t width, uint32_t height, int ncomp, int hf, int vf, uint32_t restart_interval)
{
    FrameGeometry g;
    g.blocks_per_mcu = ncomp == 3 ? hf * vf + 2 : 1;
    g.mcus_x = (width + 8 * hf - 1) / (8 * hf);
    g.mcus_y = (height + 8 * vf - 1) / (8 * vf);
    g.n_mcus = g.mcus_x * g.mcus_y;
    g.n_intervals = restart_interval ? (g.n_mcus + restart_interval - 1) / restart_interval : 1;
    return g;
}

// Index of the per-scan Huffman table built from `raw` (mode 0: DC, 1: sequential AC, 2: progressive AC with the raw
// run), shared by every scan of the batch with the same contents; -1: the code is over-subscribed.
static int ms_table(BatchPlan* p, const HjdRawHuff& raw, int mode)
{
    std::vector<uint8_t> key(17 + (size_t)raw.nvals);
    key[0] = (uint8_t)mode;
    memcpy(&key[1], raw.bits, 16);
    memcpy(&key[17], raw.vals, (size_t)raw.nvals);
    uint64_t h = 1469598103934665603ull;
    for (uint8_t v : key) { h ^= v; h *= 1099511628211ull; }
    auto range = p->ms_tab_of.equal_range(h);
    for (auto it = range.first; it != range.second; ++it)
        if (p->ms_tab_raw[it->second] == key) return (int)it->second;
    HjdHuffTable t;
    if (!(mode == 2 ? hjd_build_huff_table_raw(raw, &t) : hjd_build_huff_table(raw, mode == 1, &t))) return -1;
    p->ms_tabs.push_back(t);
    p->ms_tab_raw.push_back(std::move(key));
    p->ms_tab_of.emplace(h, (uint32_t)p->ms_tabs.size() - 1);
    return (int)p->ms_tabs.size() - 1;
}

// Scan descriptors, tables, interval starts and work items of multi-scan image i (file at arena offset dev_off).
// A scan with fewer RSTn markers than its DRI implies (a file cut inside it) gets the intervals it has: the last one
// runs to the end of the data, and the image is flagged HJD_IMG_WARN_RESTART.  HJD_IMG_OK or HJD_IMG_ERR_BAD_TABLE.
static int ms_add_image(unsigned flags, BatchPlan* p, int i, const HjdMultiParsed& mp, uint64_t dev_off)
{
    const size_t scan0 = p->scans.size(), start0 = p->ms_starts.size(), work0 = p->mswork.size();
    uint32_t items = 0, n_scans = 0;
    for (const HjdScanParsed& s : mp.scans) {
        if (!scan_is_read(flags, s)) continue;
        n_scans++;
        HjdScanDesc sd;
        memset(&sd, 0, sizeof sd);
        sd.image = (uint32_t)i;
        sd.ncomp = (uint8_t)s.ncomp;
        for (int k = 0; k < s.ncomp; k++) sd.comp[k] = (uint8_t)s.comp[k];
        sd.ss = (uint8_t)s.ss; sd.se = (uint8_t)s.se; sd.ah = (uint8_t)s.ah; sd.al = (uint8_t)s.al;
        sd.kind = (uint8_t)s.kind; sd.level = (uint8_t)(s.level < 255 ? s.level : 255);
        sd.restart_interval = s.restart_interval;
        sd.n_intervals = ms_scan_items(mp.frame, s, &sd.mcus_x, &sd.mcus_y);
        if (s.restart_interval && s.n_starts != ms_scan_items(mp.frame, s, nullptr, nullptr, true)) p->host_restart_warn[i] = 1;
        sd.start_base = (uint32_t)p->ms_starts.size();
        sd.scan_len = (uint32_t)s.len;
        sd.scan_off = dev_off + s.off;
        for (int k = 0; k < s.ncomp; k++) {
            const int td = s.dc[k].present ? ms_table(p, s.dc[k], 0) : 0;
            const int ta = s.ac[k].present ? ms_table(p, s.ac[k], s.kind == HJD_SCAN_SEQ ? 1 : 2) : 0;
            if (td < 0 || ta < 0) {
                p->scans.resize(scan0); p->ms_starts.resize(start0); p->mswork.resize(work0);
                return HJD_IMG_ERR_BAD_TABLE;
            }
            sd.dc_tab[k] = (uint32_t)td;
            sd.ac_tab[k] = (uint32_t)ta;
        }
        for (uint32_t j = 0; j < sd.n_intervals; j++) {
            p->ms_starts.push_back(mp.starts[s.first_start + j]);
            p->mswork.push_back(HjdMsWork{(uint32_t)p->scans.size(), j});
        }
        items += sd.n_intervals;
        p->scans.push_back(sd);
    }
    p->ms_items[i] = items;
    p->n_scans[i] = n_scans;
    return HJD_OK;
}

// Stage 1, header parse.  What the layout pass needs of one image's header parse.
struct Lite {
    int status;
    uint32_t width, height, restart_interval;
    int ncomp, hf, vf;
    size_t scan_off, scan_len;
    uint64_t tk, qk;
    uint64_t ms_items;         // multi-scan work items (what ms_add_image will add)
    int trep, qrep;            // image whose tables / quantisation tables these are byte-identical to (itself: a representative)
    int orientation;           // EXIF orientation the file states (1..8)
};
typedef std::vector<std::unique_ptr<HjdMultiParsed>> MultiList;

// Header parse and table hashing of every image, in parallel for large batches (8192 thumbnails: 9 ms
// of the host's time on one thread).  What the layout pass needs is kept in a small record;
// the few images that bring a new table or quantisation set are parsed once more there.
// Table and quantisation sets are shared by images with identical DHT / DQT contents.  The 64-bit
// hash only finds candidates: every worker keeps the raw tables of the images that introduced a key
// (to that worker) and compares the bytes on a hit, so an image is either byte-identical to an earlier
// image of its worker (trep / qrep = that image) or a representative itself; representatives are
// compared byte for byte with the sets built so far in the layout pass.  A hash collision therefore
// costs a set of its own, never somebody else's tables.
// HJD_FLAG_MULTI_SCAN: files the single-scan parse rejects as unsupported get the multi-scan walk; these
// images keep the result (scans, interval starts, table snapshots) in `multi` for the layout pass.
static int parse_files(const std::vector<FileRef>& files, unsigned flags, std::vector<Lite>& lite, MultiList& multi,
                       std::string* err)
{
    const int n = (int)files.size();
    auto parse_range = [&](int lo, int hi) {
        HjdParsed p;
        struct Seen { uint64_t key; int image; HjdRawTables raw; };
        std::vector<Seen> seen_t, seen_q;
        HjdRawTables raw;
        for (int i = lo; i < hi; i++) {
            Lite& l = lite[(size_t)i];
            memset(&l, 0, sizeof l);
            int st = (files[i].ptr && files[i].size > 0) ? hjd_parse_jpeg(files[i].ptr, (size_t)files[i].size, &p)
                                                         : HJD_IMG_ERR_NOT_JPEG;
            if (st == HJD_IMG_OK && p.scan_len > 0xFFFFFF00ull) st = HJD_IMG_ERR_UNSUPPORTED;
            if (st == HJD_IMG_ERR_UNSUPPORTED && (flags & HJD_FLAG_MULTI_SCAN)) {
                std::unique_ptr<HjdMultiParsed> mp(new HjdMultiParsed());
                st = hjd_parse_jpeg_multi(files[i].ptr, (size_t)files[i].size, mp.get());
                if (st == HJD_IMG_OK && mp->frame.scan_len > 0xFFFFFF00ull) st = HJD_IMG_ERR_UNSUPPORTED;
                if (st == HJD_IMG_OK) {
                    p = mp->frame;
                    for (const HjdScanParsed& sp : mp->scans)
                        if (scan_is_read(flags, sp)) l.ms_items += ms_scan_items(mp->frame, sp, nullptr, nullptr);
                    multi[(size_t)i] = std::move(mp);
                }
            }
            l.status = st;
            l.orientation = (files[i].ptr && files[i].size > 0) ? p.orientation : 1;
            if (st != HJD_IMG_OK) continue;
            l.width = p.width; l.height = p.height; l.restart_interval = p.restart_interval;
            l.ncomp = p.ncomp; l.hf = p.hf; l.vf = p.vf;
            l.scan_off = p.scan_off; l.scan_len = p.scan_len;
            l.tk = hjd_table_key(p); l.qk = hjd_quant_key(p);
            hjd_raw_tables(p, &raw);
            l.trep = l.qrep = i;
            bool hit = multi[(size_t)i] != nullptr;      // multi-scan images carry per-scan tables instead of a table set
            for (const Seen& sn : seen_t)
                if (sn.key == l.tk && memcmp(sn.raw.huff, raw.huff, sizeof raw.huff) == 0) { l.trep = sn.image; hit = true; break; }
            if (!hit && seen_t.size() < 64) seen_t.push_back(Seen{l.tk, i, raw});
            hit = false;
            for (const Seen& sn : seen_q)
                if (sn.key == l.qk && memcmp(sn.raw.quant, raw.quant, sizeof raw.quant) == 0) { l.qrep = sn.image; hit = true; break; }
            if (!hit && seen_q.size() < 64) seen_q.push_back(Seen{l.qk, i, raw});
        }
    };
    unsigned hw = std::thread::hardware_concurrency();
    int nt = n >= 2048 ? (int)(hw < 2 ? 1 : (hw > 8 ? 8 : hw)) : 1;
    if (nt <= 1) parse_range(0, n);
    else {
        std::vector<std::thread> pool;
        const int per = (n + nt - 1) / nt;
        for (int k = 0; k < nt; k++) {
            const int lo = k * per, hi = lo + per < n ? lo + per : n;
            if (lo < hi) pool.emplace_back(parse_range, lo, hi);
        }
        for (auto& th : pool) th.join();
    }

    // Multi-scan work items are numbered in int (hjd_k_multiscan's thread index), so a batch holds fewer than 2^31.
    uint64_t items = 0;
    for (const Lite& l : lite) items += l.ms_items;
    if (items >= 0x80000000ull) { *err = "batch exceeds 2^31 multi-scan work items"; return HJD_ERR_ARG; }
    return HJD_OK;
}

// Stage 2, image layout.  The table and quantisation sets of the layout pass (see parse_files): an image
// byte-identical to an earlier image of its worker takes that image's set; a representative is parsed once more and
// compared byte for byte with the sets built so far.
struct SetSharing {
    BatchPlan* p;
    std::vector<uint32_t> tset_of_img, qset_of_img;
    HjdParsed full;                    // re-parse target for the representatives
    HjdRawTables full_raw;
    bool have_full = false;            // full / full_raw hold the current image

    SetSharing(BatchPlan* plan, int n) : p(plan), tset_of_img((size_t)n, 0), qset_of_img((size_t)n, 0) {}
    void reparse(const FileRef& f)
    {
        hjd_parse_jpeg(f.ptr, (size_t)f.size, &full);
        hjd_raw_tables(full, &full_raw);
        have_full = true;
    }
    // The table set of image i in *tset; the image's status (a reused image inherits its representative's).
    int table_set(const FileRef& f, int i, const Lite& ps, uint32_t* tset)
    {
        if (ps.trep != i) {
            *tset = tset_of_img[(size_t)ps.trep];
            return p->parse_status[ps.trep];                       // e.g. an over-subscribed DHT
        }
        reparse(f);
        auto range = p->tset_of.equal_range(ps.tk);
        for (auto it = range.first; it != range.second; ++it)
            if (memcmp(p->tset_raw[it->second].huff, full_raw.huff, sizeof full_raw.huff) == 0) { *tset = it->second; return HJD_IMG_OK; }
        HjdTableSet ts;
        const int st = hjd_build_table_set(full, &ts);
        if (st == HJD_IMG_OK) {
            *tset = (uint32_t)p->tsets.size(); p->tsets.push_back(ts); p->tset_raw.push_back(full_raw);
            p->tset_of.emplace(ps.tk, *tset);
            if (ts.n_tabs > p->max_tabs) p->max_tabs = ts.n_tabs;
        }
        return st;
    }
    uint32_t quant_set(const FileRef& f, int i, const Lite& ps)
    {
        if (ps.qrep != i) return qset_of_img[(size_t)ps.qrep];
        if (!have_full) reparse(f);
        auto range = p->qset_of.equal_range(ps.qk);
        for (auto it = range.first; it != range.second; ++it)
            if (memcmp(p->qset_raw[it->second].quant, full_raw.quant, sizeof full_raw.quant) == 0) return it->second;
        HjdQuantSet qs;
        hjd_build_quant_set(full, &qs);
        p->qsets.push_back(qs); p->qset_raw.push_back(full_raw);
        p->qset_of.emplace(ps.qk, (uint32_t)p->qsets.size() - 1);
        return (uint32_t)p->qsets.size() - 1;
    }
};

// A restart-free scan goes to kernel 1b (speculative self-synchronising decode) instead of one thread.  Its sub_base /
// chunk_base follow from the chunk plan (plan_selfsync).
static void add_selfsync_image(BatchPlan* p, int i, HjdImageDesc& d)
{
    HjdSsImage si;
    memset(&si, 0, sizeof si);
    si.img = (uint32_t)i;
    si.n_subs = (d.scan_len + HJD_SS_SUB_BYTES - 1) / HJD_SS_SUB_BYTES;
    si.lead = (uint32_t)(d.scan_off & 15);
    si.n_chunks = (uint32_t)(((uint64_t)d.scan_len + si.lead + 15) / 16);
    si.dst_off = p->ss_dst_bytes;
    d.n_intervals = 0;
    d.n_subs = si.n_subs;
    p->ss.push_back(si);
    p->ss_dst_bytes += align_up((uint64_t)d.scan_len + HJD_SS_SLACK + 16, 256);   // + 16: the slack is zeroed from the next 16-byte boundary
}

// Descriptors, sets and slab offsets of every image; ms_w0[i]: the first multi-scan work item of image i (n + 1).
static int layout_images(const std::vector<FileRef>& files, const PlanConfig& cfg, const std::vector<Lite>& lite,
                         const MultiList& multi, BatchPlan* p, std::vector<uint32_t>& ms_w0, std::string* err)
{
    const int n = (int)files.size();
    SetSharing sets(p, n);
    for (int i = 0; i < n; i++) {
        HjdImageDesc& d = p->imgs[i];
        memset(&d, 0, sizeof d);
        d.interval_base = p->total_intervals;
        d.block_base = p->total_blocks;
        d.rgb_off = p->rgb_bytes;
        d.y_off = d.cb_off = d.cr_off = p->plane_bytes;
        const Lite& ps = lite[(size_t)i];
        p->orientation[i] = (uint8_t)ps.orientation;
        const HjdMultiParsed* mp = multi[(size_t)i].get();
        int st = ps.status;
        uint32_t tset = 0, qset = 0;
        sets.have_full = false;
        if (st == HJD_IMG_OK && mp) {
            st = ms_add_image(cfg.flags, p, i, *mp, files[i].dev_off);
            p->ms_image[i] = 1;
            sets.full = mp->frame;
            hjd_raw_tables(sets.full, &sets.full_raw);
            sets.have_full = true;
        } else if (st == HJD_IMG_OK) {
            st = sets.table_set(files[i], i, ps, &tset);
        }
        if (st == HJD_IMG_OK) qset = sets.quant_set(files[i], i, ps);
        sets.tset_of_img[(size_t)i] = tset; sets.qset_of_img[(size_t)i] = qset;
        p->parse_status[i] = st;
        ms_w0[(size_t)i + 1] = (uint32_t)p->mswork.size();
        if (st != HJD_IMG_OK) { p->any_parse_error = true; continue; }   // n_intervals = n_blocks = 0: skipped
        if (!mp) p->n_scans[i] = 1;

        const FrameGeometry g = frame_geometry(ps.width, ps.height, ps.ncomp, ps.hf, ps.vf, ps.restart_interval);
        d.width = ps.width; d.height = ps.height;
        d.ncomp = (uint8_t)ps.ncomp; d.hf = (uint8_t)ps.hf; d.vf = (uint8_t)ps.vf;
        d.blocks_per_mcu = (uint8_t)g.blocks_per_mcu;
        d.mcus_x = g.mcus_x; d.mcus_y = g.mcus_y; d.n_mcus = g.n_mcus;
        d.restart_interval = ps.restart_interval;
        d.n_intervals = mp ? 0 : g.n_intervals;      // multi-scan images: entropy decode by the multi-scan kernel only
        d.scan_len = (uint32_t)ps.scan_len;
        d.scan_off = files[i].dev_off + ps.scan_off;
        if (!mp && !(cfg.flags & HJD_FLAG_NO_SELFSYNC) && ps.restart_interval == 0 && ps.scan_len >= HJD_SS_MIN_BYTES)
            add_selfsync_image(p, i, d);
        d.table_set = tset; d.quant_set = qset;
        d.n_blocks = (uint64_t)d.n_mcus * d.blocks_per_mcu;
        d.y_pitch = d.mcus_x * 8 * ps.hf;
        d.c_pitch = d.mcus_x * 8;
        const uint64_t ysz = (uint64_t)d.y_pitch * d.mcus_y * 8 * ps.vf;
        const uint64_t csz = ps.ncomp == 3 ? (uint64_t)d.c_pitch * d.mcus_y * 8 : 0;
        d.y_off = p->plane_bytes;
        d.cb_off = d.y_off + align_up(ysz, 256);
        d.cr_off = d.cb_off + align_up(csz, 256);
        p->plane_bytes = d.cr_off + align_up(csz, 256);
        p->rgb_bytes += align_up(image_out_bytes(cfg.flags, ps.width, ps.height), 256);
        p->total_intervals += d.n_intervals;
        p->total_blocks += d.n_blocks;
        p->scan_bytes += ps.scan_len;
        p->pixels += (uint64_t)ps.width * ps.height;

        if ((cfg.flags & HJD_FLAG_HOST_SCAN) && d.n_intervals) {
            const size_t at = p->host_istart.size();
            p->host_istart.resize(at + d.n_intervals, (uint32_t)ps.scan_len);
            const uint32_t found = hjd_host_find_intervals(files[i].ptr + ps.scan_off, ps.scan_len,
                                                           p->host_istart.data() + at, d.n_intervals);
            if (ps.restart_interval && found != d.n_intervals) p->host_restart_warn[i] = 1;
        }
    }
    if (p->total_blocks >= 0xFFFFFFFFull) { *err = "batch exceeds 2^32 blocks"; return HJD_ERR_ARG; }
    // kernel 1b numbers the 16-byte chunks of the restart-free scans in uint32, with one gap per chunk of the plan and
    // a sentinel: about 64 GiB of restart-free scan data
    uint64_t ck = 0;
    for (const HjdSsImage& si : p->ss) ck += si.n_chunks;
    if (ck + (uint64_t)n + 2 > 0xFFFFFFFFull) {
        *err = "restart-free scans of the batch exceed 2^32 16-byte chunks (64 GiB)";
        return HJD_ERR_ARG;
    }
    p->mcu_cta.assign((size_t)n + 1, 0);
    for (int i = 0; i < n; i++)
        p->mcu_cta[i + 1] = p->mcu_cta[i] + (p->imgs[i].blocks_per_mcu ? p->imgs[i].n_mcus : 0);
    if (cfg.flags & HJD_FLAG_GRAY_OUT) {
        // fewer luma blocks than blocks (< 2^32, checked above), so the prefix fits in uint32
        p->luma_cta.assign((size_t)n + 1, 0);
        for (int i = 0; i < n; i++)
            p->luma_cta[i + 1] = p->luma_cta[i] +
                                 (p->imgs[i].blocks_per_mcu ? (uint32_t)luma_blocks(p->imgs[i].width, p->imgs[i].height) : 0);
    }
    return HJD_OK;
}

// HJD_FLAG_EXIF_ORIENT: every decodable image whose file states an orientation other than 1 is decoded into a private
// staging region behind rgb_bytes (its descriptor's rgb_off, which the decode kernels write to) and turned into its place
// in the slab (out_off) by the orientation pass.  Private regions: chunks in flight together never share one.
static void plan_staging(const PlanConfig& cfg, BatchPlan* p)
{
    const int n = (int)p->imgs.size();
    p->out_off.resize((size_t)n);
    for (int i = 0; i < n; i++) {
        HjdImageDesc& d = p->imgs[i];
        p->out_off[i] = d.rgb_off;
        if (!(cfg.flags & HJD_FLAG_EXIF_ORIENT) || p->orientation[i] == 1 || !d.blocks_per_mcu) continue;
        d.rgb_off = p->rgb_bytes + p->stage_bytes;
        p->stage_bytes += align_up(image_out_bytes(cfg.flags, d.width, d.height), 256);
    }
}

// The orientation jobs of a chunk's images, and the exclusive prefix of their tiles (one batch-wide list).  The tile
// count fits in uint32: every tile covers at least one luma block of its image, and a batch has fewer than 2^32 blocks.
static void chunk_orient(const PlanConfig& cfg, BatchPlan* p, Chunk& c)
{
    if (p->orient_tiles.empty()) p->orient_tiles.push_back(0);
    c.oj0 = (uint32_t)p->orient_jobs.size();
    for (int i = c.img0; i < c.img1; i++) {
        const HjdImageDesc& d = p->imgs[i];
        if (d.rgb_off == p->out_off[i]) continue;
        HjdOrientJob j;
        memset(&j, 0, sizeof j);
        j.src_off = d.rgb_off;
        j.dst_off = p->out_off[i];
        j.w = scaled_dim(cfg.flags, d.width);
        j.h = scaled_dim(cfg.flags, d.height);
        j.o = p->orientation[i];
        p->orient_jobs.push_back(j);
        p->orient_tiles.push_back(p->orient_tiles.back() + orient_tiles(j.w, j.h));
    }
    c.oj1 = (uint32_t)p->orient_jobs.size();
}

// Stage 3: contiguous image ranges of roughly equal block counts.
static void plan_chunks(const PlanConfig& cfg, BatchPlan* p)
{
    const int n = (int)p->imgs.size();
    if (n == 0) return;
    int want = 1;
    if (cfg.chunked && cfg.overlap) {
        const uint64_t per_chunk = cfg.overlap > 1 ? (uint64_t)cfg.overlap : 1500000ull;
        want = (int)(p->total_blocks / per_chunk);
        if (want > 8) want = 8;
        if (want > n) want = n;
        if (want < 1) want = 1;
    }
    const uint64_t target = (p->total_blocks + want - 1) / (uint64_t)want;
    const int per = (cfg.chunked && cfg.chunk_images > 0) ? cfg.chunk_images : 0;   // caller-chosen chunk length
    Chunk c;
    c.img0 = 0;
    for (int i = 0; i < n; i++) {
        c.blocks += p->imgs[i].n_blocks;
        const bool last = (i == n - 1);
        if (last || (per ? (i + 1 - c.img0 >= per) : (c.blocks >= target && (int)p->chunks.size() < want - 1))) {
            c.img1 = i + 1;
            p->chunks.push_back(c);
            c = Chunk();
            c.img0 = i + 1;
        }
    }
}

// Stage 4, the work of each chunk (never crossing a chunk boundary).
// A run of consecutive work units (restart intervals, sub-sequences) of one owner (image, kernel 1b image).
struct Run { uint32_t owner, first, n, table_set; };

// Runs grouped by table set, batch order kept inside a group.
static void sort_by_table_set(std::vector<Run>& runs)
{
    std::stable_sort(runs.begin(), runs.end(), [](const Run& x, const Run& y) { return x.table_set < y.table_set; });
}

// Packs runs into CTAs of at most `cap` units as segments, a new CTA at every change of table set, so that runs that
// share tables share CTAs.  Work and Seg are the kernel's {first_seg, n_segs, units, table_set} and its segment,
// make_seg(run, first unit of the segment, thread of the CTA that takes it, units).
template <class Work, class Seg, class MakeSeg>
static void pack_ctas(const std::vector<Run>& runs, uint32_t cap, std::vector<Work>& work, std::vector<Seg>& segs,
                      MakeSeg make_seg)
{
    struct { uint32_t first_seg, n_segs, n, table_set; } w = {(uint32_t)segs.size(), 0, 0, 0};
    auto flush = [&]() {
        if (w.n) work.push_back(Work{w.first_seg, w.n_segs, w.n, w.table_set});
        w = {(uint32_t)segs.size(), 0, 0, 0};
    };
    for (const Run& r : runs) {
        if (w.n && w.table_set != r.table_set) flush();
        uint32_t left = r.n, f = r.first;
        while (left) {
            if (w.n == cap) flush();
            w.table_set = r.table_set;
            const uint32_t take = left < (cap - w.n) ? left : (cap - w.n);
            segs.push_back(make_seg(r, f, w.n, take));
            w.n_segs++; w.n += take; f += take; left -= take;
        }
    }
    flush();
}

// The chunk's arena and output ranges, grid bounds and marker-scan slices.
static void chunk_extents(const std::vector<FileRef>& files, BatchPlan* p, Chunk& c)
{
    const int n = (int)p->imgs.size();
    c.arena_lo = ~0ull; c.arena_hi = 0;
    c.rgb_lo = p->out_off[c.img0];
    c.rgb_hi = (c.img1 < n) ? p->out_off[c.img1] : p->rgb_bytes;
    for (int i = c.img0; i < c.img1; i++) {
        const HjdImageDesc& d = p->imgs[i];
        if (files[i].ptr && files[i].size > 0) {
            if (files[i].dev_off < c.arena_lo) c.arena_lo = files[i].dev_off;
            if (files[i].dev_off + (uint64_t)files[i].size > c.arena_hi) c.arena_hi = files[i].dev_off + (uint64_t)files[i].size;
        }
        if (d.n_blocks > c.max_blocks) c.max_blocks = (uint32_t)d.n_blocks;
        if (d.n_mcus > c.max_mcus) c.max_mcus = d.n_mcus;
        if (d.blocks_per_mcu && luma_blocks(d.width, d.height) > c.max_luma) c.max_luma = (uint32_t)luma_blocks(d.width, d.height);
        if (d.width > c.max_w) c.max_w = d.width;
        if (d.height > c.max_h) c.max_h = d.height;
    }
    if (c.arena_lo == ~0ull) c.arena_lo = c.arena_hi = 0;
    // marker-scan slices of long restart-marker scans (kernel 0)
    c.slice0 = (uint32_t)p->slices.size();
    for (int i = c.img0; i < c.img1; i++) {
        const HjdImageDesc& d = p->imgs[i];
        if (d.restart_interval && d.n_intervals > 1 && d.scan_len > HJD_SCAN_SLICE_MIN) {
            const uint64_t total = (uint64_t)d.scan_len + (d.scan_off & 15);
            const uint32_t ns = (uint32_t)((total + HJD_SCAN_SLICE_BYTES - 1) / HJD_SCAN_SLICE_BYTES);
            for (uint32_t k = 0; k < ns; k++) p->slices.push_back(HjdScanSlice{(uint32_t)i, k, ns, 0});
        }
    }
    c.slice1 = (uint32_t)p->slices.size();
}

// Kernel 1a work items: the chunk's restart intervals packed into CTAs.
static void chunk_entropy_work(const PlanConfig& cfg, BatchPlan* p, Chunk& c)
{
    std::vector<Run> runs;
    uint64_t total = 0;
    for (int i = c.img0; i < c.img1; i++) {
        const HjdImageDesc& d = p->imgs[i];
        if (d.n_intervals) runs.push_back(Run{(uint32_t)i, d.interval_base, d.n_intervals, d.table_set});
        total += d.n_intervals;
    }
    sort_by_table_set(runs);
    // Intervals per CTA.  A big chunk fills its CTAs (HJD_ENT_THREADS).  A chunk of only a few waves -- one 1024-image
    // batch cut over 8 GPUs is 0.86 of a wave -- is cut into a whole number of waves of equally loaded CTAs instead:
    // with 510 full CTAs on 592 slots the SMs that got four of them set the time; 592 CTAs of 221 intervals finish
    // in 0.86 of it.  (Below half a wave the CTAs stay full: fewer table loads, and nothing to balance.)
    uint32_t cap = HJD_ENT_THREADS;
    const uint64_t slots = (uint64_t)cfg.sm_count * HJD_ENT_MINBLOCKS;
    const uint64_t full = (total + HJD_ENT_THREADS - 1) / HJD_ENT_THREADS;
    if (2 * full >= slots && full <= 4 * slots) {
        const uint64_t n_ctas = (full + slots - 1) / slots * slots;
        cap = (uint32_t)((total + n_ctas - 1) / n_ctas);
        if (cap > HJD_ENT_THREADS) cap = HJD_ENT_THREADS;
        if (cap < 32) cap = 32;
    }
    c.work0 = (uint32_t)p->work.size();
    pack_ctas(runs, cap, p->work, p->segs, [](const Run& r, uint32_t first, uint32_t tid0, uint32_t take) {
        return HjdEntropySeg{first, tid0, r.owner, take};
    });
    c.work1 = (uint32_t)p->work.size();
}

// Multi-scan work of the chunk (items [w0, w1)): by level (one launch each), then by kind, so that the lanes of a warp
// mostly run the same loop.  A counting sort: a comparison sort of the 30 M items of 1024 1080p files with restart
// markers every 8 blocks took seconds of host time.  The chunk's multi-scan images are zeroed before the first level.
static void chunk_multiscan(BatchPlan* p, Chunk& c, uint32_t w0, uint32_t w1)
{
    std::vector<uint32_t> at(256 * 5 + 1, 0);
    for (uint32_t k = w0; k < w1; k++) {
        const HjdScanDesc& sd = p->scans[p->mswork[k].scan];
        at[sd.level * 5u + sd.kind + 1]++;
    }
    for (size_t q = 1; q < at.size(); q++) at[q] += at[q - 1];
    std::vector<HjdMsWork> sorted(w1 - w0);
    for (uint32_t k = w0; k < w1; k++) {
        const HjdScanDesc& sd = p->scans[p->mswork[k].scan];
        sorted[at[sd.level * 5u + sd.kind]++] = p->mswork[k];
    }
    std::copy(sorted.begin(), sorted.end(), p->mswork.begin() + w0);
    for (uint32_t k = w0; k < w1;) {
        const uint8_t lv = p->scans[p->mswork[k].scan].level;
        uint32_t e = k;
        while (e < w1 && p->scans[p->mswork[e].scan].level == lv) e++;
        c.ms_levels.emplace_back(k, e);
        k = e;
    }
    for (int i = c.img0; i < c.img1; i++) {
        if (!p->ms_image[i] || p->parse_status[i] != HJD_IMG_OK) continue;
        const HjdImageDesc& d = p->imgs[i];
        if (!c.ms_zero.empty() && c.ms_zero.back().first + c.ms_zero.back().second == d.block_base)
            c.ms_zero.back().second += d.n_blocks;
        else
            c.ms_zero.emplace_back(d.block_base, d.n_blocks);
    }
}

// Stage 5: kernel 1b, chunk by chunk (so that restart-free images pipeline like the rest: nothing in it needs the
// host any more).  Index spaces are batch-wide with one spare entry after every chunk.  Inside a chunk the
// images are grouped by table set (batch order kept inside a group) and their sub-sequences packed into
// CTAs as segments, so small restart-free images share CTAs.  Synchronisation kernel: one range per warp;
// longer ranges make the re-decode lists denser, shorter ones give more independent warps: by the amount
// of work in the chunk.
static void plan_selfsync(const PlanConfig& cfg, BatchPlan* p)
{
    size_t k0 = 0;
    uint32_t max_scan = 0;
    for (Chunk& c : p->chunks) {
        c.ss0 = (uint32_t)k0;
        c.sub0 = p->ss_subs;
        c.ck0 = p->ss_chunks;
        while (k0 < p->ss.size() && (int)p->ss[k0].img < c.img1) {
            HjdSsImage& si = p->ss[k0++];
            si.sub_base = p->ss_subs;
            si.chunk_base = p->ss_chunks;
            p->imgs[si.img].sub_base = si.sub_base;
            p->ss_subs += si.n_subs;
            p->ss_chunks += si.n_chunks;
        }
        c.ss1 = (uint32_t)k0;
        c.n_subs = p->ss_subs - c.sub0;
        c.n_ck = p->ss_chunks - c.ck0;
        p->ss_subs += 1;                     // the gaps
        p->ss_chunks += 1;
        if (c.n_ck + 1 > max_scan) max_scan = c.n_ck + 1;
        if (4 * c.n_subs + 2 > max_scan) max_scan = 4 * c.n_subs + 2;

        std::vector<Run> runs;
        for (uint32_t k = c.ss0; k < c.ss1; k++) runs.push_back(Run{k, 0, p->ss[k].n_subs, p->imgs[p->ss[k].img].table_set});
        sort_by_table_set(runs);
        c.sw0 = (uint32_t)p->sswork.size();
        pack_ctas(runs, HJD_SS_THREADS, p->sswork, p->sssegs, [](const Run& r, uint32_t first, uint32_t tid0, uint32_t take) {
            return HjdSsSeg{r.owner, first, tid0, take};
        });
        c.sw1 = c.sf0 = (uint32_t)p->sswork.size();
        c.ss_range = cfg.ss_range_req ? cfg.ss_range_req : c.n_subs >= 400000 ? 256 : c.n_subs >= 150000 ? 128 : 64;
        if (!cfg.ss_range_req && HJD_SS_FIX_MAXR >= 512 && c.n_subs >= 1000000) c.ss_range = 512;
        // synchronisation rounds: one range per warp, up to HJD_SS_FIX_WARPS per CTA
        HjdSsWork w{(uint32_t)p->sssegs.size(), 0, 0, 0};
        auto flush = [&]() {
            if (w.n_subs) p->sswork.push_back(w);
            w = HjdSsWork{(uint32_t)p->sssegs.size(), 0, 0, 0};
        };
        for (const Run& r : runs) {
            for (uint32_t f = 0; f < r.n; f += c.ss_range) {
                if (w.n_segs == HJD_SS_FIX_WARPS || (w.n_segs && w.table_set != r.table_set)) flush();
                w.table_set = r.table_set;
                const uint32_t take = r.n - f < c.ss_range ? r.n - f : c.ss_range;
                p->sssegs.push_back(HjdSsSeg{r.owner, f, 0, take});
                w.n_segs++; w.n_subs += take;
            }
        }
        flush();
        c.sf1 = (uint32_t)p->sswork.size();
    }
    p->ss_tmp_stride = max_scan / 2048 + 8;
}

int hjd_plan_batch(const std::vector<FileRef>& files, const PlanConfig& cfg, BatchPlan* p, std::string* err)
{
    const size_t n = files.size();
    p->imgs.assign(n, HjdImageDesc());
    p->parse_status.assign(n, 0);
    p->host_restart_warn.assign(n, 0);
    p->ms_items.assign(n, 0); p->n_scans.assign(n, 0); p->ms_image.assign(n, 0);
    p->orientation.assign(n, 1);
    std::vector<Lite> lite(n);
    MultiList multi(n);
    int rc = parse_files(files, cfg.flags, lite, multi, err);
    if (rc != HJD_OK) return rc;
    std::vector<uint32_t> ms_w0(n + 1, 0);
    rc = layout_images(files, cfg, lite, multi, p, ms_w0, err);
    if (rc != HJD_OK) return rc;
    plan_staging(cfg, p);
    plan_chunks(cfg, p);
    for (Chunk& c : p->chunks) {
        chunk_extents(files, p, c);
        chunk_orient(cfg, p, c);
        chunk_entropy_work(cfg, p, c);
        chunk_multiscan(p, c, ms_w0[(size_t)c.img0], ms_w0[(size_t)c.img1]);
    }
    plan_selfsync(cfg, p);
    return HJD_OK;
}
