// tests/plan_driver.cpp -- runs the batch planner (csrc/batch_plan.cpp) on files and prints the plan as JSON.
// Built by tests/test_batch_plan.py with g++ alone: no CUDA header or library, so it also shows the planner needs none.
//
//   plan_driver FLAGS OVERLAP CHUNK_IMAGES CHUNKED REPEAT FILE...
//
// The files, in order, repeated REPEAT times (one buffer per file, shared by its repeats), get arena offsets as
// hjd_batch_upload gives them: each file at the next 16-byte boundary.
#include "../hls_jpeg_decoder_b200/csrc/batch_plan.h"

#include <stdio.h>
#include <stdlib.h>
#include <vector>

template <class T, class F>
static void array(const char* name, const std::vector<T>& v, F row)
{
    printf(",\n\"%s\": [", name);
    for (size_t k = 0; k < v.size(); k++) { printf(k ? ",\n [" : "\n ["); row(v[k]); printf("]"); }
    printf("]");
}

int main(int argc, char** argv)
{
    if (argc < 6) { fprintf(stderr, "usage: %s FLAGS OVERLAP CHUNK_IMAGES CHUNKED REPEAT FILE...\n", argv[0]); return 2; }
    PlanConfig cfg;
    cfg.flags = (unsigned)strtoul(argv[1], nullptr, 0);
    cfg.overlap = atoi(argv[2]);
    cfg.chunk_images = atoi(argv[3]);
    cfg.chunked = atoi(argv[4]) != 0;
    const int repeat = atoi(argv[5]);
    std::vector<std::vector<uint8_t>> bufs;
    for (int a = 6; a < argc; a++) {
        FILE* fp = fopen(argv[a], "rb");
        if (!fp) { perror(argv[a]); return 2; }
        fseek(fp, 0, SEEK_END);
        std::vector<uint8_t> b((size_t)ftell(fp));
        fseek(fp, 0, SEEK_SET);
        if (fread(b.data(), 1, b.size(), fp) != b.size()) { perror(argv[a]); return 2; }
        fclose(fp);
        bufs.push_back(std::move(b));
    }
    std::vector<FileRef> files;
    uint64_t off = 0;
    for (int r = 0; r < repeat; r++)
        for (const auto& b : bufs) {
            files.push_back(FileRef{b.data(), (int64_t)b.size(), off});
            off += align_up(b.size(), 16);
        }

    BatchPlan p;
    std::string err;
    const int rc = hjd_plan_batch(files, cfg, &p, &err);
    printf("{\"rc\": %d, \"err\": \"%s\", \"ent_threads\": %d, \"ss_threads\": %d, \"ss_fix_warps\": %d", rc, err.c_str(),
           HJD_ENT_THREADS, HJD_SS_THREADS, HJD_SS_FIX_WARPS);
    if (rc != HJD_OK) { printf("}\n"); return 0; }
    size_t i = 0;
    array("images", p.imgs, [&](const HjdImageDesc& d) {
        printf("%d, %u, %u, %u, %u, %u, %u, %u, %u, %u, %u, %u, %u, %u, %llu, %llu, %u, %u, %u, %u", p.parse_status[i],
               d.width, d.height, d.ncomp, d.hf, d.vf, d.blocks_per_mcu, d.mcus_x, d.mcus_y, d.restart_interval,
               d.n_intervals, d.interval_base, d.scan_len, d.table_set, (unsigned long long)d.block_base,
               (unsigned long long)d.n_blocks, d.n_subs, p.ms_items[i], p.n_scans[i], p.ms_image[i]);
        i++;
    });
    array("chunks", p.chunks, [](const Chunk& c) {
        printf("%d, %d, %u, %u, %u, %u, %u, %u, %u, %u, [", c.img0, c.img1, c.work0, c.work1, c.ss0, c.ss1, c.sw0, c.sw1,
               c.sf0, c.sf1);
        for (size_t k = 0; k < c.ms_levels.size(); k++) printf("%s[%u, %u]", k ? ", " : "", c.ms_levels[k].first, c.ms_levels[k].second);
        printf("]");
    });
    array("work", p.work, [](const HjdEntropyWork& w) { printf("%u, %u, %u, %u", w.first_seg, w.n_segs, w.n_intervals, w.table_set); });
    array("segs", p.segs, [](const HjdEntropySeg& s) { printf("%u, %u, %u, %u", s.first_interval, s.tid0, s.image, s.n); });
    array("ss", p.ss, [](const HjdSsImage& s) { printf("%u, %u, %u", s.img, s.sub_base, s.n_subs); });
    array("sswork", p.sswork, [](const HjdSsWork& w) { printf("%u, %u, %u, %u", w.first_seg, w.n_segs, w.n_subs, w.table_set); });
    array("sssegs", p.sssegs, [](const HjdSsSeg& s) { printf("%u, %u, %u, %u", s.ss, s.first_sub, s.tid0, s.n); });
    array("scans", p.scans, [](const HjdScanDesc& s) { printf("%u, %u, %u", s.image, s.level, s.n_intervals); });
    array("mswork", p.mswork, [](const HjdMsWork& w) { printf("%u, %u", w.scan, w.interval); });
    printf("}\n");
    return 0;
}
