// tests/orient_driver.cpp -- the host side of HJD_FLAG_EXIF_ORIENT without a GPU: the batch plan's staging and
// orientation jobs as JSON, and a seeded mutation fuzz of the Exif APP1 parse.  Built by tests/test_orient_host.py with
// g++ alone (and -fsanitize=address,undefined).
//
//   orient_driver plan FLAGS OVERLAP CHUNK_IMAGES CHUNKED FILE...
//   orient_driver fuzz SEED COUNT FILE      FILE: a JPEG whose first segment after SOI is an Exif APP1
//
// fuzz mutates the APP1 payload COUNT times (bytes, 16- and 32-bit fields set to extremes, truncation with the segment
// length rewritten), and runs both marker walks on each file and hjd_exif_orientation on the payload, each input in a
// heap buffer of exactly its size so that the sanitizer sees any read past it.  It prints a histogram of the results.
#include "../hls_jpeg_decoder_b200/csrc/batch_plan.h"

#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <memory>
#include <random>
#include <vector>

static std::vector<uint8_t> read_file(const char* path)
{
    FILE* fp = fopen(path, "rb");
    if (!fp) { perror(path); exit(2); }
    fseek(fp, 0, SEEK_END);
    std::vector<uint8_t> b((size_t)ftell(fp));
    fseek(fp, 0, SEEK_SET);
    if (fread(b.data(), 1, b.size(), fp) != b.size()) { perror(path); exit(2); }
    fclose(fp);
    return b;
}

static int plan(int argc, char** argv)
{
    PlanConfig cfg;
    cfg.flags = (unsigned)strtoul(argv[2], nullptr, 0);
    cfg.overlap = atoi(argv[3]);
    cfg.chunk_images = atoi(argv[4]);
    cfg.chunked = atoi(argv[5]) != 0;
    std::vector<std::vector<uint8_t>> bufs;
    for (int a = 6; a < argc; a++) bufs.push_back(read_file(argv[a]));
    std::vector<FileRef> files;
    uint64_t off = 0;
    for (const auto& b : bufs) {
        files.push_back(FileRef{b.data(), (int64_t)b.size(), off});
        off += align_up(b.size(), 16);
    }
    BatchPlan p;
    std::string err;
    const int rc = hjd_plan_batch(files, cfg, &p, &err);
    printf("{\"rc\": %d, \"rgb_bytes\": %llu, \"stage_bytes\": %llu", rc, (unsigned long long)p.rgb_bytes,
           (unsigned long long)p.stage_bytes);
    if (rc == HJD_OK) {
        printf(",\n\"images\": [");      // status, orientation, rgb_off (kernels), out_off (host), out_w, out_h, out bytes
        for (size_t i = 0; i < p.imgs.size(); i++) {
            const HjdImageDesc& d = p.imgs[i];
            uint32_t w, h;
            out_size(cfg.flags, d.width, d.height, p.orientation[i], &w, &h);
            printf("%s[%d, %d, %llu, %llu, %u, %u, %llu]", i ? ",\n " : "\n ", p.parse_status[i], p.orientation[i],
                   (unsigned long long)d.rgb_off, (unsigned long long)p.out_off[i], w, h,
                   (unsigned long long)(d.blocks_per_mcu ? image_out_bytes(cfg.flags, d.width, d.height) : 0));
        }
        printf("],\n\"chunks\": [");     // img0, img1, rgb_lo, rgb_hi, oj0, oj1
        for (size_t k = 0; k < p.chunks.size(); k++) {
            const Chunk& c = p.chunks[k];
            printf("%s[%d, %d, %llu, %llu, %u, %u]", k ? ", " : "", c.img0, c.img1, (unsigned long long)c.rgb_lo,
                   (unsigned long long)c.rgb_hi, c.oj0, c.oj1);
        }
        printf("],\n\"jobs\": [");       // src_off, dst_off, w, h, o
        for (size_t k = 0; k < p.orient_jobs.size(); k++) {
            const HjdOrientJob& j = p.orient_jobs[k];
            printf("%s[%llu, %llu, %u, %u, %u]", k ? ",\n " : "\n ", (unsigned long long)j.src_off,
                   (unsigned long long)j.dst_off, j.w, j.h, j.o);
        }
        printf("],\n\"tiles\": [");
        for (size_t k = 0; k < p.orient_tiles.size(); k++) printf("%s%u", k ? ", " : "", p.orient_tiles[k]);
        printf("], \"tile\": %d", HJD_ORIENT_TILE);
    }
    printf("}\n");
    return 0;
}

static int fuzz(char** argv)
{
    std::mt19937_64 rng(strtoull(argv[2], nullptr, 0));
    const long count = atol(argv[3]);
    const std::vector<uint8_t> base = read_file(argv[4]);
    if (base.size() < 6 || base[2] != 0xFF || base[3] != 0xE1) { fprintf(stderr, "no APP1 after SOI\n"); return 2; }
    const size_t seg_len = (size_t)base[4] << 8 | base[5];
    const std::vector<uint8_t> payload(base.begin() + 6, base.begin() + 4 + seg_len);
    const std::vector<uint8_t> rest(base.begin() + 4 + seg_len, base.end());
    long hist[10] = {0};          // [0]: not Exif (direct call), [1..8], [9]: out of range
    long parse_hist[9] = {0};
    auto pick = [&](size_t n) { return n ? (size_t)(rng() % n) : 0; };
    for (long it = 0; it < count; it++) {
        std::vector<uint8_t> m = payload;
        const int n_mut = 1 + (int)(rng() % 6);
        for (int k = 0; k < n_mut; k++) {
            const int kind = (int)(rng() % 6);
            // most mutations hit the TIFF header and IFD0, where every offset and count lives
            const size_t at = (rng() % 4) ? pick(m.size() < 64 ? m.size() : 64) : pick(m.size());
            if (m.empty()) break;
            if (kind == 0) m[at] = (uint8_t)rng();
            else if (kind == 1) m[at] ^= (uint8_t)(1u << (rng() % 8));
            else if (kind == 2 && at + 1 < m.size()) { const uint8_t v = (rng() & 1) ? 0xFF : 0x00; m[at] = v; m[at + 1] = (rng() & 1) ? v : 0xFE; }
            else if (kind == 3 && at + 3 < m.size()) {
                const uint32_t vals[] = {0xFFFFFFFFu, 0x7FFFFFFFu, 0x80000000u, (uint32_t)m.size(), (uint32_t)m.size() - 6,
                                         (uint32_t)m.size() - 7, (uint32_t)m.size() - 8, 0u};
                const uint32_t v = vals[rng() % 8];
                for (int q = 0; q < 4; q++) m[at + q] = (uint8_t)(v >> ((rng() & 1) ? 8 * q : 24 - 8 * q));
            } else if (kind == 4) m.resize(pick(m.size() + 1));
            else if (kind == 5 && at + 1 < m.size()) { m[at] = (rng() & 1) ? 0x01 : 0x12; m[at + 1] = (rng() & 1) ? 0x12 : 0x01; }
        }
        {
            std::unique_ptr<uint8_t[]> buf(new uint8_t[m.size() ? m.size() : 1]);
            if (!m.empty()) memcpy(buf.get(), m.data(), m.size());
            const int v = hjd_exif_orientation(buf.get(), m.size());
            hist[v >= 0 && v <= 8 ? v : 9]++;
        }
        std::vector<uint8_t> f = {0xFF, 0xD8, 0xFF, 0xE1, (uint8_t)((m.size() + 2) >> 8), (uint8_t)(m.size() + 2)};
        f.insert(f.end(), m.begin(), m.end());
        f.insert(f.end(), rest.begin(), rest.end());
        std::unique_ptr<uint8_t[]> fb(new uint8_t[f.size()]);
        memcpy(fb.get(), f.data(), f.size());
        HjdParsed ps;
        hjd_parse_jpeg(fb.get(), f.size(), &ps);
        HjdMultiParsed mp;
        hjd_parse_jpeg_multi(fb.get(), f.size(), &mp);
        const int a = ps.orientation, b = mp.frame.orientation;
        parse_hist[a >= 1 && a <= 8 && a == b ? a : 0]++;
    }
    printf("{\"direct\": [");
    for (int k = 0; k < 10; k++) printf("%s%ld", k ? ", " : "", hist[k]);
    printf("], \"parsed\": [");
    for (int k = 0; k < 9; k++) printf("%s%ld", k ? ", " : "", parse_hist[k]);
    printf("]}\n");
    return 0;
}

int main(int argc, char** argv)
{
    if (argc >= 6 && !strcmp(argv[1], "plan")) return plan(argc, argv);
    if (argc == 5 && !strcmp(argv[1], "fuzz")) return fuzz(argv);
    fprintf(stderr, "usage: %s plan FLAGS OVERLAP CHUNK_IMAGES CHUNKED FILE... | fuzz SEED COUNT FILE\n", argv[0]);
    return 2;
}
