// gseg_cli.cpp -- C++ host program over the C-ABI of include/gseg.h.
//
// Mirrors the command line of the reference's executables as far as it is known: the report's CPU
// baseline is Felzenszwalb's `segment sigma k min input(ppm) output(ppm)` (Report.pdf p4 "Baseline",
// ref [23]); the GPU branches take the same parameters plus the hierarchy level (BASELINE.json
// north_star) and time 20 iterations excluding disk I/O (Report.pdf p4 s4.1).  No compute happens in
// this file: it parses arguments, reads/writes PPM and calls libgseg.so.
//
//   gseg [options] sigma k min_size input output
//     input: binary PPM/PGM, PNG or JPEG (by content; JPEG is decoded on the GPU through
//     gseg_segment_jpeg / nvJPEG); output: PNG if the name ends in .png, else PPM
//     (gseg_imageio.hpp; the GPU branches read through cv::imread, SURVEY.md s8(f) N1)
//     --variant felz|hier|superpix   reference branch semantics (default felz)
//     --conn 4|8                     grid connectivity (default 8, as in `segment`)
//     --level L                      hierarchy level to write (hier/superpix; default last)
//     --labels FILE                  also write the label image as raw little-endian int32, row-major
//     --regions FILE                 also write the region table (gseg_regions: 8 little-endian uint64 per component)
//     --render random|mean|overlay   output picture: random colour per component (default), each region's mean colour,
//                                    or the input with the region boundaries in red (gseg_render)
//     --synth WxH:SEED               ignore input.ppm, segment the deterministic synthetic image
//     --iters N                      timing loop: N runs after 2 warm-ups, mean +- std (excludes I/O)
//     --device D                     CUDA device ordinal
//     --host-loop                    host-driven schedule (one read-back per round, the reference's "conventional" driver)
//     --tail E,V                     largest round (edges, components) the single-cluster tail kernel takes; 0,0 = never
//   gseg --batch IN_DIR OUT_DIR [options] sigma k min_size
//     every image file of IN_DIR (PPM/PGM/PNG, or JPEG decoded on the GPU) through the batch pipeline gseg_pool_*
//     (--contexts S contexts in flight, default 8); writes OUT_DIR/<name>.png (random colours per component, same
//     colours as the single-image mode) and prints one "name: got N components" line per image plus the throughput;
//     --render mean: the jobs return the region table with the labels (GSEG_OUT_REGIONS) and the mean-colour picture is
//     painted on the host from it, without a second pass on the device
//   gseg --convert input output      file conversion only (no GPU): exercises the readers/writers
#include <dirent.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "gseg.h"
#include "gseg_imageio.hpp"

// The colour k_colorize gives a label (counter-based hash: SplitMix64 twice), for label images that come back from the pool.
static inline uint64_t sm64(uint64_t x) {
    uint64_t z = x + 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
static inline void label_colour(uint64_t seed, uint32_t label, uint8_t *rgb) {
    const uint64_t h = sm64(sm64(seed ^ ((uint64_t)label * 0xD6E8FEB86659FD93ull)) + 3);
    rgb[0] = (uint8_t)(h & 255); rgb[1] = (uint8_t)((h >> 8) & 255); rgb[2] = (uint8_t)((h >> 16) & 255);
}
// Rounded mean colour of record c of a region table: (sum + count / 2) / count, as gseg_render(GSEG_RENDER_MEAN).
static inline void mean_colour(const uint64_t *table, uint32_t c, uint8_t *rgb) {
    const uint64_t *t = table + 8 * (size_t)c, n = t[0] ? t[0] : 1;
    for (int k = 0; k < 3; ++k) rgb[k] = (uint8_t)((t[1 + k] + n / 2) / n);
}

#define RENDER_RANDOM (-1)

// gseg --batch IN_DIR OUT_DIR: the reference's loop over a directory of images, through the batch pipeline.
static int run_batch(const char *in_dir, const char *out_dir, const gseg_params &p, int level, int device, int contexts, int render) {
    std::vector<std::string> names;
    if (DIR *d = opendir(in_dir)) {
        while (dirent *e = readdir(d)) {
            const std::string n = e->d_name;
            const size_t dot = n.rfind('.');
            if (dot == std::string::npos) continue;
            std::string ext = n.substr(dot + 1);
            std::transform(ext.begin(), ext.end(), ext.begin(), [](unsigned char c) { return (char)tolower(c); });
            if (ext == "ppm" || ext == "pgm" || ext == "png" || ext == "jpg" || ext == "jpeg") names.push_back(n);
        }
        closedir(d);
    } else { fprintf(stderr, "gseg: cannot open directory %s\n", in_dir); return 1; }
    std::sort(names.begin(), names.end());
    if (names.empty()) { fprintf(stderr, "gseg: no image files in %s\n", in_dir); return 1; }
    struct Item { std::vector<uint8_t> px, jpeg; int w = 0, h = 0; };
    std::vector<Item> items(names.size());
    int max_w = 0, max_h = 0;
    for (size_t i = 0; i < names.size(); ++i) {
        const std::string path = std::string(in_dir) + "/" + names[i];
        std::vector<uint8_t> raw;
        std::string err;
        Item &it = items[i];
        if (gsegio::read_file(path.c_str(), raw) && raw.size() > 2 && raw[0] == 0xFF && raw[1] == 0xD8) {
            const int rc = gseg_jpeg_info(raw.data(), raw.size(), &it.w, &it.h);
            if (rc) { fprintf(stderr, "gseg: cannot read JPEG %s: %s\n", path.c_str(), gseg_strerror(rc)); return 1; }
            it.jpeg.swap(raw);
        } else if (!gsegio::read_image(path.c_str(), it.px, it.w, it.h, err)) {
            fprintf(stderr, "gseg: cannot read %s: %s\n", path.c_str(), err.c_str());
            return 1;
        }
        max_w = std::max(max_w, it.w); max_h = std::max(max_h, it.h);
    }
    // every context is sized for the largest image (width and height taken separately, so any of them fits)
    gseg_pool *pool = nullptr;
    int rc = gseg_pool_create(&pool, device, max_w, max_h, p.connectivity, contexts, p.variant == GSEG_SUPERPIX ? GSEG_CAP_SUPERPIX : 0u);
    if (rc) { fprintf(stderr, "gseg: gseg_pool_create: %s\n", gseg_strerror(rc)); return 1; }
    const size_t n = items.size();
    std::vector<gseg_pool_job> jobs(n);
    std::vector<gseg_pool_result> res(n);
    std::vector<void *> pinned;
    for (size_t i = 0; i < n; ++i) {
        Item &it = items[i];
        gseg_pool_job &j = jobs[i];
        memset(&j, 0, sizeof j);
        const size_t V = (size_t)it.w * it.h;
        if (!it.jpeg.empty()) { j.input = it.jpeg.data(); j.jpeg_bytes = it.jpeg.size(); }
        else {
            void *in = gseg_host_alloc(V * 3);
            if (!in) { fprintf(stderr, "gseg: pinned allocation failed\n"); return 1; }
            memcpy(in, it.px.data(), V * 3);
            pinned.push_back(in);
            j.input = in;
        }
        j.w = it.w; j.h = it.h; j.stride_bytes = 3 * it.w; j.mem_kind = GSEG_MEM_HOST; j.params = p;
        j.out_mode = GSEG_OUT_LABELS; j.level = p.variant == GSEG_FELZ ? -1 : level; j.elem_bytes = 4; j.out_mem_kind = GSEG_MEM_HOST;
        j.out_capacity = V * 4;
        if (render == GSEG_RENDER_MEAN) { // labels, then the table at the next 64-byte boundary; a FELZ component has >= min_size pixels
            const size_t ncap = p.variant == GSEG_FELZ && p.min_size > 1 ? (V + p.min_size - 1) / p.min_size : V;
            j.out_mode = GSEG_OUT_REGIONS;
            j.out_capacity = ((V * 4 + 63) & ~(size_t)63) + 64 * ncap;
        }
        j.out = gseg_host_alloc(j.out_capacity);
        if (!j.out) { fprintf(stderr, "gseg: pinned allocation failed\n"); return 1; }
        pinned.push_back(j.out);
    }
    const auto t0 = std::chrono::steady_clock::now();
    rc = gseg_pool_run(pool, jobs.data(), (int)n, res.data());
    const double ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    if (rc) { fprintf(stderr, "gseg: gseg_pool_run: %s (%s)\n", gseg_strerror(rc), gseg_pool_last_error(pool)); return 1; }
    double mpix = 0;
    for (size_t i = 0; i < n; ++i) {
        const size_t V = (size_t)res[i].w * res[i].h;
        mpix += V / 1e6;
        std::vector<uint8_t> out(V * 3);
        const int32_t *lab = (const int32_t *)jobs[i].out;
        if (render == GSEG_RENDER_MEAN) {
            const uint64_t *table = (const uint64_t *)((const uint8_t *)jobs[i].out + res[i].offsets[1]);
            for (size_t q = 0; q < V; ++q) mean_colour(table, (uint32_t)lab[q], &out[3 * q]);
        } else {
            for (size_t q = 0; q < V; ++q) label_colour(1, (uint32_t)lab[q], &out[3 * q]);
        }
        const std::string stem = names[i].substr(0, names[i].rfind('.'));
        const std::string path = std::string(out_dir) + "/" + stem + ".png";
        if (!gsegio::write_image(path.c_str(), out.data(), res[i].w, res[i].h)) { fprintf(stderr, "gseg: cannot write %s\n", path.c_str()); return 1; }
        printf("%s: got %d components\n", names[i].c_str(), res[i].n_components);
    }
    printf("batch of %zu images, %d contexts: %.3f ms (H2D and D2H included, disk excluded) = %.1f Mpixel/s\n", n, contexts, ms, mpix / (ms / 1e3));
    gseg_pool_destroy(pool);
    for (void *q : pinned) gseg_host_free(q);
    return 0;
}

static int usage() {
    fprintf(stderr,
            "usage: gseg [--variant felz|hier|superpix] [--conn 4|8] [--level L] [--labels FILE] [--regions FILE]\n"
            "            [--render random|mean|overlay] [--synth WxH:SEED] [--iters N] [--device D] [--host-loop] [--tail E,V]\n"
            "            sigma k min_size input.{ppm,pgm,png,jpg} output.{ppm,png}\n"
            "       gseg --batch IN_DIR OUT_DIR [--contexts S] [--variant ...] [--conn 4|8] [--level L] [--render random|mean]\n"
            "            [--device D] sigma k min_size\n"
            "       gseg --convert input output\n");
    return 2;
}

int main(int argc, char **argv) {
    if (argc == 4 && !strcmp(argv[1], "--convert")) {
        std::vector<uint8_t> px;
        int cw = 0, ch = 0;
        std::string err;
        if (!gsegio::read_image(argv[2], px, cw, ch, err)) { fprintf(stderr, "gseg: %s: %s\n", argv[2], err.c_str()); return 1; }
        if (!gsegio::write_image(argv[3], px.data(), cw, ch)) { fprintf(stderr, "gseg: cannot write %s\n", argv[3]); return 1; }
        printf("%dx%d\n", cw, ch);
        return 0;
    }
    gseg_params p;
    memset(&p, 0, sizeof p);
    p.connectivity = 8;
    p.variant = GSEG_FELZ;
    int level = -1, iters = 0, device = 0, sw = 0, sh = 0;
    long long tail_e = -1, tail_v = -1;
    int contexts = 8;
    const char *batch_in = nullptr, *batch_out = nullptr;
    unsigned long long sseed = 0;
    const char *labels_path = nullptr, *regions_path = nullptr;
    int render = RENDER_RANDOM;
    std::vector<const char *> pos;
    for (int i = 1; i < argc; ++i) {
        std::string a = argv[i];
        auto need = [&](const char *name) -> const char * {
            if (i + 1 >= argc) { fprintf(stderr, "gseg: %s needs a value\n", name); exit(2); }
            return argv[++i];
        };
        if (a == "--variant") {
            std::string v = need("--variant");
            if (v == "felz") p.variant = GSEG_FELZ;
            else if (v == "hier") p.variant = GSEG_HIER;
            else if (v == "superpix") p.variant = GSEG_SUPERPIX;
            else return usage();
        } else if (a == "--conn") p.connectivity = atoi(need("--conn"));
        else if (a == "--level") level = atoi(need("--level"));
        else if (a == "--labels") labels_path = need("--labels");
        else if (a == "--regions") regions_path = need("--regions");
        else if (a == "--render") {
            std::string v = need("--render");
            if (v == "random") render = RENDER_RANDOM;
            else if (v == "mean") render = GSEG_RENDER_MEAN;
            else if (v == "overlay") render = GSEG_RENDER_OVERLAY;
            else return usage();
        }
        else if (a == "--iters") iters = atoi(need("--iters"));
        else if (a == "--device") device = atoi(need("--device"));
        else if (a == "--host-loop") p.flags |= GSEG_FLAG_HOST_LOOP;
        else if (a == "--contexts") contexts = atoi(need("--contexts"));
        else if (a == "--batch") { batch_in = need("--batch"); batch_out = need("--batch"); }
        else if (a == "--tail") { if (sscanf(need("--tail"), "%lld,%lld", &tail_e, &tail_v) != 2 || tail_e < 0 || tail_v < 0) return usage(); }
        else if (a == "--synth") {
            if (sscanf(need("--synth"), "%dx%d:%llu", &sw, &sh, &sseed) != 3 || sw < 1 || sh < 1) return usage();
        } else if (a.size() > 2 && a[0] == '-' && a[1] == '-') return usage();
        else pos.push_back(argv[i]);
    }
    if (batch_in) {
        if (pos.size() != 3 || contexts < 1 || contexts > 64 || render == GSEG_RENDER_OVERLAY || regions_path) return usage();
        p.sigma = (float)atof(pos[0]); p.k = (float)atof(pos[1]); p.min_size = atoi(pos[2]);
        return run_batch(batch_in, batch_out, p, level, device, contexts, render);
    }
    if (pos.size() != 5) return usage();
    p.sigma = (float)atof(pos[0]);
    p.k = (float)atof(pos[1]);
    p.min_size = atoi(pos[2]);
    const char *in_path = pos[3], *out_path = pos[4];

    std::vector<uint8_t> img;
    int w = sw, h = sh;
    std::string ioerr;
    std::vector<uint8_t> jpeg; // JPEG input: decoded on the GPU by gseg_segment_jpeg (nvJPEG), not by this program
    if (!sw) {
        std::vector<uint8_t> raw;
        if (gsegio::read_file(in_path, raw) && raw.size() > 2 && raw[0] == 0xFF && raw[1] == 0xD8) {
            const int jrc = gseg_jpeg_info(raw.data(), raw.size(), &w, &h);
            if (jrc) { fprintf(stderr, "gseg: cannot read JPEG %s: %s\n", in_path, gseg_strerror(jrc)); return 1; }
            jpeg.swap(raw);
        } else if (!gsegio::read_image(in_path, img, w, h, ioerr)) {
            fprintf(stderr, "gseg: cannot read %s: %s\n", in_path, ioerr.c_str());
            return 1;
        }
    }
    gseg_ctx *ctx = nullptr;
    int rc = gseg_create(&ctx, device, w, h);
    if (rc) { fprintf(stderr, "gseg: gseg_create: %s\n", gseg_strerror(rc)); return 1; }
    if (tail_e >= 0) gseg_set_tail(ctx, (uint32_t)tail_e, (uint32_t)tail_v);
    if (!jpeg.empty()) { // first run straight from the compressed bytes; the decoded pixels come back for the timing loop
        rc = gseg_segment_jpeg(ctx, jpeg.data(), jpeg.size(), &p, &w, &h);
        if (rc) { fprintf(stderr, "gseg: gseg_segment_jpeg: %s (%s)\n", gseg_strerror(rc), gseg_last_error(ctx)); return 1; }
        img.resize((size_t)w * h * 3);
        rc = gseg_input_rgb(ctx, img.data(), GSEG_MEM_HOST);
        if (rc) { fprintf(stderr, "gseg: gseg_input_rgb: %s\n", gseg_strerror(rc)); return 1; }
    }
    if (sw) {
        img.resize((size_t)w * h * 3);
        rc = gseg_synth(ctx, img.data(), w, h, sseed, GSEG_MEM_HOST);
        if (rc) { fprintf(stderr, "gseg: gseg_synth: %s\n", gseg_strerror(rc)); return 1; }
    }
    auto run = [&]() { return gseg_segment(ctx, img.data(), w, h, 3 * w, GSEG_MEM_HOST, &p); };
    rc = run();
    if (rc) { fprintf(stderr, "gseg: gseg_segment: %s (%s)\n", gseg_strerror(rc), gseg_last_error(ctx)); return 1; }
    if (iters > 0) { // the reference's timing loop: same input, disk I/O excluded (Report.pdf p4 s4.1)
        run();
        std::vector<double> ms;
        for (int i = 0; i < iters; ++i) {
            const auto t0 = std::chrono::steady_clock::now();
            rc = run();
            const auto t1 = std::chrono::steady_clock::now();
            if (rc) { fprintf(stderr, "gseg: gseg_segment: %s\n", gseg_strerror(rc)); return 1; }
            ms.push_back(std::chrono::duration<double, std::milli>(t1 - t0).count());
        }
        double mean = 0, var = 0;
        for (double v : ms) mean += v;
        mean /= ms.size();
        for (double v : ms) var += (v - mean) * (v - mean);
        printf("time_ms mean %.4f std %.4f over %d runs (%dx%d, H2D copy included) = %.1f Mpixel/s\n", mean,
               std::sqrt(var / ms.size()), iters, w, h, (double)w * h / 1e3 / mean);
    }
    const int nlev = gseg_num_levels(ctx);
    if (p.variant != GSEG_FELZ && level >= nlev) {
        fprintf(stderr, "gseg: level %d out of range, %d levels produced\n", level, nlev);
        return 1;
    }
    const int ncomp = gseg_num_components(ctx, p.variant == GSEG_FELZ ? -1 : level);
    std::vector<uint8_t> out((size_t)w * h * 3);
    const int olevel = p.variant == GSEG_FELZ ? -1 : level;
    if (render == RENDER_RANDOM) {
        rc = gseg_colorize(ctx, olevel, 1, out.data(), GSEG_MEM_HOST);
        if (rc) { fprintf(stderr, "gseg: gseg_colorize: %s\n", gseg_strerror(rc)); return 1; }
    } else { // the input the context staged (the last gseg_segment read host memory)
        rc = gseg_render(ctx, olevel, render, 0xFF0000u, nullptr, 0, GSEG_MEM_HOST, out.data(), GSEG_MEM_HOST);
        if (rc) { fprintf(stderr, "gseg: gseg_render: %s (%s)\n", gseg_strerror(rc), gseg_last_error(ctx)); return 1; }
    }
    if (!gsegio::write_image(out_path, out.data(), w, h)) { fprintf(stderr, "gseg: cannot write %s\n", out_path); return 1; }
    if (labels_path) {
        std::vector<int32_t> lab((size_t)w * h);
        rc = gseg_labels(ctx, p.variant == GSEG_FELZ ? -1 : level, lab.data(), GSEG_MEM_HOST);
        if (rc) { fprintf(stderr, "gseg: gseg_labels: %s\n", gseg_strerror(rc)); return 1; }
        FILE *f = fopen(labels_path, "wb");
        if (!f || fwrite(lab.data(), sizeof(int32_t), lab.size(), f) != lab.size()) {
            fprintf(stderr, "gseg: cannot write %s\n", labels_path);
            return 1;
        }
        fclose(f);
    }
    if (regions_path) {
        std::vector<uint64_t> table((size_t)ncomp * 8);
        rc = gseg_regions(ctx, olevel, nullptr, 0, GSEG_MEM_HOST, table.data(), ncomp, GSEG_MEM_HOST);
        if (rc < 0) { fprintf(stderr, "gseg: gseg_regions: %s (%s)\n", gseg_strerror(rc), gseg_last_error(ctx)); return 1; }
        FILE *f = fopen(regions_path, "wb");
        if (!f || fwrite(table.data(), sizeof(uint64_t), table.size(), f) != table.size()) {
            fprintf(stderr, "gseg: cannot write %s\n", regions_path);
            return 1;
        }
        fclose(f);
    }
    printf("got %d components", ncomp); // `segment` prints "got %d components"
    if (p.variant != GSEG_FELZ) printf(" at level %d of %d", level < 0 ? nlev - 1 : level, nlev);
    printf("\n");
    gseg_destroy(ctx);
    return 0;
}
