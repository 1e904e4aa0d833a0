// Headless front end of the SHARDED offline job over the C ABI (include/vstab.h): the reference's --file loop
// (/root/reference/src/main.cpp:196-236, src/main_utils.cpp:397-417, :459-493) for a clip that is split over GPUs by
// contiguous frame ranges -- one process per GPU, every process runs this program with its own --rank.
//
//   vstab_offline --file in.bgr --width 1920 --height 1080 --out out.bgr
//                 [--past-window 60] [--future-window 45] [--working-height 360] [--batch 128]
//                 [--mode global|lock|orb|sift] [--mode-at CALL] [--frames N]
//                 [--rank R --world S --id-file PATH] [--device D] [--checksums FILE]
//
// Every rank reads ITS frames [first, last) (and the halo frame first-1) of the raw BGR24 clip into pinned host memory, calls
// vstab_offline_run once (estimation -> ncclAllGather of the 3x3 transforms inside the library -> smoothing / lock -> warp)
// and writes the outputs of ITS calls [call_first, call_last) at their offsets of the raw BGR24 output file, so the ranks
// together produce the file the single-process streaming front end (examples/vstab_file.cpp) writes.
// The 128-byte NCCL id travels through --id-file: rank 0 writes it, the other ranks wait for it (any shared path will do;
// a launcher with its own transport -- MPI, torchrun -- would pass the bytes itself).  --world 1 needs no id.
// --checksums writes "call checksum" lines (the 64-bit per-frame checksum the warp kernel fuses, vstab_frame_checksum).
// Exit status: 0 ok, 1 bad usage, 2 I/O, 3 stabilizer error.
#include <chrono>
#include <cstdio>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>

#include "vstab.h"

namespace {

struct Options {
    std::string in, out, id_file, checksums;
    int width = 0, height = 0, working_height = 360, batch = 128, rank = 0, world = 1, device = -1;
    long frames = -1, mode_at = 0, past = 60, future = 45;        // 2.0 s / 1.5 s at 30 fps (src/main.cpp:205-206)
    int mode = VSTAB_GLOBAL_SMOOTHING;
    double crop = 1.0, crop_release = 0.002;                      // auto-crop (1: off)
};

bool parse_mode(const std::string& s, int& m) {
    if (s == "global") m = VSTAB_GLOBAL_SMOOTHING;
    else if (s == "lock") m = VSTAB_ACCUMULATED_FULL_LOCK;
    else if (s == "orb") m = VSTAB_ORB_FULL_LOCK;
    else if (s == "sift") m = VSTAB_SIFT_FULL_LOCK;
    else return false;
    return true;
}

// --crop MAX_ZOOM[,RELEASE]: 1 < MAX_ZOOM <= 4, RELEASE > 0 (default 0.002 per call), ceil((MAX_ZOOM - 1) / RELEASE) <= 4096
bool parse_crop(const std::string& s, double& max_zoom, double& release) {
    const size_t comma = s.find(',');
    const std::string a = s.substr(0, comma), b = comma == std::string::npos ? "" : s.substr(comma + 1);
    if (a.empty() || (comma != std::string::npos && b.empty())) return false;
    char* end = nullptr;
    max_zoom = std::strtod(a.c_str(), &end);
    if (*end) return false;
    release = 0.002;
    if (!b.empty()) { release = std::strtod(b.c_str(), &end); if (*end) return false; }
    return max_zoom > 1.0 && max_zoom <= 4.0 && release > 0.0 && std::isfinite(release) &&
           std::ceil((max_zoom - 1.0) / release) <= 4096.0;
}

int usage(const char* argv0) {
    std::fprintf(stderr,
                 "usage: %s --file <in.bgr> --width W --height H --out <out.bgr> [--past-window N] [--future-window N]\n"
                 "          [--working-height N] [--batch N] [--mode global|lock|orb|sift] [--mode-at CALL] [--frames N]\n"
                 "          [--rank R --world S --id-file PATH] [--device D] [--checksums FILE] [--crop MAX_ZOOM[,RELEASE]]\n", argv0);
    return 1;
}

bool pread_full(int fd, uint8_t* p, size_t n, off_t off) {
    while (n) {
        const ssize_t r = pread(fd, p, n, off);
        if (r <= 0) return false;
        p += r; n -= (size_t)r; off += r;
    }
    return true;
}

bool pwrite_full(int fd, const uint8_t* p, size_t n, off_t off) {
    while (n) {
        const ssize_t r = pwrite(fd, p, n, off);
        if (r <= 0) return false;
        p += r; n -= (size_t)r; off += r;
    }
    return true;
}

// rank 0 publishes the id (written to a temporary name, then renamed: readers never see a partial file)
bool exchange_id(const Options& o, vstab_nccl_id* id) {
    if (o.rank == 0) {
        if (vstab_nccl_get_unique_id(id) != VSTAB_OK) return false;
        const std::string tmp = o.id_file + ".tmp";
        std::FILE* f = std::fopen(tmp.c_str(), "wb");
        if (!f) return false;
        const bool ok = std::fwrite(id->bytes, 1, sizeof id->bytes, f) == sizeof id->bytes;
        std::fclose(f);
        return ok && std::rename(tmp.c_str(), o.id_file.c_str()) == 0;
    }
    for (int tries = 0; tries < 6000; ++tries) {                   // up to 60 s
        std::FILE* f = std::fopen(o.id_file.c_str(), "rb");
        if (f) {
            const size_t n = std::fread(id->bytes, 1, sizeof id->bytes, f);
            std::fclose(f);
            if (n == sizeof id->bytes) return true;
        }
        std::this_thread::sleep_for(std::chrono::milliseconds(10));
    }
    return false;
}

}  // namespace

int main(int argc, char** argv) {
    Options o;
    for (int i = 1; i < argc; ++i) {
        const std::string a = argv[i];
        auto next = [&](const char* what) -> const char* {
            if (i + 1 >= argc) { std::fprintf(stderr, "Error: %s requires a value\n", what); std::exit(1); }
            return argv[++i];
        };
        if (a == "--file") o.in = next("--file");
        else if (a == "--out") o.out = next("--out");
        else if (a == "--width") o.width = std::atoi(next("--width"));
        else if (a == "--height") o.height = std::atoi(next("--height"));
        else if (a == "--past-window") o.past = std::atol(next("--past-window"));
        else if (a == "--future-window") o.future = std::atol(next("--future-window"));
        else if (a == "--working-height") o.working_height = std::atoi(next("--working-height"));
        else if (a == "--batch") o.batch = std::atoi(next("--batch"));
        else if (a == "--frames") o.frames = std::atol(next("--frames"));
        else if (a == "--mode-at") o.mode_at = std::atol(next("--mode-at"));
        else if (a == "--mode") { if (!parse_mode(next("--mode"), o.mode)) return usage(argv[0]); }
        else if (a == "--rank") o.rank = std::atoi(next("--rank"));
        else if (a == "--world") o.world = std::atoi(next("--world"));
        else if (a == "--id-file") o.id_file = next("--id-file");
        else if (a == "--device") o.device = std::atoi(next("--device"));
        else if (a == "--checksums") o.checksums = next("--checksums");
        else if (a == "--crop") { if (!parse_crop(next("--crop"), o.crop, o.crop_release)) return usage(argv[0]); }
        else return usage(argv[0]);
    }
    if (o.in.empty() || o.out.empty() || o.width <= 0 || o.height <= 0 || o.batch < 1 || o.past < 0 || o.future < 0 ||
        o.world < 1 || o.rank < 0 || o.rank >= o.world || (o.world > 1 && o.id_file.empty()))
        return usage(argv[0]);
    if (o.device < 0) o.device = o.rank;
    const size_t row_bytes = (size_t)o.width * 3, frame_bytes = row_bytes * (size_t)o.height;

    const int fin = open(o.in.c_str(), O_RDONLY);
    if (fin < 0) { std::fprintf(stderr, "Error: cannot open %s\n", o.in.c_str()); return 2; }
    struct stat sb;
    if (fstat(fin, &sb) != 0) { std::fprintf(stderr, "Error: cannot stat %s\n", o.in.c_str()); return 2; }
    long n_total = (long)((size_t)sb.st_size / frame_bytes);
    if (o.frames >= 0 && o.frames < n_total) n_total = o.frames;
    if (n_total < 1) { std::fprintf(stderr, "Error: %s holds no complete %dx%d frame\n", o.in.c_str(), o.width, o.height); return 2; }

    // the instance: argument errors (window 0/0, working height <= 90: src/stabilizer.cpp:40-49) come back before any device work
    vstab_offline_t* job = nullptr;
    vstab_status st = vstab_offline_create((size_t)o.past, (size_t)o.future, o.working_height, o.height, o.width, o.batch, o.device, &job);
    if (st != VSTAB_OK) {
        std::fprintf(stderr, "Error: %s\n", vstab_offline_last_error(nullptr));
        return st == VSTAB_ERR_INVALID_ARGUMENT ? 1 : 3;
    }
    auto fail = [&](int code, const char* what) {
        std::fprintf(stderr, "Error: %s: %s\n", what, vstab_offline_last_error(job));
        vstab_offline_destroy(job);
        return code;
    };
    if (o.crop > 1.0 && vstab_offline_set_crop(job, o.crop, o.crop_release) != VSTAB_OK) return fail(1, "vstab_offline_set_crop");
    if (o.world > 1) {
        vstab_nccl_id id;
        if (!exchange_id(o, &id)) return fail(2, "NCCL id exchange through --id-file failed");
        if (vstab_offline_comm_init(job, &id, o.rank, o.world) != VSTAB_OK) return fail(3, "vstab_offline_comm_init");
    }
    vstab_shard_plan pl;
    if (vstab_offline_plan(n_total, o.world, o.rank, (size_t)o.future, &pl) != VSTAB_OK) return fail(3, "vstab_offline_plan");
    const long n_local = pl.last - pl.first, n_calls = pl.call_last - pl.call_first;

    // this rank's frames (+ halo) and outputs in pinned host memory
    uint8_t* shard = (uint8_t*)vstab_host_alloc(frame_bytes * (size_t)(n_local > 0 ? n_local : 1));
    uint8_t* halo = pl.first > 0 ? (uint8_t*)vstab_host_alloc(frame_bytes) : nullptr;
    uint8_t* outb = (uint8_t*)vstab_host_alloc(frame_bytes * (size_t)(n_calls > 0 ? n_calls : 1));
    std::vector<uint64_t> sums((size_t)(n_calls > 0 ? n_calls : 1));
    if (!shard || !outb || (pl.first > 0 && !halo)) return fail(3, "vstab_host_alloc");
    if (n_local > 0 && !pread_full(fin, shard, frame_bytes * (size_t)n_local, (off_t)((size_t)pl.first * frame_bytes))) return fail(2, "short read of the shard");
    if (halo && !pread_full(fin, halo, frame_bytes, (off_t)((size_t)(pl.first - 1) * frame_bytes))) return fail(2, "short read of the halo frame");
    close(fin);

    vstab_offline_cfg cfg;
    std::memset(&cfg, 0, sizeof cfg);
    cfg.n_total = n_total; cfg.mode = o.mode; cfg.lock_call = o.mode_at;
    cfg.source = VSTAB_SRC_HOST;
    cfg.host_frames = shard; cfg.frame_stride = frame_bytes; cfg.step = row_bytes; cfg.host_halo = halo;
    cfg.host_out = outb; cfg.out_frame_stride = frame_bytes; cfg.out_step = row_bytes;
    cfg.checksums = sums.data();
    vstab_offline_report rep;
    std::memset(&rep, 0, sizeof rep);
    const auto t0 = std::chrono::steady_clock::now();
    if (vstab_offline_run(job, &cfg, &rep) != VSTAB_OK) return fail(3, "vstab_offline_run");
    const double wall = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();

    // every rank writes its calls at their place of the output clip
    const int fout = open(o.out.c_str(), O_WRONLY | O_CREAT, 0644);
    if (fout < 0) return fail(2, "cannot open the output file");
    if (n_calls > 0 && !pwrite_full(fout, outb, frame_bytes * (size_t)n_calls, (off_t)((size_t)pl.call_first * frame_bytes))) return fail(2, "short write");
    close(fout);
    if (!o.checksums.empty()) {
        std::FILE* f = std::fopen((o.world > 1 ? o.checksums + "." + std::to_string(o.rank) : o.checksums).c_str(), "w");
        if (!f) return fail(2, "cannot open the checksum file");
        for (long c = 0; c < n_calls; ++c) std::fprintf(f, "%ld %016llx\n", pl.call_first + c, (unsigned long long)sums[(size_t)c]);
        std::fclose(f);
    }
    std::fprintf(stderr,
                 "{\"rank\": %d, \"world\": %d, \"frames\": [%ld, %ld], \"calls\": [%ld, %ld], \"device_ms\": %.3f, \"source_ms\": %.3f, "
                 "\"estimate_ms\": %.3f, \"exchange_ms\": %.3f, \"render_ms\": %.3f, \"wall_s\": %.3f}\n",
                 o.rank, o.world, pl.first, pl.last, pl.call_first, pl.call_last, rep.total_ms, rep.source_ms, rep.estimate_ms,
                 rep.exchange_ms, rep.render_ms, wall);
    vstab_host_free(shard); vstab_host_free(halo); vstab_host_free(outb);
    vstab_offline_destroy(job);
    return 0;
}
