// project_main.cpp -- the `project` command line on the B200 pipeline.
//
//   project                      mode 0 (message says "mono", like the reference)
//   project <mode 0-3> <1|2|m|s> [--taps N] [--chunk-blocks K] [--device D] [--tune HZ] [--stats]
//
// --tune HZ: decode the station HZ (an integer, may be negative) above the capture's centre
// frequency (fmrx_set_tuning); |HZ| < rf_fs/2 of the mode, else the usage message and exit 1.
//
// stdin : raw interleaved u8 I/Q at the mode's RF rate
// stdout: raw s16le PCM, interleaved R,L, 48 or 44.1 kS/s -- for either channel
//         argument, exactly as the reference (src/project.cpp:301-302,183-193: the
//         argument only changes the stderr message)
// stderr: "Operating in mode M, mono|stereo", then "End of input stream reached!" at
//         EOF; exit status 1 (src/project.cpp:51-54).  A trailing partial block is
//         dropped as the reference drops it; unlike the reference (which loses up to 4
//         queued blocks when rf_thread calls exit) every complete block is emitted.
//
// Replaces the reference's rf_thread / audio_thread pair and their queue
// (src/project.cpp:19-197, one mutex, one condition variable, capacity 3) with the same
// shape one level up: a READER thread fills a ring of pinned chunk slots from stdin
// (K blocks each, ~0.2 s of signal by default), the main thread hands each filled slot to
// fmrx_process() -- whose CUDA streams overlap copy-in, the four kernels and copy-out --
// and a WRITER thread drains finished slots to stdout, so that reading chunk i+1,
// processing chunk i and writing chunk i-1 overlap (live use: rtl_sdr | project | aplay,
// src/project.cpp:392-393).  --stats prints the sustained real-time factor and the
// per-chunk latency (last input byte read -> last PCM byte written) on stderr.
#include <chrono>
#include <condition_variable>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <thread>
#include <vector>
#include <unistd.h>

#include "fmrx.h"

namespace {

[[noreturn]] void usage(const char *argv0)
{
    std::fprintf(stderr, "Usage: %s\nor \nUsage %s <mode> <channels>\n"
                         "\t\t<mode> is a value from 0 to 3\n\t\t   <channels> is either 1 or 2\n",
                 argv0, argv0);
    std::exit(1);
}

size_t read_full(int fd, uint8_t *dst, size_t want)
{
    size_t got = 0;
    while (got < want) {
        const ssize_t r = ::read(fd, dst + got, want - got);
        if (r <= 0)
            break;
        got += static_cast<size_t>(r);
    }
    return got;
}

bool write_full(int fd, const uint8_t *src, size_t n)
{
    while (n) {
        const ssize_t w = ::write(fd, src, n);
        if (w <= 0)
            return false;
        src += w;
        n -= static_cast<size_t>(w);
    }
    return true;
}

}  // namespace

int main(int argc, char *argv[])
{
    int mode = 0, channels = 1, taps = 51, chunk_blocks = 0, device = -1;
    long long tune_hz = 0;
    bool stats = false;
    // positional part, as src/project.cpp:278-299
    int npos = 0;
    const char *pos[2] = { nullptr, nullptr };
    for (int i = 1; i < argc; i++) {
        const std::string a = argv[i];
        auto next = [&](int &dst) {
            if (i + 1 >= argc) usage(argv[0]);
            dst = std::atoi(argv[++i]);
        };
        if (a == "--taps") next(taps);
        else if (a == "--chunk-blocks") next(chunk_blocks);
        else if (a == "--device") next(device);
        else if (a == "--tune") {
            if (i + 1 >= argc) usage(argv[0]);
            char *end = nullptr;
            tune_hz = std::strtoll(argv[++i], &end, 10);
            if (end == argv[i] || *end) usage(argv[0]);
        }
        else if (a == "--stats") stats = true;
        else if (npos < 2) pos[npos++] = argv[i];
        else usage(argv[0]);
    }
    if (npos < 2) {
        std::fprintf(stderr, "Operating in default mode 0, mono\n");      // a single argument is ignored
    } else {
        mode = std::atoi(pos[0]);
        if (!std::strcmp(pos[1], "m")) channels = 1;
        else if (!std::strcmp(pos[1], "s")) channels = 2;
        else channels = std::atoi(pos[1]);
        if (mode < 0 || mode > 3) {
            std::fprintf(stderr, "Invalid mode: %d!\n", mode);
            return 1;
        }
        if (channels < 1 || channels > 2) {
            std::fprintf(stderr, "Invaild channel: %d!\n", channels);      // sic, as the reference
            return 1;
        }
    }
    std::fprintf(stderr, "Operating in mode %d, %s\n", mode, channels == 1 ? "mono" : "stereo");

    fmrx_mode_info mi;
    if (fmrx_mode_table(mode, taps, &mi) != FMRX_OK) {
        std::fprintf(stderr, "Invalid taps: %d!\n", taps);
        return 1;
    }
    if (!(std::llabs(tune_hz) < mi.rf_fs / 2))
        usage(argv[0]);
    if (chunk_blocks <= 0) {
        // about 0.2 s of signal per call: low latency for a live rtl_sdr pipe
        chunk_blocks = static_cast<int>(0.2 * mi.rf_fs * 2 / mi.block_size);
        if (chunk_blocks < 1) chunk_blocks = 1;
    }
    fmrx_config cfg;
    std::memset(&cfg, 0, sizeof(cfg));
    cfg.mode = mode;
    cfg.taps = taps;
    cfg.n_captures = 1;
    cfg.device = device;
    cfg.chunk_blocks = chunk_blocks;
    fmrx_pipeline *p = nullptr;
    int rc = fmrx_create(&p, &cfg);
    if (rc != FMRX_OK) {
        std::fprintf(stderr, "fmrx_create: %s (%s)\n", fmrx_strerror(rc), fmrx_last_error());
        return 1;
    }
    if (tune_hz && (rc = fmrx_set_tuning(p, 0, static_cast<double>(tune_hz))) != FMRX_OK) {
        std::fprintf(stderr, "fmrx_set_tuning: %s (%s)\n", fmrx_strerror(rc), fmrx_last_error());
        return 1;
    }
    const size_t in_bytes = static_cast<size_t>(chunk_blocks) * mi.block_size;
    const size_t out_elems = static_cast<size_t>(chunk_blocks) * 2 * mi.audio_per_block;
    using clk = std::chrono::steady_clock;
    // the ring: a slot goes EMPTY -> (reader) FILLED -> (main) DONE -> (writer) EMPTY, in order
    enum { EMPTY, FILLED, DONE };
    struct Slot {
        void *iq = nullptr, *pcm = nullptr;
        size_t blocks = 0;
        bool last = false;               // the reader hit EOF in (or right after) this slot
        int state = EMPTY;
        clk::time_point t_read;          // its last input byte was read
    };
    constexpr int kSlots = 4;
    std::vector<Slot> ring(kSlots);
    for (auto &sl : ring)
        if (fmrx_host_alloc(&sl.iq, in_bytes) != FMRX_OK || fmrx_host_alloc(&sl.pcm, out_elems * sizeof(int16_t)) != FMRX_OK) {
            std::fprintf(stderr, "pinned allocation failed (%s)\n", fmrx_last_error());
            return 1;
        }
    std::mutex mu;
    std::condition_variable cv;
    bool failed = false;
    double lat_sum = 0.0, lat_max = 0.0, lat_min = 1e30, proc_sum = 0.0;
    size_t n_chunks = 0, n_blocks = 0;
    const clk::time_point t_start = clk::now();

    std::thread reader([&] {
        for (int i = 0;; i = (i + 1) % kSlots) {
            Slot &sl = ring[i];
            {
                std::unique_lock<std::mutex> lk(mu);
                cv.wait(lk, [&] { return sl.state == EMPTY || failed; });
                if (failed)
                    return;
            }
            const size_t got = read_full(STDIN_FILENO, static_cast<uint8_t *>(sl.iq), in_bytes);
            sl.blocks = got / mi.block_size;                            // partial block: dropped
            sl.last = got < in_bytes;
            sl.t_read = clk::now();
            {
                std::lock_guard<std::mutex> lk(mu);
                sl.state = FILLED;
            }
            cv.notify_all();
            if (sl.last)
                return;
        }
    });
    std::thread writer([&] {
        for (int i = 0;; i = (i + 1) % kSlots) {
            Slot &sl = ring[i];
            {
                std::unique_lock<std::mutex> lk(mu);
                cv.wait(lk, [&] { return sl.state == DONE || failed; });
                if (failed)
                    return;
            }
            bool ok = true;
            if (sl.blocks)
                ok = write_full(STDOUT_FILENO, static_cast<const uint8_t *>(sl.pcm), sl.blocks * 2 * mi.audio_per_block * sizeof(int16_t));
            const double lat = std::chrono::duration<double>(clk::now() - sl.t_read).count();
            const bool last = sl.last;
            {
                std::lock_guard<std::mutex> lk(mu);
                if (sl.blocks) {
                    lat_sum += lat;
                    lat_max = lat > lat_max ? lat : lat_max;
                    lat_min = lat < lat_min ? lat : lat_min;
                    n_chunks++;
                    n_blocks += sl.blocks;
                }
                sl.state = EMPTY;
                if (!ok)
                    failed = true;
            }
            cv.notify_all();
            if (last || !ok)
                return;
        }
    });
    for (int i = 0;; i = (i + 1) % kSlots) {
        Slot &sl = ring[i];
        {
            std::unique_lock<std::mutex> lk(mu);
            cv.wait(lk, [&] { return sl.state == FILLED || failed; });
            if (failed)
                break;
        }
        if (sl.blocks) {
            const clk::time_point t0 = clk::now();
            rc = fmrx_process(p, static_cast<const uint8_t *>(sl.iq), in_bytes, sl.blocks, static_cast<int16_t *>(sl.pcm), out_elems);
            proc_sum += std::chrono::duration<double>(clk::now() - t0).count();
            if (rc != FMRX_OK)
                std::fprintf(stderr, "fmrx_process: %s (%s)\n", fmrx_strerror(rc), fmrx_last_error());
        }
        const bool last = sl.last;
        {
            std::lock_guard<std::mutex> lk(mu);
            sl.state = DONE;
            if (rc != FMRX_OK)
                failed = true;
        }
        cv.notify_all();
        if (last || rc != FMRX_OK)
            break;
    }
    {
        std::unique_lock<std::mutex> lk(mu);
        if (failed) {                    // (the reader may sit in read(2) for ever: no join)
            lk.unlock();
            std::fflush(stderr);
            std::_Exit(1);
        }
    }
    reader.join();
    writer.join();
    {
        std::lock_guard<std::mutex> lk(mu);
        if (failed) {
            std::fflush(stderr);
            std::_Exit(1);
        }
    }
    std::fprintf(stderr, "End of input stream reached!\n");
    if (stats && n_chunks) {
        const double wall = std::chrono::duration<double>(clk::now() - t_start).count();
        const double signal_s = static_cast<double>(n_blocks) * mi.block_size / 2.0 / mi.rf_fs;
        std::fprintf(stderr,
                     "fmrx stats: {\"mode\": %d, \"taps\": %d, \"chunk_blocks\": %d, \"chunk_seconds\": %.4f, \"chunks\": %zu, "
                     "\"signal_seconds\": %.3f, \"wall_seconds\": %.3f, \"real_time_factor\": %.2f, "
                     "\"process_ms_per_chunk\": %.3f, \"latency_ms\": {\"min\": %.3f, \"mean\": %.3f, \"max\": %.3f}}\n",
                     mode, taps, chunk_blocks, static_cast<double>(chunk_blocks) * mi.block_size / 2.0 / mi.rf_fs, n_chunks, signal_s, wall,
                     signal_s / wall, 1e3 * proc_sum / n_chunks, 1e3 * lat_min, 1e3 * lat_sum / n_chunks, 1e3 * lat_max);
    }
    for (auto &sl : ring) {
        fmrx_host_free(sl.iq);
        fmrx_host_free(sl.pcm);
    }
    fmrx_destroy(p);
    return 1;                                                       // the reference's exit status at EOF
}
