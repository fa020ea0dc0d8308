// project_main.cpp -- the `project` command line on the B200 pipeline.
//
//   project                      mode 0 (message says "mono", like the reference)
//   project <mode 0-3> <1|2|m|s> [--taps N] [--chunk-blocks K] [--device D] [--tune HZ] [--stats]
//   project <mode 0-3> <1|2|m|s> --scan SECONDS [--fft N] [--threshold DB] [--device D]
//
// --tune HZ: decode the station HZ (an integer, may be negative) above the capture's centre
// frequency (fmrx_set_tuning); |HZ| < rf_fs/2 of the mode, else the usage message and exit 1.
//
// --scan SECONDS: decode nothing; find the stations in up to SECONDS of signal at the mode's
// RF rate (0: until EOF), read and scanned chunk by chunk (fmrx_scan_process, so a live
// rtl_sdr pipe works), and print one line per station on stdout in ascending offset:
// offset_hz<TAB>level_db<TAB>snr_db, the offset an integer, the levels to 0.1 dB
// (fmrx_find_stations) -- the offsets are what --tune takes.  Exit status 0.  --fft N: the
// Welch segment length, a power of two in 256..16384 (default 4096); --threshold DB: the
// detection threshold above the noise floor (default 10).  Malformed values, --fft or
// --threshold without --scan, and --scan with --tune: the usage message and exit 1.
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
#include <algorithm>
#include <chrono>
#include <cmath>
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
                         "\t\t<mode> is a value from 0 to 3\n\t\t   <channels> is either 1 or 2\n"
                         "or\nUsage %s <mode> <channels> --scan SECONDS [--fft N] [--threshold DB]\n",
                 argv0, argv0, argv0);
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

// --scan: the stations in up to `seconds` of stdin (0: until EOF); exit status 0
int scan_stdin(const fmrx_mode_info &mi, int device, double seconds, int fft, double threshold_db)
{
    fmrx_scan *sc = nullptr;
    int rc = fmrx_scan_create(&sc, fft, mi.rf_fs, device);
    if (rc != FMRX_OK) {
        std::fprintf(stderr, "fmrx_scan_create: %s (%s)\n", fmrx_strerror(rc), fmrx_last_error());
        return 1;
    }
    const uint64_t limit = seconds > 0 ? static_cast<uint64_t>(seconds * mi.rf_fs) : UINT64_MAX;
    const size_t chunk = static_cast<size_t>(0.2 * mi.rf_fs);      // pairs per read: about 0.2 s of signal
    void *buf = nullptr;
    if (fmrx_host_alloc(&buf, 2 * chunk) != FMRX_OK) {
        std::fprintf(stderr, "pinned allocation failed (%s)\n", fmrx_last_error());
        return 1;
    }
    for (uint64_t done = 0; done < limit;) {
        const size_t want = static_cast<size_t>(std::min<uint64_t>(chunk, limit - done));
        const size_t got = read_full(STDIN_FILENO, static_cast<uint8_t *>(buf), 2 * want) / 2;   // whole pairs
        if (got && (rc = fmrx_scan_process(sc, static_cast<const uint8_t *>(buf), got)) != FMRX_OK) {
            std::fprintf(stderr, "fmrx_scan_process: %s (%s)\n", fmrx_strerror(rc), fmrx_last_error());
            return 1;
        }
        done += got;
        if (got < want)
            break;
    }
    std::vector<double> psd(fft);
    uint64_t n_seg = 0;
    std::vector<fmrx_station> st(fft);
    int found = 0;
    if ((rc = fmrx_scan_read(sc, psd.data(), psd.size(), &n_seg)) != FMRX_OK ||
        (rc = fmrx_find_stations(psd.data(), fft, mi.rf_fs, threshold_db, 0.0, st.data(), fft, &found)) != FMRX_OK) {
        std::fprintf(stderr, "band scan: %s (%s)\n", fmrx_strerror(rc), fmrx_last_error());
        return 1;
    }
    for (int i = 0; i < found; i++)
        std::printf("%lld\t%.1f\t%.1f\n", std::llround(st[i].offset_hz), st[i].level_db, st[i].snr_db);
    std::fflush(stdout);
    fmrx_host_free(buf);
    fmrx_scan_destroy(sc);
    return 0;
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
    bool stats = false, tuned = false, scan = false, scan_opts = false;
    double scan_s = 0.0, threshold_db = 10.0;
    int fft = 4096;
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
            tuned = true;
        }
        else if (a == "--scan" || a == "--threshold") {
            if (i + 1 >= argc) usage(argv[0]);
            char *end = nullptr;
            const double v = std::strtod(argv[++i], &end);
            if (end == argv[i] || *end || !std::isfinite(v)) usage(argv[0]);
            if (a == "--scan") {
                if (v < 0) usage(argv[0]);
                scan = true;
                scan_s = v;
            } else {
                threshold_db = v;
                scan_opts = true;
            }
        }
        else if (a == "--fft") {
            if (i + 1 >= argc) usage(argv[0]);
            char *end = nullptr;
            const long v = std::strtol(argv[++i], &end, 10);
            if (end == argv[i] || *end || v < 256 || v > 16384 || (v & (v - 1))) usage(argv[0]);
            fft = static_cast<int>(v);
            scan_opts = true;
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
    if ((scan && tuned) || (scan_opts && !scan))
        usage(argv[0]);
    std::fprintf(stderr, "Operating in mode %d, %s\n", mode, channels == 1 ? "mono" : "stereo");

    fmrx_mode_info mi;
    if (fmrx_mode_table(mode, taps, &mi) != FMRX_OK) {
        std::fprintf(stderr, "Invalid taps: %d!\n", taps);
        return 1;
    }
    if (!(std::llabs(tune_hz) < mi.rf_fs / 2))
        usage(argv[0]);
    if (scan)
        return scan_stdin(mi, device, scan_s, fft, threshold_db);
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
