// fmrx_api.cu -- the extern "C" boundary (include/fmrx.h): per-operator entry
// points on host pointers, and the fused multi-capture pipeline.
//
// Pipeline scheduling.  A call is cut into chunks of whole blocks.  Three CUDA
// streams form a software pipeline over chunks, the device-side counterpart of
// the reference's rf_thread -> queue -> audio_thread hand-off
// (src/project.cpp:71-80,133-141):
//     front : [H2D] -> K1 rf+demod -> K2 band-pass pair
//     pll   : K3 PLL recurrence (the long pole: one dependent chain per capture)
//     back  : K4 audio -> [D2H]
// Chunk i+1's front stage and chunk i-1's back stage run under chunk i's PLL.
// Buffers rotate over kSets sets; the FIR history each stage needs from the
// previous chunk is kept in a small per-capture "tail" (CarryLayout), written by
// the stream that produces the data, and copied in front of the next chunk's buffer.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <memory>
#include <numeric>
#include <new>
#include <type_traits>
#include <vector>

#include "fmrx.h"
#include "fmrx_internal.h"

using namespace fmrx;

namespace {

// Owners of the handles' device memory, events and streams: each releases its resource exactly once.
struct DevFree {
    void operator()(void *q) const { cudaFree(q); }
};
struct EventDestroy {
    void operator()(cudaEvent_t e) const { cudaEventDestroy(e); }
};
struct StreamDestroy {
    void operator()(cudaStream_t s) const { cudaStreamDestroy(s); }
};
template <class T> using dptr = std::unique_ptr<T, DevFree>;
using event_ptr = std::unique_ptr<std::remove_pointer_t<cudaEvent_t>, EventDestroy>;
using stream_ptr = std::unique_ptr<std::remove_pointer_t<cudaStream_t>, StreamDestroy>;

// `count` elements (at least one) in place of q's buffer, which is freed first
template <class T> cudaError_t dalloc(dptr<T> &q, size_t count)
{
    q.reset();
    T *raw = nullptr;
    const cudaError_t e = cudaMalloc(reinterpret_cast<void **>(&raw), (count ? count : 1) * sizeof(T));
    q.reset(raw);
    return e;
}

// The same in stream order on s, without a host synchronisation: the old buffer goes to cudaFreeAsync, where reset()
// would call cudaFree, which waits for the whole device.
template <class T> cudaError_t dalloc_async(dptr<T> &q, size_t count, cudaStream_t s)
{
    if (q) {
        const cudaError_t e = cudaFreeAsync(q.release(), s);
        if (e != cudaSuccess)
            return e;
    }
    T *raw = nullptr;
    const cudaError_t e = cudaMallocAsync(reinterpret_cast<void **>(&raw), count * sizeof(T), s);
    q.reset(raw);
    return e;
}

cudaError_t make_event(event_ptr &ev, unsigned flags = cudaEventDisableTiming)
{
    cudaEvent_t raw = nullptr;
    const cudaError_t e = cudaEventCreateWithFlags(&raw, flags);
    ev.reset(raw);
    return e;
}

cudaError_t make_stream(stream_ptr &s, int priority = 0)
{
    cudaStream_t raw = nullptr;
    const cudaError_t e = cudaStreamCreateWithPriority(&raw, cudaStreamNonBlocking, priority);
    s.reset(raw);
    return e;
}

thread_local char g_err[256] = "";

int cuda_fail(cudaError_t e, const char *what)
{
    std::snprintf(g_err, sizeof(g_err), "%s: %s", what, cudaGetErrorString(e));
    cudaGetLastError();   // consumed here, so that the failure does not resurface from the next launch's error check
    if (e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver ||
        e == cudaErrorNoKernelImageForDevice)
        return FMRX_ERR_NO_DEVICE;
    if (e == cudaErrorMemoryAllocation)
        return FMRX_ERR_ALLOC;
    return FMRX_ERR_CUDA;
}

#define CU(call)                                            \
    do {                                                    \
        cudaError_t e_ = (call);                            \
        if (e_ != cudaSuccess)                              \
            return cuda_fail(e_, #call);                    \
    } while (0)

// Device scratch of the operator entry points: a per-thread arena that only ever grows, so that a block loop
// calling the operators (the unmodified reference main linked against host/filter_shim.cpp does: eleven calls
// per block, src/project.cpp:65-175) pays for cudaMalloc / cudaFree once and not forty times per block.
// A DevBuf takes the next slot of the calling thread's arena for the duration of one entry point.
struct Arena {
    static constexpr int kSlots = 6;
    void *p[kSlots] = {};
    size_t cap[kSlots] = {};
    int device = -1, used = 0;
    ~Arena() { release(); }
    void release()
    {
        for (int i = 0; i < kSlots; i++) {
            if (p[i])
                cudaFree(p[i]);      // (after the context has gone at process exit this fails, harmlessly)
            p[i] = nullptr;
            cap[i] = 0;
        }
    }
};
thread_local Arena g_arena;

struct DevBuf {
    void *p = nullptr;
    int slot = -1;
    DevBuf() { slot = g_arena.used < Arena::kSlots ? g_arena.used++ : -1; }
    ~DevBuf()
    {
        if (slot >= 0)
            g_arena.used--;
        else if (p)
            cudaFree(p);
    }
    cudaError_t alloc(size_t bytes)
    {
        bytes = bytes ? bytes : 1;
        if (slot < 0)
            return cudaMalloc(&p, bytes);
        int dev = 0;
        cudaError_t e = cudaGetDevice(&dev);
        if (e != cudaSuccess)
            return e;
        if (dev != g_arena.device) {
            g_arena.release();
            g_arena.device = dev;
        }
        if (g_arena.cap[slot] < bytes) {
            if (g_arena.p[slot])
                cudaFree(g_arena.p[slot]);
            g_arena.p[slot] = nullptr;
            g_arena.cap[slot] = 0;
            const size_t want = bytes + bytes / 2;       // (some headroom: block sizes vary by a few taps)
            e = cudaMalloc(&g_arena.p[slot], want);
            if (e != cudaSuccess)
                return e;
            g_arena.cap[slot] = want;
        }
        p = g_arena.p[slot];
        return cudaSuccess;
    }
    template <class T> T *as() { return static_cast<T *>(p); }
};

PllParams make_pll_params(float freq, float Fs, float scale, float adjust, float bw)
{
    // src/filter.cpp:139-143,167 -- float products, then (2*PI)*(double)(freq/Fs)
    PllParams p;
    const float cp = 2.666f, ci = 3.555f;
    p.kp = bw * cp;
    p.ki = (bw * bw) * ci;
    const float rho = freq / Fs;
    p.w = (2.0 * 3.14159265358979323846) * static_cast<double>(rho);
    p.scale = scale;
    p.adjust = adjust;
    return p;
}

}  // namespace

// ---------------------------------------------------------------------------
// misc
// ---------------------------------------------------------------------------

extern "C" const char *fmrx_strerror(int s)
{
    switch (s) {
    case FMRX_OK: return "ok";
    case FMRX_ERR_ARG: return "invalid argument";
    case FMRX_ERR_NO_DEVICE: return "no usable CUDA (sm_100) device";
    case FMRX_ERR_CUDA: return "CUDA runtime error";
    case FMRX_ERR_ALLOC: return "out of memory";
    case FMRX_ERR_STATE: return "state blob does not match pipeline";
    default: return "unknown status";
    }
}

extern "C" const char *fmrx_last_error(void) { return g_err; }
extern "C" int fmrx_abi_version(void) { return FMRX_ABI_VERSION; }

extern "C" int fmrx_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

extern "C" int fmrx_host_alloc(void **ptr, size_t bytes)
{
    if (!ptr)
        return FMRX_ERR_ARG;
    CU(cudaHostAlloc(ptr, bytes ? bytes : 1, cudaHostAllocDefault));
    return FMRX_OK;
}

extern "C" int fmrx_host_free(void *ptr)
{
    if (ptr)
        CU(cudaFreeHost(ptr));
    return FMRX_OK;
}

// ---------------------------------------------------------------------------
// per-operator entry points (host pointers)
// ---------------------------------------------------------------------------

extern "C" int fmrx_u8_to_f32(const uint8_t *raw, size_t n, float *out)
{
    if ((!raw || !out) && n)
        return FMRX_ERR_ARG;
    if (n == 0)
        return FMRX_OK;
    DevBuf din, dout;
    CU(din.alloc(n));
    CU(dout.alloc(n * sizeof(float)));
    CU(cudaMemcpy(din.p, raw, n, cudaMemcpyHostToDevice));
    CU(launch_u8_to_f32(din.as<uint8_t>(), n, dout.as<float>(), 0));
    CU(cudaMemcpy(out, dout.p, n * sizeof(float), cudaMemcpyDeviceToHost));
    return FMRX_OK;
}

extern "C" int fmrx_resample(float *out, size_t *out_len, float *state, size_t state_len,
                             const float *in, size_t in_len, const float *coeff, int taps,
                             int up, int down)
{
    if (!out_len || !state || !in || !coeff || taps < 1 || up < 1 || down < 1)
        return FMRX_ERR_ARG;
    if (in_len < static_cast<size_t>(taps - 1) || in_len > 0x7fffffffu / static_cast<size_t>(up))
        return FMRX_ERR_ARG;
    const int n_in = static_cast<int>(in_len);
    const int n_out = static_cast<int>(static_cast<long long>(n_in) * up / down);   // src/filter.cpp:77
    if (n_out && !out)
        return FMRX_ERR_ARG;
    DevBuf d_in, d_state, d_coeff, d_out;
    CU(d_in.alloc(in_len * sizeof(float)));
    CU(d_state.alloc(state_len * sizeof(float)));
    CU(d_coeff.alloc(taps * sizeof(float)));
    CU(d_out.alloc(static_cast<size_t>(n_out) * sizeof(float)));
    CU(cudaMemcpy(d_in.p, in, in_len * sizeof(float), cudaMemcpyHostToDevice));
    if (state_len)
        CU(cudaMemcpy(d_state.p, state, state_len * sizeof(float), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(d_coeff.p, coeff, taps * sizeof(float), cudaMemcpyHostToDevice));
    CU(launch_resample(d_out.as<float>(), n_out, d_state.as<float>(), static_cast<int>(state_len),
                       d_in.as<float>(), n_in, d_coeff.as<float>(), taps, up, down, 0));
    if (n_out)
        CU(cudaMemcpy(out, d_out.p, static_cast<size_t>(n_out) * sizeof(float), cudaMemcpyDeviceToHost));
    else
        CU(cudaDeviceSynchronize());
    // src/filter.cpp:95-102: state := last taps-1 inputs (a copy; no arithmetic)
    std::memmove(state, in + (in_len - (taps - 1)), static_cast<size_t>(taps - 1) * sizeof(float));
    *out_len = static_cast<size_t>(n_out);
    return FMRX_OK;
}

extern "C" int fmrx_fmdemod(float *out, float *prev_i, float *prev_q, const float *i_ds,
                            const float *q_ds, size_t n)
{
    if (!prev_i || !prev_q || ((!out || !i_ds || !q_ds) && n) || n > 0x7fffffffu)
        return FMRX_ERR_ARG;
    if (n == 0)
        return FMRX_OK;
    DevBuf di, dq, dout;
    CU(di.alloc(n * sizeof(float)));
    CU(dq.alloc(n * sizeof(float)));
    CU(dout.alloc(n * sizeof(float)));
    CU(cudaMemcpy(di.p, i_ds, n * sizeof(float), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(dq.p, q_ds, n * sizeof(float), cudaMemcpyHostToDevice));
    CU(launch_fmdemod(dout.as<float>(), di.as<float>(), dq.as<float>(), static_cast<int>(n),
                      *prev_i, *prev_q, 0));
    CU(cudaMemcpy(out, dout.p, n * sizeof(float), cudaMemcpyDeviceToHost));
    *prev_i = i_ds[n - 1];   // src/filter.cpp:130-131 (a copy)
    *prev_q = q_ds[n - 1];
    return FMRX_OK;
}

extern "C" int fmrx_pll(float *inout, size_t n, float freq, float Fs, float nco_scale,
                        float phase_adjust, float norm_bandwidth, float state[6])
{
    if (!state || (!inout && n) || n > 0x7fffffffu)
        return FMRX_ERR_ARG;
    if (n == 0)
        return FMRX_OK;   // the reference would index ncoOut[-1]; nothing to do
    DevBuf d_x, d_trig, d_state;
    CU(d_x.alloc(n * sizeof(float)));
    CU(d_trig.alloc(n * sizeof(float)));
    CU(d_state.alloc(8 * sizeof(float)));
    float st8[8] = { state[0], state[1], state[2], state[3], state[4], state[5], 0.0f, 0.0f };
    CU(cudaMemcpy(d_x.p, inout, n * sizeof(float), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(d_state.p, st8, sizeof(st8), cudaMemcpyHostToDevice));
    PllArgs a{};
    a.pilot = d_x.as<float>();
    a.pilot_stride = n;
    a.trig = d_trig.as<float>();
    a.if_stride = n;
    a.if_off = 0;
    a.n_if = static_cast<int>(n);
    a.state = d_state.as<float>();
    a.state_stride = 8;
    a.prm = make_pll_params(freq, Fs, nco_scale, phase_adjust, norm_bandwidth);
    CU(launch_pll(a, 1, 0));
    CU(launch_nco(d_x.as<float>(), d_trig.as<float>(), n, nco_scale, phase_adjust, 0));
    CU(cudaMemcpy(inout, d_x.p, n * sizeof(float), cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(st8, d_state.p, sizeof(st8), cudaMemcpyDeviceToHost));
    for (int i = 0; i < 6; i++)
        state[i] = st8[i];
    return FMRX_OK;
}

extern "C" int fmrx_mixer(float *out, const float *a, const float *b, size_t n)
{
    if ((!out || !a || !b) && n)
        return FMRX_ERR_ARG;
    if (n == 0)
        return FMRX_OK;
    DevBuf da, db, dout;
    CU(da.alloc(n * sizeof(float)));
    CU(db.alloc(n * sizeof(float)));
    CU(dout.alloc(n * sizeof(float)));
    CU(cudaMemcpy(da.p, a, n * sizeof(float), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(db.p, b, n * sizeof(float), cudaMemcpyHostToDevice));
    CU(launch_mixer(dout.as<float>(), da.as<float>(), db.as<float>(), n, 0));
    CU(cudaMemcpy(out, dout.p, n * sizeof(float), cudaMemcpyDeviceToHost));
    return FMRX_OK;
}

extern "C" int fmrx_lr_extract(float *left, float *right, const float *mono, const float *stereo,
                               size_t n)
{
    if ((!left || !right || !mono || !stereo) && n)
        return FMRX_ERR_ARG;
    if (n == 0)
        return FMRX_OK;
    DevBuf dm, ds, dl, dr;
    CU(dm.alloc(n * sizeof(float)));
    CU(ds.alloc(n * sizeof(float)));
    CU(dl.alloc(n * sizeof(float)));
    CU(dr.alloc(n * sizeof(float)));
    CU(cudaMemcpy(dm.p, mono, n * sizeof(float), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(ds.p, stereo, n * sizeof(float), cudaMemcpyHostToDevice));
    CU(launch_lr_extract(dl.as<float>(), dr.as<float>(), dm.as<float>(), ds.as<float>(), n, 0));
    CU(cudaMemcpy(left, dl.p, n * sizeof(float), cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(right, dr.p, n * sizeof(float), cudaMemcpyDeviceToHost));
    return FMRX_OK;
}

extern "C" int fmrx_pcm_pack(int16_t *pcm, const float *left, const float *right, size_t n)
{
    if ((!pcm || !left || !right) && n)
        return FMRX_ERR_ARG;
    if (n == 0)
        return FMRX_OK;
    DevBuf dl, dr, dp;
    CU(dl.alloc(n * sizeof(float)));
    CU(dr.alloc(n * sizeof(float)));
    CU(dp.alloc(2 * n * sizeof(int16_t)));
    CU(cudaMemcpy(dl.p, left, n * sizeof(float), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(dr.p, right, n * sizeof(float), cudaMemcpyHostToDevice));
    CU(launch_pcm_pack(dp.as<int16_t>(), dl.as<float>(), dr.as<float>(), n, 0));
    CU(cudaMemcpy(pcm, dp.p, 2 * n * sizeof(int16_t), cudaMemcpyDeviceToHost));
    return FMRX_OK;
}

// ---------------------------------------------------------------------------
// fused pipeline
// ---------------------------------------------------------------------------

namespace {
constexpr int kDefaultSets = 3;
constexpr uint32_t kStateMagic = 0x58524d46u;   // "FMRX"

struct StateHeader {
    uint32_t magic, mode, taps, hist_if, hist_pairs, reserved;
    int64_t blocks_done;
};

// The PLL state at the start of a stream (src/project.cpp:106-111, :219-224): feedbackI = ncoOut = 1, the rest 0
constexpr float kPllInitState[8] = { 0.0f, 0.0f, 1.0f, 0.0f, 1.0f, 0.0f, 0.0f, 0.0f };

struct BufferSet {
    dptr<uint8_t> iq;           // host-path staging: [C][chunk_blocks*block_size]
    dptr<float> demod;          // [C][H + chunk_if]
    dptr<float> chan;           // [C][H + chunk_if]
    dptr<float> trig;           // [C][H + chunk_if]
    dptr<float> pilot;          // [C][chunk_if]
    dptr<int16_t> pcm;          // host-path staging: [C][chunk_blocks*2*audio_per_block]
    event_ptr front_done, pll_done, free_ev;
    bool free_pending = false;  // free_ev has been recorded at least once
    event_ptr h2d_done, iq_free;   // host path: staging filled / staging read for the last time
    bool iq_free_pending = false;
};

// The sizes every pipeline of a mode derives, and time shards take their halo and chunk size from: H, the IF history
// kept in front of every IF-rate buffer (the band-pass needs T-1, the audio stage T-1 + 5 delayed frames), and the
// most blocks a chunk may hold.  A chunk is one launch of each kernel: its IF samples per capture must stay below 2^26
// (k_pll's table stamps keep the step in 26 bits) and its bytes per capture below 2^31 (int indexing in the FIR
// kernels).
struct PipelineSizes {
    int H;
    long long max_chunk_blocks;
};

PipelineSizes pipeline_sizes(const fmrx_mode_info &mi)
{
    const int delay_if = (kMonoDelay * mi.audio_decim + mi.audio_interp - 1) / mi.audio_interp;
    return { ((mi.taps + delay_if + 8 + 31) / 32) * 32,
             std::min<long long>(((1ll << 26) - 1) / mi.if_per_block, ((1ll << 31) - 1) / mi.block_size) };
}

// What a capture carries from one chunk to the next: one record per capture (fmrx_pipeline::d_carry) holding the bytes
// that follow StateHeader in its blob, in the same order, padded to `pitch` on the device only:
//     [IQ history: 2*hist_pairs bytes, padded to 4][demod tail: H f32][chan tail: H f32] [trig tail: H f32][PLL: 8 f32]
// The first three are FMRX_STATE_FEEDFORWARD, the last two FMRX_STATE_PLL, which is also what a time shard hands on.
struct ByteRange {
    size_t off, len;
};
struct CarryLayout {
    size_t hist_bytes;              // the IQ history, at offset 0
    size_t demod, chan, trig, pll;  // offsets
    ByteRange feedforward, pll_part;
    size_t body;                    // a blob is sizeof(StateHeader) + body bytes
    size_t pitch;                   // body rounded up to 16 bytes: every record is 16-byte aligned
};

CarryLayout carry_layout(int hist_pairs, int H)
{
    const size_t fH = static_cast<size_t>(H) * sizeof(float);
    CarryLayout l;
    l.hist_bytes = 2 * static_cast<size_t>(hist_pairs);
    l.demod = (l.hist_bytes + 3) & ~static_cast<size_t>(3);
    l.chan = l.demod + fH;
    l.trig = l.chan + fH;
    l.pll = l.trig + fH;
    l.body = l.pll + 8 * sizeof(float);
    l.pitch = (l.body + 15) & ~static_cast<size_t>(15);
    l.feedforward = { 0, l.trig };
    l.pll_part = { l.trig, l.body - l.trig };
    return l;
}

// What every handle's creator does first: refuse without a device, resolve -1 to the current device, make `dev`
// current and refuse anything but sm_100.
int open_device(int &dev, size_t *mem_pitch = nullptr)
{
    if (fmrx_device_count() < 1) {
        std::snprintf(g_err, sizeof(g_err), "no CUDA device");
        return FMRX_ERR_NO_DEVICE;
    }
    if (dev < 0)
        CU(cudaGetDevice(&dev));
    CU(cudaSetDevice(dev));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, dev));
    if (prop.major != 10) {
        std::snprintf(g_err, sizeof(g_err), "device %d is sm_%d%d; this library is sm_100a only", dev,
                      prop.major, prop.minor);
        return FMRX_ERR_NO_DEVICE;
    }
    if (mem_pitch)
        *mem_pitch = prop.memPitch;
    return FMRX_OK;
}
}  // namespace

struct fmrx_pipeline {
    fmrx_mode_info mi{};
    int C = 0, device = 0;
    int chunk_blocks = 0;       // blocks per chunk
    bool ramp = false;          // automatic chunk size: the first two chunks of a call are a quarter and a half of it
    int chunk_if = 0;           // IF samples per chunk per capture
    int H = 0;                  // IF history kept in front of every IF-rate buffer
    int hist_pairs = 0;         // IQ pairs of history for K1
    size_t if_stride = 0;       // H + chunk_if
    bool keep_stages = false, timing = false;
    PllParams pll_prm{};
    CarryLayout carry{};

    dptr<float> d_rf_taps, d_pilot_taps, d_chan_taps, d_audio_pm;
    dptr<uint8_t> d_carry;          // [C][carry.pitch]: each capture's carried state
    std::vector<BufferSet> sets;    // the ring of chunk buffers (fmrx_config.n_sets; 3 by default)
    stream_ptr s_front, s_pll, s_back;
    stream_ptr s_h2d;               // host path: the H2D copies, so that chunk i+1 comes in under K1/K2 of chunk i
    event_ptr ev_in, ev_out;
    std::vector<long long> blocks_done;   // per capture: blocks since the start of ITS stream (state blobs carry it)
    long long blocks_run = 0;             // blocks the chunk loop has run since create/reset (the same for every capture)
    long long chunk_counter = 0;
    // tuning (fmrx_set_tuning): configuration, not state.  tune[c] is mirrored in d_tune for K1 and written only
    // while the device is idle (create, reset, fmrx_set_tuning, fmrx_set_state), so a call never uploads it.
    std::vector<RfTune> tune;
    dptr<RfTune> d_tune;                  // [C]
    dptr<float2> d_tune_cs;               // the mixer table (65536 cos, sin), allocated when a capture is first tuned
    bool tuned = false;                   // some capture has a nonzero phase step: K1 runs its tuned variant
    // RDS (fmrx_set_rds): configuration like tuning.  The decoder's buffers are allocated when a capture first turns
    // it on; its kernels run on the front stream after front_done, so every buffer has one user at a time.
    std::vector<int> rds_on;              // [C]
    std::vector<int> rds_caps;            // the captures with RDS on, mirrored in d_rds_caps
    dptr<int> d_rds_caps;
    RdsParams rds_prm{};
    dptr<float> d_rds_taps, d_rds_dtail;  // dtail: [C][rds_dtail_len] demod samples before the chunk
    dptr<float2> d_rds_mix, d_rds_y;      // y: [C][rds_y_len]
    dptr<double2> d_rds_phase;
    dptr<RdsDecState> d_rds_state;        // [C]
    dptr<fmrx_rds_group> d_rds_ring;      // [C][kRdsRing]
    int rds_dtail_len = 0, rds_ytail_len = 0;
    size_t rds_y_len = 0;
    std::vector<uint64_t> rds_read, rds_lost;   // per capture: groups drained / dropped since (re)start
    size_t mem_pitch = 0;       // cudaDeviceProp::memPitch: the largest pitch cudaMemcpy2D takes
    uint64_t launches = 0;

    // keep_stages storage (sized for the last call)
    dptr<float> d_stage[FMRX_STAGE_COUNT];
    size_t stage_if_len = 0, stage_au_len = 0;

    // timing: 8 events per chunk, recorded on the launching streams and only READ when the caller asks
    // (fmrx_last_timing), so that enabling it adds no synchronisation to fmrx_process_device
    std::vector<event_ptr> tev;       // event pool
    size_t tev_used = 0;              // events recorded since the last read
    float last_ms[4] = { 0, 0, 0, 0 };

    ~fmrx_pipeline()
    {
        cudaSetDevice(device);
        cudaDeviceSynchronize();
    }
};

namespace {

// The RDS decoder of `capture` from its stream position blocks_done[capture]: search, no bits, zero history, empty
// ring.  The device must be idle.
int rds_restart(fmrx_pipeline *p, int capture)
{
    const RdsParams &P = p->rds_prm;
    const long long n = p->blocks_done[capture] * p->mi.if_per_block;
    const long long m = (n + P.D - 1) / P.D;                 // the first kept sample from here
    RdsDecState st;
    std::memset(&st, 0, sizeof(st));
    st.n_offset = (p->blocks_done[capture] - p->blocks_run) * p->mi.if_per_block;
    st.w_first = st.w_next = m / P.M;
    st.j = static_cast<long long>(std::ceil(static_cast<double>(m) / (P.fs2 / 1187.5)));
    for (auto &h : st.last_hit)
        h = kRdsNoHit;
    CU(cudaMemcpy(p->d_rds_state.get() + capture, &st, sizeof(st), cudaMemcpyHostToDevice));
    CU(cudaMemset(p->d_rds_dtail.get() + static_cast<size_t>(capture) * p->rds_dtail_len, 0,
                  p->rds_dtail_len * sizeof(float)));
    CU(cudaMemset(p->d_rds_y.get() + static_cast<size_t>(capture) * p->rds_y_len, 0, p->rds_y_len * sizeof(float2)));
    p->rds_read[capture] = 0;
    p->rds_lost[capture] = 0;
    return FMRX_OK;
}

// Copy `rows` rows of `width` bytes between pitched device arrays.
cudaError_t copy2d(void *dst, size_t dpitch, const void *src, size_t spitch, size_t width,
                   size_t rows, cudaStream_t s, cudaMemcpyKind kind = cudaMemcpyDeviceToDevice, size_t max_pitch = 0)
{
    // one row, or a pitch beyond what cudaMemcpy2D takes (cudaDeviceProp::memPitch, ~2 GiB: 7.5 minutes
    // of mode-0 IQ per capture): plain copies, row by row
    if (rows == 1 || (max_pitch && (dpitch > max_pitch || spitch > max_pitch))) {
        for (size_t r = 0; r < rows; r++) {
            cudaError_t e = cudaMemcpyAsync(static_cast<char *>(dst) + r * dpitch, static_cast<const char *>(src) + r * spitch,
                                            width, kind, s);
            if (e != cudaSuccess)
                return e;
        }
        return cudaSuccess;
    }
    return cudaMemcpy2DAsync(dst, dpitch, src, spitch, width, rows, kind, s);
}

// Rows 1 .. rows-1 of a pitched device array, each a copy of the first `width` bytes of row 0: log2(rows) doubling
// copies (what copy2d cannot do: cudaMemcpy2DAsync refuses a source pitch of 0).
cudaError_t broadcast_rows(uint8_t *dst, size_t pitch, size_t width, size_t rows, cudaStream_t s)
{
    cudaError_t e = cudaSuccess;
    for (size_t k = 1; k < rows && e == cudaSuccess; k *= 2)
        e = copy2d(dst + k * pitch, pitch, dst, pitch, width, std::min(k, rows - k), s);
    return e;
}

int reset_state(fmrx_pipeline *p)
{
    const size_t C = p->C;
    const CarryLayout &L = p->carry;
    std::vector<uint8_t> rec(L.pitch, 0);
    std::fill_n(rec.begin(), L.hist_bytes, uint8_t{ 0x80 });      // u8 128 == 0.0f
    std::memcpy(rec.data() + L.pll, kPllInitState, sizeof(kPllInitState));
    // on the front stream, which runs first in every chunk; done before return, since a time shard's hand-off
    // writes into record 0 from another stream
    CU(cudaMemcpyAsync(p->d_carry.get(), rec.data(), L.pitch, cudaMemcpyHostToDevice, p->s_front.get()));
    CU(broadcast_rows(p->d_carry.get(), L.pitch, L.pitch, C, p->s_front.get()));
    CU(cudaStreamSynchronize(p->s_front.get()));
    p->blocks_done.assign(C, 0);
    p->blocks_run = 0;
    for (auto &t : p->tune)
        t.pair_offset = 0;
    CU(cudaMemcpy(p->d_tune.get(), p->tune.data(), C * sizeof(RfTune), cudaMemcpyHostToDevice));
    for (size_t c = 0; c < C; c++)
        if (p->rds_on[c]) {
            const int rc = rds_restart(p, static_cast<int>(c));
            if (rc != FMRX_OK)
                return rc;
        }
    return FMRX_OK;
}

// Lazily allocated staging for the host-pointer path.
int ensure_host_staging(fmrx_pipeline *p)
{
    const size_t C = p->C;
    for (auto &s : p->sets) {
        if (!s.iq)
            CU(dalloc(s.iq, C * static_cast<size_t>(p->chunk_blocks) * p->mi.block_size));
        if (!s.pcm)
            CU(dalloc(s.pcm, C * static_cast<size_t>(p->chunk_blocks) * 2 * p->mi.audio_per_block));
    }
    return FMRX_OK;
}

int ensure_stage_storage(fmrx_pipeline *p, size_t n_blocks)
{
    const size_t if_len = n_blocks * p->mi.if_per_block, au_len = n_blocks * p->mi.audio_per_block;
    if (if_len <= p->stage_if_len && au_len <= p->stage_au_len && p->d_stage[0]) {
        p->stage_if_len = if_len;   // logical length of the last call
        p->stage_au_len = au_len;
        return FMRX_OK;
    }
    for (auto &q : p->d_stage)
        q.reset();
    for (int s = 0; s < FMRX_STAGE_COUNT; s++) {
        const size_t len = (s >= FMRX_STAGE_MONO) ? au_len : if_len;
        CU(dalloc(p->d_stage[s], static_cast<size_t>(p->C) * len));
    }
    p->stage_if_len = if_len;
    p->stage_au_len = au_len;
    return FMRX_OK;
}

// The chunk loop shared by the host- and device-pointer entry points.
// feedforward_only: K1 and K2 only -- what a time shard runs over the blocks in FRONT of its own (its halo), from the
// zero state, to arrive at the IQ / demod / channel histories the stream has at the shard's first block.
int run(fmrx_pipeline *p, const uint8_t *iq, size_t iq_stride, size_t n_blocks, int16_t *pcm,
        size_t pcm_stride, bool host_io, cudaStream_t user, bool feedforward_only = false)
{
    const fmrx_mode_info &mi = p->mi;
    const int C = p->C, T = mi.taps, H = p->H;
    const size_t fH = static_cast<size_t>(H) * sizeof(float);
    const size_t if_pitch = p->if_stride * sizeof(float);
    const CarryLayout &L = p->carry;
    uint8_t *const carry = p->d_carry.get();

    if (host_io) {
        const int rc = ensure_host_staging(p);
        if (rc != FMRX_OK) return rc;
    }
    if (p->keep_stages) {
        const int rc = ensure_stage_storage(p, n_blocks);
        if (rc != FMRX_OK) return rc;
    }
    if (!host_io) {
        // order after the caller's stream
        CU(cudaEventRecord(p->ev_in.get(), user));
        CU(cudaStreamWaitEvent(p->s_front.get(), p->ev_in.get(), 0));
        CU(cudaStreamWaitEvent(p->s_pll.get(), p->ev_in.get(), 0));
        CU(cudaStreamWaitEvent(p->s_back.get(), p->ev_in.get(), 0));
    }

    // chunk sizes: with the automatic size a quarter and a half chunk first, so that the pipeline
    // (and, from the host, the first H2D copy) fills quickly
    std::vector<int> chunk_nb;
    for (size_t done = 0; done < n_blocks;) {
        int want = p->chunk_blocks;
        if (p->ramp && chunk_nb.size() == 0)
            want = std::max(1, p->chunk_blocks / 4);
        else if (p->ramp && chunk_nb.size() == 1)
            want = std::max(1, p->chunk_blocks / 2);
        const int nb = static_cast<int>(std::min<size_t>(want, n_blocks - done));
        chunk_nb.push_back(nb);
        done += nb;
    }
    const size_t n_chunks = chunk_nb.size();
    if (p->timing) {
        while (p->tev.size() < p->tev_used + 8 * n_chunks) {
            event_ptr e;
            CU(make_event(e, cudaEventDefault));
            p->tev.push_back(std::move(e));
        }
    }
    const size_t tev0 = p->tev_used;

    size_t b_next = 0;
    for (size_t ci = 0; ci < n_chunks; ci++) {
        const size_t b0 = b_next;
        const int nb = chunk_nb[ci];
        b_next += nb;
        const int n_if = nb * mi.if_per_block;
        const size_t chunk_bytes = static_cast<size_t>(nb) * mi.block_size;
        const size_t chunk_pcm = static_cast<size_t>(nb) * 2 * mi.audio_per_block;
        BufferSet &S = p->sets[p->chunk_counter % p->sets.size()];
        const event_ptr *te = p->timing ? &p->tev[tev0 + 8 * ci] : nullptr;

        // ---------------- front: [H2D] K1 K2 ----------------
        if (S.free_pending)
            CU(cudaStreamWaitEvent(p->s_front.get(), S.free_ev.get(), 0));
        const uint8_t *iq_dev;
        size_t iq_dev_stride;
        if (host_io) {
            iq_dev = S.iq.get();
            // iq_stride 0: every capture reads one stream, which crosses the host link once
            iq_dev_stride = iq_stride ? static_cast<size_t>(p->chunk_blocks) * mi.block_size : 0;
            // on its own stream: the copy of a chunk only waits for the staging buffer (read for the
            // last time by K1 three chunks ago), not for K1/K2 of the chunk before
            if (S.iq_free_pending)
                CU(cudaStreamWaitEvent(p->s_h2d.get(), S.iq_free.get(), 0));
            CU(copy2d(S.iq.get(), iq_dev_stride, iq + b0 * mi.block_size, iq_stride, chunk_bytes, iq_stride ? C : 1,
                      p->s_h2d.get(), cudaMemcpyHostToDevice, p->mem_pitch));
            CU(cudaEventRecord(S.h2d_done.get(), p->s_h2d.get()));
            CU(cudaStreamWaitEvent(p->s_front.get(), S.h2d_done.get(), 0));
        } else {
            iq_dev = iq + b0 * mi.block_size;
            iq_dev_stride = iq_stride;
        }
        if (te) CU(cudaEventRecord(te[0].get(), p->s_front.get()));
        CU(copy2d(S.demod.get(), if_pitch, carry + L.demod, L.pitch, fH, C, p->s_front.get()));
        CU(copy2d(S.chan.get(), if_pitch, carry + L.chan, L.pitch, fH, C, p->s_front.get()));
        {
            RfDemodArgs a{};
            a.iq = iq_dev;
            a.iq_stride = iq_dev_stride;
            a.hist = carry;
            a.hist_pairs = p->hist_pairs;
            a.hist_stride = static_cast<int>(L.pitch);
            a.taps = p->d_rf_taps.get();
            a.T = T;
            a.decim = mi.rf_decim;
            a.n_if = n_if;
            a.demod = S.demod.get();
            a.if_stride = p->if_stride;
            a.if_off = H;
            if (p->keep_stages) {
                a.i_ds = p->d_stage[FMRX_STAGE_I_DS].get();
                a.q_ds = p->d_stage[FMRX_STAGE_Q_DS].get();
                a.stage_stride = p->stage_if_len;
                a.stage_off = b0 * mi.if_per_block;
            }
            const RfTuneArgs tu{ p->d_tune_cs.get(), p->d_tune.get(), p->blocks_run * (mi.block_size / 2) };
            CU(launch_rf_demod(a, C, p->s_front.get(), p->tuned ? &tu : nullptr));
            p->launches++;
        }
        if (te) CU(cudaEventRecord(te[1].get(), p->s_front.get()));
        // IQ history for the next chunk: the last hist_pairs pairs of this chunk (per capture, also when the
        // captures share one stream: state blobs are per capture)
        CU(copy2d(carry, L.pitch, iq_dev + chunk_bytes - L.hist_bytes, iq_dev_stride, L.hist_bytes, iq_dev_stride ? C : 1,
                  p->s_front.get()));
        if (!iq_dev_stride)
            CU(broadcast_rows(carry, L.pitch, L.hist_bytes, C, p->s_front.get()));
        if (host_io) {
            CU(cudaEventRecord(S.iq_free.get(), p->s_front.get()));
            S.iq_free_pending = true;
        }
        {
            BandpassArgs a{};
            a.demod = S.demod.get();
            a.if_stride = p->if_stride;
            a.if_off = H;
            a.taps_pilot = p->d_pilot_taps.get();
            a.taps_chan = p->d_chan_taps.get();
            a.T = T;
            a.n_if = n_if;
            a.pilot = S.pilot.get();
            a.pilot_stride = p->chunk_if;
            a.chan = S.chan.get();
            CU(launch_bandpass_pair(a, C, p->s_front.get()));
            p->launches++;
        }
        if (te) CU(cudaEventRecord(te[2].get(), p->s_front.get()));
        // tails for the next chunk's front stage
        CU(copy2d(carry + L.demod, L.pitch, S.demod.get() + n_if, if_pitch, fH, C, p->s_front.get()));
        CU(copy2d(carry + L.chan, L.pitch, S.chan.get() + n_if, if_pitch, fH, C, p->s_front.get()));
        CU(cudaEventRecord(S.front_done.get(), p->s_front.get()));
        if (!p->rds_caps.empty() && !feedforward_only) {
            // RDS beside K3: on the front stream after front_done, so that K3 does not wait for it
            const long long if_run = p->blocks_run * mi.if_per_block;
            RdsBasebandArgs b{};
            b.prm = p->rds_prm;
            b.caps = p->d_rds_caps.get();
            b.state = p->d_rds_state.get();
            b.demod = S.demod.get();
            b.if_stride = p->if_stride;
            b.if_off = H;
            b.n_if = n_if;
            b.if_run = if_run;
            b.dtail = p->d_rds_dtail.get();
            b.dtail_len = p->rds_dtail_len;
            b.taps = p->d_rds_taps.get();
            b.mix = p->d_rds_mix.get();
            b.ybuf = p->d_rds_y.get();
            b.ybuf_len = p->rds_y_len;
            b.ytail_len = p->rds_ytail_len;
            RdsBitsArgs r{};
            r.prm = p->rds_prm;
            r.caps = p->d_rds_caps.get();
            r.state = p->d_rds_state.get();
            r.n_if = n_if;
            r.if_run = if_run;
            r.ybuf = p->d_rds_y.get();
            r.ybuf_len = p->rds_y_len;
            r.ytail_len = p->rds_ytail_len;
            r.bitphase = p->d_rds_phase.get();
            r.ring = p->d_rds_ring.get();
            CU(launch_rds(b, r, static_cast<int>(p->rds_caps.size()), p->s_front.get()));
            p->launches += 2;
            const size_t dt = static_cast<size_t>(p->rds_dtail_len) * sizeof(float);
            CU(copy2d(p->d_rds_dtail.get(), dt, S.demod.get() + H + n_if - p->rds_dtail_len, if_pitch, dt, C,
                      p->s_front.get()));
        }
        if (feedforward_only) {
            CU(cudaEventRecord(S.free_ev.get(), p->s_front.get()));
            S.free_pending = true;
            p->chunk_counter++;
            continue;
        }

        // ---------------- pll: K3 ----------------
        CU(cudaStreamWaitEvent(p->s_pll.get(), S.front_done.get(), 0));
        CU(copy2d(S.trig.get(), if_pitch, carry + L.trig, L.pitch, fH, C, p->s_pll.get()));
        if (te) CU(cudaEventRecord(te[3].get(), p->s_pll.get()));
        {
            PllArgs a{};
            a.pilot = S.pilot.get();
            a.pilot_stride = p->chunk_if;
            a.trig = S.trig.get();
            a.if_stride = p->if_stride;
            a.if_off = H;
            a.n_if = n_if;
            a.state = reinterpret_cast<float *>(carry + L.pll);
            a.state_stride = static_cast<int>(L.pitch / sizeof(float));
            a.prm = p->pll_prm;
            CU(launch_pll(a, C, p->s_pll.get()));
            p->launches++;
        }
        if (te) CU(cudaEventRecord(te[4].get(), p->s_pll.get()));
        CU(copy2d(carry + L.trig, L.pitch, S.trig.get() + n_if, if_pitch, fH, C, p->s_pll.get()));
        CU(cudaEventRecord(S.pll_done.get(), p->s_pll.get()));

        // ---------------- back: K4 [D2H] ----------------
        CU(cudaStreamWaitEvent(p->s_back.get(), S.pll_done.get(), 0));
        if (te) CU(cudaEventRecord(te[5].get(), p->s_back.get()));
        {
            AudioArgs a{};
            a.demod = S.demod.get();
            a.chan = S.chan.get();
            a.trig = S.trig.get();
            a.if_stride = p->if_stride;
            a.if_off = H;
            a.coef_pm = p->d_audio_pm.get();
            a.T = T;
            a.U = mi.audio_interp;
            a.D = mi.audio_decim;
            a.if_per_block = mi.if_per_block;
            a.audio_per_block = mi.audio_per_block;
            a.n_blocks = nb;
            a.scale = p->pll_prm.scale;
            a.adjust = p->pll_prm.adjust;
            if (host_io) {
                a.pcm = S.pcm.get();
                a.pcm_stride = static_cast<size_t>(p->chunk_blocks) * 2 * mi.audio_per_block;
            } else {
                a.pcm = pcm + b0 * 2 * mi.audio_per_block;
                a.pcm_stride = pcm_stride;
            }
            if (p->keep_stages) {
                a.nco = p->d_stage[FMRX_STAGE_NCO].get();
                a.mixer = p->d_stage[FMRX_STAGE_MIXER].get();
                a.if_stage_stride = p->stage_if_len;
                a.if_stage_off = b0 * mi.if_per_block;
                a.mono = p->d_stage[FMRX_STAGE_MONO].get();
                a.mono_shift = p->d_stage[FMRX_STAGE_MONO_SHIFT].get();
                a.stereo = p->d_stage[FMRX_STAGE_STEREO].get();
                a.left = p->d_stage[FMRX_STAGE_LEFT].get();
                a.right = p->d_stage[FMRX_STAGE_RIGHT].get();
                a.au_stage_stride = p->stage_au_len;
                a.au_stage_off = b0 * mi.audio_per_block;
            }
            CU(launch_audio(a, C, p->s_back.get()));
            p->launches++;
        }
        if (te) CU(cudaEventRecord(te[6].get(), p->s_back.get()));
        if (p->keep_stages) {
            const size_t w = static_cast<size_t>(n_if) * sizeof(float);
            const size_t dp = p->stage_if_len * sizeof(float);
            const size_t off = b0 * mi.if_per_block;
            CU(copy2d(p->d_stage[FMRX_STAGE_DEMOD].get() + off, dp, S.demod.get() + H, if_pitch, w, C, p->s_back.get()));
            CU(copy2d(p->d_stage[FMRX_STAGE_CHAN].get() + off, dp, S.chan.get() + H, if_pitch, w, C, p->s_back.get()));
            CU(copy2d(p->d_stage[FMRX_STAGE_TRIG].get() + off, dp, S.trig.get() + H, if_pitch, w, C, p->s_back.get()));
            CU(copy2d(p->d_stage[FMRX_STAGE_PILOT].get() + off, dp, S.pilot.get(),
                      static_cast<size_t>(p->chunk_if) * sizeof(float), w, C, p->s_back.get()));
        }
        if (host_io)
            CU(copy2d(pcm + b0 * 2 * mi.audio_per_block, pcm_stride * sizeof(int16_t), S.pcm.get(),
                      static_cast<size_t>(p->chunk_blocks) * 2 * mi.audio_per_block * sizeof(int16_t),
                      chunk_pcm * sizeof(int16_t), C, p->s_back.get(), cudaMemcpyDeviceToHost, p->mem_pitch));
        if (te) CU(cudaEventRecord(te[7].get(), p->s_back.get()));
        CU(cudaEventRecord(S.free_ev.get(), p->s_back.get()));
        S.free_pending = true;

        for (auto &bd : p->blocks_done)
            bd += nb;
        p->blocks_run += nb;
        p->chunk_counter++;
    }

    if (host_io) {
        CU(cudaStreamSynchronize(p->s_back.get()));
        CU(cudaStreamSynchronize(p->s_pll.get()));
        CU(cudaStreamSynchronize(p->s_front.get()));
    } else {
        CU(cudaEventRecord(p->ev_out.get(), p->s_back.get()));
        CU(cudaStreamWaitEvent(user, p->ev_out.get(), 0));
        CU(cudaEventRecord(p->ev_out.get(), p->s_pll.get()));
        CU(cudaStreamWaitEvent(user, p->ev_out.get(), 0));
        CU(cudaEventRecord(p->ev_out.get(), p->s_front.get()));
        CU(cudaStreamWaitEvent(user, p->ev_out.get(), 0));
    }
    if (p->timing)
        p->tev_used = tev0 + 8 * n_chunks;
    return FMRX_OK;
}

int check_io(const fmrx_pipeline *p, const void *iq, size_t iq_stride, size_t n_blocks,
             const void *pcm, size_t pcm_stride)
{
    if (!p || !iq || !pcm)
        return FMRX_ERR_ARG;
    const size_t need_iq = n_blocks * p->mi.block_size;
    const size_t need_pcm = n_blocks * 2 * p->mi.audio_per_block;
    // K1 reads IQ pairs as 16-bit words, K4 writes R,L frames as 32-bit words
    if ((reinterpret_cast<uintptr_t>(iq) & 1u) || (reinterpret_cast<uintptr_t>(pcm) & 3u))
        return FMRX_ERR_ARG;
    // the strides only matter with more than one capture (a single capture may be a truncated file of
    // any length: the trailing partial block is the caller's to drop); iq_stride 0 = one stream for all
    if (p->C > 1 && ((iq_stride && iq_stride < need_iq) || pcm_stride < need_pcm || (iq_stride & 1u) || (pcm_stride & 1u)))
        return FMRX_ERR_ARG;
    return FMRX_OK;
}

}  // namespace

extern "C" int fmrx_create(fmrx_pipeline **out, const fmrx_config *cfg)
{
    if (!out || !cfg || cfg->n_captures < 1 || cfg->n_captures > 65535)   // captures are gridDim.y of K1, K2, K4
        return FMRX_ERR_ARG;
    for (int r : cfg->reserved)
        if (r != 0)
            return FMRX_ERR_ARG;
    if (cfg->n_sets < 0 || cfg->n_sets == 1 || cfg->n_sets > 64)
        return FMRX_ERR_ARG;
    *out = nullptr;
    fmrx_mode_info mi;
    if (fmrx_mode_table(cfg->mode, cfg->taps, &mi) != FMRX_OK)
        return FMRX_ERR_ARG;
    int dev = cfg->device;
    size_t mem_pitch = 0;
    const int rc = open_device(dev, &mem_pitch);
    if (rc != FMRX_OK)
        return rc;
    std::unique_ptr<fmrx_pipeline> p(new (std::nothrow) fmrx_pipeline());
    if (!p)
        return FMRX_ERR_ALLOC;
    p->mi = mi;
    p->device = dev;
    p->mem_pitch = mem_pitch;
    const int T = mi.taps, U = mi.audio_interp;
    p->C = cfg->n_captures;
    p->keep_stages = cfg->keep_stages != 0;
    p->sets.resize(cfg->n_sets > 0 ? cfg->n_sets : kDefaultSets);
    const size_t C = p->C;

    const PipelineSizes sz = pipeline_sizes(mi);
    p->H = sz.H;
    p->hist_pairs = T - 1 + mi.rf_decim;
    if (mi.if_per_block < p->H || mi.block_size / 2 < p->hist_pairs)
        return FMRX_ERR_ARG;
    p->carry = carry_layout(p->hist_pairs, p->H);
    const long long cb_max = sz.max_chunk_blocks;
    if (cb_max < 1)
        return FMRX_ERR_ARG;
    int cb = static_cast<int>(std::min<long long>(cfg->chunk_blocks, cb_max));
    if (cb <= 0) {
        // aim at ~256 MiB per IF-rate array per chunk: a K3 launch has to wait for whole SMs to drain
        // of the FIR CTAs of the neighbouring chunks (its CTAs claim a whole SM each), a third of a
        // millisecond that is 12 % of a launch at 32 MiB, 3 % at 128 and 1.5 % at 256
        const size_t target_if = (256u << 20) / sizeof(float) / C;
        cb = static_cast<int>(std::max<size_t>(1, target_if / mi.if_per_block));
        cb = static_cast<int>(std::min<long long>(std::min(cb, 8192), cb_max));
    }
    p->ramp = cfg->chunk_blocks <= 0;
    p->chunk_blocks = cb;
    p->chunk_if = cb * mi.if_per_block;
    p->if_stride = static_cast<size_t>(p->H) + p->chunk_if;

    // filters (src/project.cpp:37,97,104,117)
    std::vector<float> rf(T), pil(T), ch(T), au(mi.audio_taps), au_pm(mi.audio_taps);
    fmrx_impulse_response_lpf(rf.data(), static_cast<float>(mi.rf_fs), 100000.0f, T, 1);
    fmrx_impulse_response_bpf(ch.data(), static_cast<float>(mi.bp_fs), 22000.0f, 54000.0f, T);
    fmrx_impulse_response_bpf(pil.data(), static_cast<float>(mi.bp_fs), 18500.0f, 19500.0f, T);
    fmrx_impulse_response_lpf(au.data(), static_cast<float>(mi.if_fs), 16000.0f, mi.audio_taps, U);
    for (int ph = 0; ph < U; ph++)
        for (int t = 0; t < T; t++)
            au_pm[static_cast<size_t>(ph) * T + t] = au[ph + static_cast<size_t>(t) * U];
    // src/project.cpp:166: PLL(19000, if_fs, 2, 0, 0.01)
    p->pll_prm = make_pll_params(19000.0f, static_cast<float>(mi.if_fs), 2.0f, 0.0f, 0.01f);

    CU(dalloc(p->d_rf_taps, T));
    CU(dalloc(p->d_pilot_taps, T));
    CU(dalloc(p->d_chan_taps, T));
    CU(dalloc(p->d_audio_pm, au_pm.size()));
    CU(cudaMemcpy(p->d_rf_taps.get(), rf.data(), T * sizeof(float), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(p->d_pilot_taps.get(), pil.data(), T * sizeof(float), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(p->d_chan_taps.get(), ch.data(), T * sizeof(float), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(p->d_audio_pm.get(), au_pm.data(), au_pm.size() * sizeof(float), cudaMemcpyHostToDevice));

    CU(dalloc(p->d_carry, C * p->carry.pitch));
    CU(dalloc(p->d_tune, C));
    p->tune.assign(C, RfTune{ 0, 0 });
    p->rds_on.assign(C, 0);
    p->rds_read.assign(C, 0);
    p->rds_lost.assign(C, 0);
    for (auto &s : p->sets) {
        CU(dalloc(s.demod, C * p->if_stride));
        CU(dalloc(s.chan, C * p->if_stride));
        CU(dalloc(s.trig, C * p->if_stride));
        CU(dalloc(s.pilot, C * static_cast<size_t>(p->chunk_if)));
        CU(make_event(s.front_done));
        CU(make_event(s.pll_done));
        CU(make_event(s.free_ev));
        CU(make_event(s.h2d_done));
        CU(make_event(s.iq_free));
    }
    int lo = 0, hi = 0;
    CU(cudaDeviceGetStreamPriorityRange(&lo, &hi));
    CU(make_stream(p->s_front, lo));
    CU(make_stream(p->s_pll, hi));   // the long pole first
    CU(make_stream(p->s_back, lo));
    CU(make_stream(p->s_h2d, lo));
    CU(make_event(p->ev_in));
    CU(make_event(p->ev_out));
    const int rs = reset_state(p.get());
    if (rs != FMRX_OK)
        return rs;
    *out = p.release();
    return FMRX_OK;
}

extern "C" int fmrx_destroy(fmrx_pipeline *p)
{
    delete p;
    return FMRX_OK;
}

extern "C" int fmrx_info(const fmrx_pipeline *p, fmrx_mode_info *out)
{
    if (!p || !out)
        return FMRX_ERR_ARG;
    *out = p->mi;
    return FMRX_OK;
}

extern "C" int fmrx_reset(fmrx_pipeline *p)
{
    if (!p)
        return FMRX_ERR_ARG;
    CU(cudaSetDevice(p->device));
    CU(cudaDeviceSynchronize());
    return reset_state(p);
}

extern "C" int fmrx_process(fmrx_pipeline *p, const uint8_t *iq, size_t iq_stride, size_t n_blocks,
                            int16_t *pcm, size_t pcm_stride)
{
    if (n_blocks == 0)
        return p ? FMRX_OK : FMRX_ERR_ARG;
    const int rc = check_io(p, iq, iq_stride, n_blocks, pcm, pcm_stride);
    if (rc != FMRX_OK)
        return rc;
    CU(cudaSetDevice(p->device));
    if (p->C == 1) {
        iq_stride = n_blocks * p->mi.block_size;
        pcm_stride = n_blocks * 2 * p->mi.audio_per_block;
    }
    return run(p, iq, iq_stride, n_blocks, pcm, pcm_stride, true, nullptr);
}

extern "C" int fmrx_process_device(fmrx_pipeline *p, const uint8_t *iq_dev, size_t iq_stride,
                                   size_t n_blocks, int16_t *pcm_dev, size_t pcm_stride, void *stream)
{
    if (n_blocks == 0)
        return p ? FMRX_OK : FMRX_ERR_ARG;
    const int rc = check_io(p, iq_dev, iq_stride, n_blocks, pcm_dev, pcm_stride);
    if (rc != FMRX_OK)
        return rc;
    CU(cudaSetDevice(p->device));
    if (p->C == 1) {
        iq_stride = n_blocks * p->mi.block_size;
        pcm_stride = n_blocks * 2 * p->mi.audio_per_block;
    }
    return run(p, iq_dev, iq_stride, n_blocks, pcm_dev, pcm_stride, false,
               static_cast<cudaStream_t>(stream));
}

extern "C" int fmrx_read_stage(fmrx_pipeline *p, int stage, int capture, float *out, size_t n,
                               size_t *n_out)
{
    if (!p || stage < 0 || stage >= FMRX_STAGE_COUNT || capture < 0 || capture >= p->C || !out)
        return FMRX_ERR_ARG;
    if (!p->keep_stages || !p->d_stage[stage])
        return FMRX_ERR_STATE;
    CU(cudaSetDevice(p->device));
    CU(cudaDeviceSynchronize());
    const size_t len = (stage >= FMRX_STAGE_MONO) ? p->stage_au_len : p->stage_if_len;
    const size_t k = std::min(n, len);
    if (k)
        CU(cudaMemcpy(out, p->d_stage[stage].get() + static_cast<size_t>(capture) * len, k * sizeof(float),
                      cudaMemcpyDeviceToHost));
    if (n_out)
        *n_out = k;
    return FMRX_OK;
}

extern "C" size_t fmrx_state_size(const fmrx_pipeline *p)
{
    if (!p)
        return 0;
    return sizeof(StateHeader) + p->carry.body;
}

extern "C" int fmrx_get_state(fmrx_pipeline *p, int capture, void *blob, size_t blob_size)
{
    if (!p || !blob || capture < 0 || capture >= p->C || blob_size < fmrx_state_size(p))
        return FMRX_ERR_ARG;
    CU(cudaSetDevice(p->device));
    CU(cudaDeviceSynchronize());
    const CarryLayout &L = p->carry;
    StateHeader h{ kStateMagic, static_cast<uint32_t>(p->mi.mode), static_cast<uint32_t>(p->mi.taps),
                   static_cast<uint32_t>(p->H), static_cast<uint32_t>(p->hist_pairs), 0, p->blocks_done[capture] };
    std::memcpy(blob, &h, sizeof(h));
    uint8_t *b = static_cast<uint8_t *>(blob) + sizeof(h);
    CU(cudaMemcpy(b, p->d_carry.get() + capture * L.pitch, L.body, cudaMemcpyDeviceToHost));
    // the padding after the IQ history is not state: zeros, whatever a blob given to fmrx_set_state held there
    std::memset(b + L.hist_bytes, 0, L.demod - L.hist_bytes);
    return FMRX_OK;
}

extern "C" int fmrx_set_state(fmrx_pipeline *p, int capture, const void *blob, size_t blob_size,
                              int parts)
{
    if (!p || !blob || capture < 0 || capture >= p->C || blob_size < fmrx_state_size(p) ||
        !(parts & FMRX_STATE_ALL))
        return FMRX_ERR_ARG;
    const uint8_t *b = static_cast<const uint8_t *>(blob);
    StateHeader h;
    std::memcpy(&h, b, sizeof(h));
    if (h.magic != kStateMagic || h.mode != static_cast<uint32_t>(p->mi.mode) ||
        h.taps != static_cast<uint32_t>(p->mi.taps) || h.hist_if != static_cast<uint32_t>(p->H) ||
        h.hist_pairs != static_cast<uint32_t>(p->hist_pairs))
        return FMRX_ERR_STATE;
    CU(cudaSetDevice(p->device));
    CU(cudaDeviceSynchronize());
    b += sizeof(h);
    uint8_t *rec = p->d_carry.get() + capture * p->carry.pitch;
    const ByteRange &ff = p->carry.feedforward, &pll = p->carry.pll_part;
    if (parts & FMRX_STATE_FEEDFORWARD)
        CU(cudaMemcpy(rec + ff.off, b + ff.off, ff.len, cudaMemcpyHostToDevice));
    if (parts & FMRX_STATE_PLL) {
        CU(cudaMemcpy(rec + pll.off, b + pll.off, pll.len, cudaMemcpyHostToDevice));
        p->blocks_done[capture] = h.blocks_done;
        p->tune[capture].pair_offset = (h.blocks_done - p->blocks_run) * (p->mi.block_size / 2);
        CU(cudaMemcpy(p->d_tune.get() + capture, &p->tune[capture], sizeof(RfTune), cudaMemcpyHostToDevice));
    }
    if (p->rds_on[capture])
        return rds_restart(p, capture);
    return FMRX_OK;
}

extern "C" int fmrx_set_rds(fmrx_pipeline *p, int capture, int enable)
{
    if (!p || capture < 0 || capture >= p->C || (enable != 0 && enable != 1))
        return FMRX_ERR_ARG;
    if (p->blocks_done[capture] != 0)
        return FMRX_ERR_STATE;
    CU(cudaSetDevice(p->device));
    CU(cudaDeviceSynchronize());   // the RDS kernels of calls still in flight read d_rds_caps
    const size_t C = p->C;
    if (enable && !p->d_rds_state) {
        const RdsParams P = rds_params(p->mi.bp_fs);
        std::vector<float> taps(P.taps);
        std::vector<float2> mix(P.P);
        std::vector<double2> ph(P.Q);
        rds_tables(P, taps.data(), mix.data(), ph.data());
        // demod history: the FIR input of the first u a tile needs; y history: two windows and a bit of slack
        // (the bits still to be decided lie at most two windows back)
        const int dtail = ((2 * P.L + 1) * P.D + P.taps + 31) / 32 * 32;
        const int ytail = 2 * P.M + 64;
        const size_t y_len = ytail + static_cast<size_t>(p->chunk_if) / P.D + 2;
        if (dtail > p->mi.if_per_block)
            return FMRX_ERR_ARG;
        CU(dalloc(p->d_rds_taps, taps.size()));
        CU(dalloc(p->d_rds_mix, mix.size()));
        CU(dalloc(p->d_rds_phase, ph.size()));
        CU(dalloc(p->d_rds_dtail, C * dtail));
        CU(dalloc(p->d_rds_y, C * y_len));
        CU(dalloc(p->d_rds_ring, C * kRdsRing));
        CU(dalloc(p->d_rds_caps, C));
        CU(cudaMemcpy(p->d_rds_taps.get(), taps.data(), taps.size() * sizeof(float), cudaMemcpyHostToDevice));
        CU(cudaMemcpy(p->d_rds_mix.get(), mix.data(), mix.size() * sizeof(float2), cudaMemcpyHostToDevice));
        CU(cudaMemcpy(p->d_rds_phase.get(), ph.data(), ph.size() * sizeof(double2), cudaMemcpyHostToDevice));
        CU(dalloc(p->d_rds_state, C));     // last: it marks the decoder's buffers as present
        p->rds_prm = P;
        p->rds_dtail_len = dtail;
        p->rds_ytail_len = ytail;
        p->rds_y_len = y_len;
    }
    p->rds_on[capture] = enable;
    p->rds_caps.clear();
    for (size_t c = 0; c < C; c++)
        if (p->rds_on[c])
            p->rds_caps.push_back(static_cast<int>(c));
    if (!p->rds_caps.empty())
        CU(cudaMemcpy(p->d_rds_caps.get(), p->rds_caps.data(), p->rds_caps.size() * sizeof(int),
                      cudaMemcpyHostToDevice));
    return enable ? rds_restart(p, capture) : FMRX_OK;
}

extern "C" int fmrx_read_rds(fmrx_pipeline *p, int capture, fmrx_rds_group *out, size_t max, size_t *n_out,
                             uint64_t *n_lost)
{
    if (!p || capture < 0 || capture >= p->C || !out || !n_out)
        return FMRX_ERR_ARG;
    *n_out = 0;
    if (n_lost)
        *n_lost = p->rds_lost[capture];
    if (!p->rds_on[capture])
        return FMRX_OK;
    CU(cudaSetDevice(p->device));
    CU(cudaStreamSynchronize(p->s_front.get()));
    uint64_t written = 0;
    CU(cudaMemcpy(&written, &p->d_rds_state.get()[capture].written, sizeof(written), cudaMemcpyDeviceToHost));
    uint64_t &rd = p->rds_read[capture];
    if (written - rd > static_cast<uint64_t>(kRdsRing)) {
        p->rds_lost[capture] += written - rd - kRdsRing;
        rd = written - kRdsRing;
    }
    const fmrx_rds_group *ring = p->d_rds_ring.get() + static_cast<size_t>(capture) * kRdsRing;
    size_t k = static_cast<size_t>(std::min<uint64_t>(written - rd, max));
    size_t done = 0;
    while (done < k) {
        const size_t at = static_cast<size_t>((rd + done) % kRdsRing);
        const size_t run = std::min(k - done, static_cast<size_t>(kRdsRing) - at);
        CU(cudaMemcpy(out + done, ring + at, run * sizeof(fmrx_rds_group), cudaMemcpyDeviceToHost));
        done += run;
    }
    rd += k;
    *n_out = k;
    if (n_lost)
        *n_lost = p->rds_lost[capture];
    return FMRX_OK;
}

extern "C" int fmrx_rds_probe(fmrx_pipeline *p, int capture, fmrx_rds_probe_info *out, float *y, size_t y_max,
                              size_t *y_n)
{
    if (!p || capture < 0 || capture >= p->C || !out || (!y && y_max))
        return FMRX_ERR_ARG;
    if (!p->rds_on[capture])
        return FMRX_ERR_STATE;
    CU(cudaSetDevice(p->device));
    CU(cudaStreamSynchronize(p->s_front.get()));
    RdsDecState st;
    CU(cudaMemcpy(&st, p->d_rds_state.get() + capture, sizeof(st), cudaMemcpyDeviceToHost));
    const RdsParams &P = p->rds_prm;
    const long long n = p->blocks_done[capture] * p->mi.if_per_block;
    std::memset(out, 0, sizeof(*out));
    out->m_end = static_cast<uint64_t>((n + P.D - 1) / P.D);
    out->w_next = st.w_next;
    out->j = st.j;
    out->nbits = st.nbits;
    out->written = st.written;
    out->reg = st.reg & ((1ull << 52) - 1);
    out->t_prev = st.have_prev ? st.t_prev : std::nan("");
    out->tau = st.w_next > st.w_first ? st.tau[(st.w_next - 1) & 3] : std::nan("");
    out->synced = st.synced;
    // after every chunk the buffer starts with y[m_end - ytail_len .. m_end)
    const size_t k = std::min(y_max, static_cast<size_t>(p->rds_ytail_len));
    if (k)
        CU(cudaMemcpy(y, p->d_rds_y.get() + static_cast<size_t>(capture) * p->rds_y_len + (p->rds_ytail_len - k),
                      k * sizeof(float2), cudaMemcpyDeviceToHost));
    if (y_n)
        *y_n = y_max ? k : static_cast<size_t>(p->rds_ytail_len);
    return FMRX_OK;
}

extern "C" int fmrx_set_tuning(fmrx_pipeline *p, int capture, double offset_hz)
{
    if (!p || capture < 0 || capture >= p->C || !(std::fabs(offset_hz) < 0.5 * p->mi.rf_fs))
        return FMRX_ERR_ARG;
    if (p->blocks_done[capture] != 0)
        return FMRX_ERR_STATE;   // FIR history mixed with another offset: retuning mid-stream is not supported
    const uint32_t inc = static_cast<uint32_t>(std::llrint(offset_hz * 4294967296.0 / p->mi.rf_fs));
    CU(cudaSetDevice(p->device));
    CU(cudaDeviceSynchronize());   // K1 of calls still in flight reads d_tune
    if (inc && !p->d_tune_cs) {
        std::vector<float> cs(2 * 65536);
        mixer_table(cs.data());
        CU(dalloc(p->d_tune_cs, cs.size() / 2));
        CU(cudaMemcpy(p->d_tune_cs.get(), cs.data(), cs.size() * sizeof(float), cudaMemcpyHostToDevice));
    }
    p->tune[capture].inc = inc;
    CU(cudaMemcpy(p->d_tune.get() + capture, &p->tune[capture], sizeof(RfTune), cudaMemcpyHostToDevice));
    p->tuned = std::any_of(p->tune.begin(), p->tune.end(), [](const RfTune &t) { return t.inc != 0; });
    return FMRX_OK;
}

extern "C" int fmrx_get_pll_state(fmrx_pipeline *p, int capture, float out[6])
{
    if (!p || !out || capture < 0 || capture >= p->C)
        return FMRX_ERR_ARG;
    CU(cudaSetDevice(p->device));
    CU(cudaDeviceSynchronize());
    CU(cudaMemcpy(out, p->d_carry.get() + capture * p->carry.pitch + p->carry.pll, 6 * sizeof(float),
                  cudaMemcpyDeviceToHost));
    return FMRX_OK;
}

extern "C" uint64_t fmrx_kernel_launches(const fmrx_pipeline *p) { return p ? p->launches : 0; }

extern "C" int fmrx_set_timing(fmrx_pipeline *p, int enable)
{
    if (!p)
        return FMRX_ERR_ARG;
    p->timing = enable != 0;
    p->tev_used = 0;
    return FMRX_OK;
}

extern "C" int fmrx_last_timing(fmrx_pipeline *p, float out_ms[4])
{
    if (!p || !out_ms)
        return FMRX_ERR_ARG;
    if (p->tev_used) {
        CU(cudaSetDevice(p->device));
        CU(cudaStreamSynchronize(p->s_back.get()));
        CU(cudaStreamSynchronize(p->s_pll.get()));
        CU(cudaStreamSynchronize(p->s_front.get()));
        float acc[4] = { 0, 0, 0, 0 };
        for (size_t i = 0; i < p->tev_used; i += 8) {
            const event_ptr *te = &p->tev[i];
            float ms = 0;
            CU(cudaEventElapsedTime(&ms, te[0].get(), te[1].get())); acc[0] += ms;
            CU(cudaEventElapsedTime(&ms, te[1].get(), te[2].get())); acc[1] += ms;
            CU(cudaEventElapsedTime(&ms, te[3].get(), te[4].get())); acc[2] += ms;
            CU(cudaEventElapsedTime(&ms, te[5].get(), te[6].get())); acc[3] += ms;
        }
        std::memcpy(p->last_ms, acc, sizeof(acc));
        p->tev_used = 0;
    }
    std::memcpy(out_ms, p->last_ms, sizeof(p->last_ms));
    return FMRX_OK;
}

// ---------------------------------------------------------------------------
// One long capture, time-sharded over several devices (SURVEY.md 8(e), BASELINE.json configs[4])
// ---------------------------------------------------------------------------
//
// The capture is cut into consecutive runs of whole blocks, one per device.  What shards in time is everything
// feed-forward: K1 and K2 have finite memory, so a shard that runs them over a HALO of blocks in front of its own
// (from the zero state) arrives at exactly the IQ / demod / channel histories the stream has at its first block,
// and then runs K1/K2 of its whole shard at once -- every device at the same time, nothing waiting for anybody.
// What does not shard is the PLL recurrence (one dependent chain per capture; speculative restarts never re-merge
// bit for bit: DESIGN.md 4.1): K3 of shard r starts when K3 of shard r-1 has finished, from its state -- the PLL
// scalars and the trigArg history K4's mixer tail needs, ~1.5 KB, moved with cudaMemcpyPeerAsync straight into
// shard r's pipeline and ordered with an event; K4 follows K3 per shard.  The PCM of every shard is gathered on
// the first device with peer copies (NVLink where the devices have it).  All of it is enqueued from one host
// thread without a single host synchronisation until the end.

namespace {
// One shard's resources, on its device
struct TimeShard {
    int device = 0;
    std::unique_ptr<fmrx_pipeline> pipe;
    dptr<int16_t> d_pcm;
    dptr<uint8_t> d_iq;          // host path: halo + shard staged on the device
    event_ptr handed;            // this shard's PLL state has arrived in the next shard's pipeline
    stream_ptr s_io;             // staging copies
    ~TimeShard() { cudaSetDevice(device); }
};
}  // namespace

struct fmrx_long_capture {
    fmrx_mode_info mi{};
    int n = 0;                                   // shards
    size_t n_blocks = 0;
    int halo_blocks = 0;
    std::vector<size_t> first, count;            // blocks of each shard
    std::vector<std::unique_ptr<TimeShard>> shard;
    event_ptr t0, t1;                            // (after `shard`: released before it, with the first device current)
    float last_ms = 0.0f;

    ~fmrx_long_capture()
    {
        if (!shard.empty())
            cudaSetDevice(shard[0]->device);
    }
};

extern "C" int fmrx_long_create(fmrx_long_capture **out, int mode, int taps, int n_shards, const int *devices,
                                size_t n_blocks_total)
{
    if (!out || n_shards < 1 || n_shards > 64 || !devices || n_blocks_total < static_cast<size_t>(n_shards))
        return FMRX_ERR_ARG;
    *out = nullptr;
    fmrx_mode_info mi;
    if (fmrx_mode_table(mode, taps, &mi) != FMRX_OK)
        return FMRX_ERR_ARG;
    std::unique_ptr<fmrx_long_capture> L(new (std::nothrow) fmrx_long_capture());
    if (!L)
        return FMRX_ERR_ALLOC;
    L->mi = mi;
    L->n = n_shards;
    L->n_blocks = n_blocks_total;
    // The halo: IF samples of history the feed-forward stages must have RIGHT at the shard's first block are
    // H (what every IF-rate array keeps in front); the channel filter reaches T-1 further back into demod, the RF
    // filter (T-1)/decim + 2 IF samples further into the IQ (SURVEY.md 8(e)).  In whole blocks:
    const int T = mi.taps;
    const PipelineSizes sz = pipeline_sizes(mi);
    const int need_if = sz.H + (T - 1) + (T - 1) / mi.rf_decim + 2;
    L->halo_blocks = (need_if + mi.if_per_block - 1) / mi.if_per_block;
    const size_t base = n_blocks_total / n_shards, extra = n_blocks_total % n_shards;
    size_t at = 0, longest = 0;
    for (int r = 0; r < n_shards; r++) {
        const size_t cnt = base + (static_cast<size_t>(r) < extra ? 1 : 0);
        L->first.push_back(at);
        L->count.push_back(cnt);
        longest = std::max(longest, cnt);
        at += cnt;
    }
    // chunks as large as a launch may be, and enough buffer sets for the feed-forward stages of the whole shard to
    // run ahead of the PLL
    const size_t target_if = (256u << 20) / sizeof(float);                      // ~256 MiB per IF-rate array per chunk
    const size_t cb = std::max<size_t>(1, std::min<size_t>(std::min<size_t>(static_cast<size_t>(sz.max_chunk_blocks), target_if / mi.if_per_block), longest));
    const int n_sets = static_cast<int>(std::min<size_t>(64, std::max<size_t>(2, (longest + cb - 1) / cb + 1)));
    for (int r = 0; r < n_shards; r++) {
        fmrx_config cfg{};
        cfg.mode = mode;
        cfg.taps = taps;
        cfg.n_captures = 1;
        cfg.device = devices[r];
        cfg.chunk_blocks = static_cast<int>(cb);
        cfg.n_sets = n_sets;
        fmrx_pipeline *pipe = nullptr;
        const int rc = fmrx_create(&pipe, &cfg);
        if (rc != FMRX_OK)
            return rc;
        // (a shard is added once its device is known to be one: it makes that device current when it goes)
        L->shard.emplace_back(new TimeShard{ devices[r], std::unique_ptr<fmrx_pipeline>(pipe) });
        TimeShard &s = *L->shard.back();
        CU(dalloc(s.d_pcm, L->count[r] * 2 * mi.audio_per_block));
        CU(make_event(s.handed));
        CU(make_stream(s.s_io));
        // direct peer copies between neighbouring shards and to the gathering device, where the hardware has them
        for (int o : { r > 0 ? devices[r - 1] : devices[r], devices[0] }) {
            int can = 0;
            if (o != devices[r] && cudaDeviceCanAccessPeer(&can, devices[r], o) == cudaSuccess && can)
                if (cudaDeviceEnablePeerAccess(o, 0) != cudaSuccess)
                    cudaGetLastError();      // (already enabled)
        }
    }
    CU(cudaSetDevice(devices[0]));
    CU(make_event(L->t0, cudaEventDefault));
    CU(make_event(L->t1, cudaEventDefault));
    *out = L.release();
    return FMRX_OK;
}

extern "C" int fmrx_long_destroy(fmrx_long_capture *L)
{
    delete L;
    return FMRX_OK;
}

extern "C" int fmrx_long_shard(const fmrx_long_capture *L, int shard, size_t *first_block, size_t *n_blocks, size_t *halo_blocks)
{
    if (!L || shard < 0 || shard >= L->n)
        return FMRX_ERR_ARG;
    if (first_block) *first_block = L->first[shard];
    if (n_blocks) *n_blocks = L->count[shard];
    if (halo_blocks) *halo_blocks = shard ? std::min<size_t>(L->halo_blocks, L->first[shard]) : 0;
    return FMRX_OK;
}

// iq_dev[r]: on shard r's device, the first HALO block of shard r (block first[r] - halo[r] of the capture), halo
// and shard contiguous.  pcm_dev0: on the first shard's device, the whole capture's PCM.
extern "C" int fmrx_long_process_device(fmrx_long_capture *L, const uint8_t *const *iq_dev, int16_t *pcm_dev0)
{
    if (!L || !iq_dev || !pcm_dev0)
        return FMRX_ERR_ARG;
    const fmrx_mode_info &mi = L->mi;
    const size_t pcm_per_block = 2 * static_cast<size_t>(mi.audio_per_block);
    for (int r = 0; r < L->n; r++) {
        CU(cudaSetDevice(L->shard[r]->device));
        const int rc = fmrx_reset(L->shard[r]->pipe.get());
        if (rc != FMRX_OK)
            return rc;
    }
    CU(cudaSetDevice(L->shard[0]->device));
    CU(cudaEventRecord(L->t0.get(), L->shard[0]->pipe->s_front.get()));
    for (int r = 0; r < L->n; r++) {
        TimeShard &s = *L->shard[r];
        fmrx_pipeline *p = s.pipe.get();
        CU(cudaSetDevice(s.device));
        size_t halo = 0;
        fmrx_long_shard(L, r, nullptr, nullptr, &halo);
        if (!iq_dev[r])
            return FMRX_ERR_ARG;
        // the feed-forward histories at the shard's first block, from the halo (K1, K2 only; front stream)
        if (halo) {
            const int rc = run(p, iq_dev[r], halo * mi.block_size, halo, nullptr, 0, false, p->s_front.get(), true);
            if (rc != FMRX_OK)
                return rc;
        }
        // the PLL-dependent state arrives from shard r-1 (enqueued there, below); K3 and K4 of this shard wait for it,
        // K1 and K2 do not
        if (r > 0) {
            CU(cudaStreamWaitEvent(p->s_pll.get(), L->shard[r - 1]->handed.get(), 0));
            CU(cudaStreamWaitEvent(p->s_back.get(), L->shard[r - 1]->handed.get(), 0));
        }
        // (run() orders its three streams after `user` and makes `user` wait for them: the shard's own I/O stream, so
        // that nothing here waits for anything but what it needs)
        {
            const int rc = run(p, iq_dev[r] + halo * mi.block_size, L->count[r] * mi.block_size, L->count[r], s.d_pcm.get(),
                               L->count[r] * pcm_per_block, false, s.s_io.get());
            if (rc != FMRX_OK)
                return rc;
        }
        // hand the PLL part of the carried state on (what FMRX_STATE_PLL restores): behind this shard's last K3 and
        // its trigArg tail copy on the PLL stream
        if (r + 1 < L->n) {
            const TimeShard &next = *L->shard[r + 1];
            const ByteRange &pll = p->carry.pll_part;
            CU(cudaMemcpyPeerAsync(next.pipe->d_carry.get() + pll.off, next.device, p->d_carry.get() + pll.off, s.device,
                                   pll.len, p->s_pll.get()));
            CU(cudaEventRecord(s.handed.get(), p->s_pll.get()));
        }
        // gather: this shard's PCM to the first device, behind its K4
        CU(cudaMemcpyPeerAsync(pcm_dev0 + L->first[r] * pcm_per_block, L->shard[0]->device, s.d_pcm.get(), s.device,
                               L->count[r] * pcm_per_block * sizeof(int16_t), s.s_io.get()));
    }
    for (int r = 0; r < L->n; r++) {
        CU(cudaSetDevice(L->shard[r]->device));
        CU(cudaStreamSynchronize(L->shard[r]->s_io.get()));
        CU(cudaStreamSynchronize(L->shard[r]->pipe->s_pll.get()));
    }
    CU(cudaSetDevice(L->shard[0]->device));
    CU(cudaEventRecord(L->t1.get(), L->shard[0]->pipe->s_front.get()));
    CU(cudaEventSynchronize(L->t1.get()));
    CU(cudaEventElapsedTime(&L->last_ms, L->t0.get(), L->t1.get()));
    return FMRX_OK;
}

// HOST buffers: the whole capture in, the whole PCM out (pinned buffers make the staging copies asynchronous).
extern "C" int fmrx_long_process(fmrx_long_capture *L, const uint8_t *iq, int16_t *pcm)
{
    if (!L || !iq || !pcm)
        return FMRX_ERR_ARG;
    const fmrx_mode_info &mi = L->mi;
    std::vector<const uint8_t *> ptr(L->n, nullptr);
    for (int r = 0; r < L->n; r++) {
        TimeShard &s = *L->shard[r];
        CU(cudaSetDevice(s.device));
        size_t halo = 0;
        fmrx_long_shard(L, r, nullptr, nullptr, &halo);
        const size_t bytes = (halo + L->count[r]) * mi.block_size;
        if (!s.d_iq)
            CU(dalloc(s.d_iq, bytes));
        CU(cudaMemcpyAsync(s.d_iq.get(), iq + (L->first[r] - halo) * mi.block_size, bytes, cudaMemcpyHostToDevice, s.s_io.get()));
        ptr[r] = s.d_iq.get();
    }
    for (int r = 0; r < L->n; r++) {
        CU(cudaSetDevice(L->shard[r]->device));
        CU(cudaStreamSynchronize(L->shard[r]->s_io.get()));
    }
    CU(cudaSetDevice(L->shard[0]->device));
    dptr<int16_t> d_all;
    const size_t n_pcm = L->n_blocks * 2 * mi.audio_per_block;
    CU(dalloc(d_all, n_pcm));
    const int rc = fmrx_long_process_device(L, ptr.data(), d_all.get());
    if (rc != FMRX_OK)
        return rc;
    CU(cudaMemcpy(pcm, d_all.get(), n_pcm * sizeof(int16_t), cudaMemcpyDeviceToHost));
    return FMRX_OK;
}

/* Device time of the last fmrx_long_process_device call: from the first enqueue to the gathered PCM. */
extern "C" int fmrx_long_last_ms(const fmrx_long_capture *L, float *ms)
{
    if (!L || !ms)
        return FMRX_ERR_ARG;
    *ms = L->last_ms;
    return FMRX_OK;
}

extern "C" int fmrx_long_pll_state(fmrx_long_capture *L, float out[6])
{
    if (!L || !out)
        return FMRX_ERR_ARG;
    return fmrx_get_pll_state(L->shard.back()->pipe.get(), 0, out);
}

// ---------------------------------------------------------------------------
// The reference's RDS sketch (src/project.cpp:200-271)
// ---------------------------------------------------------------------------
// rds_thread is compiled into the reference but never started: channel extraction (54-60 kHz band-pass of the
// demodulated FM), squarer, 113.5-114.5 kHz band-pass, PLL(114000, bp_fs, 0.5, 0, 0.01), a delay of channel_delay
// samples on the channel, mixer -- and there the sketch ends (the 3 kHz low-pass is designed, :231, never applied).
// The same steps on the device, per call = per block of demodulated samples, with the carried states of
// :207-224 in device memory: the operator FIR kernel (k_resample), k_pll unchanged with the sketch's parameters,
// and two element-wise kernels.
struct fmrx_rds {
    int device = 0, taps = 0, delay = 0;
    float fs = 0;
    PllParams prm{};
    dptr<float> d_extract, d_carrier;         // taps
    dptr<float> d_chan_state, d_car_state;    // taps-1
    dptr<float> d_shift_state;                // delay
    dptr<float> d_pll_state;                  // 8
    dptr<float> d_buf;                        // 6 arrays of cap floats: demod, chan, sq, car, trig, out
    size_t cap = 0;

    ~fmrx_rds()
    {
        cudaSetDevice(device);
        cudaDeviceSynchronize();
    }
};

namespace {
int rds_reset_state(fmrx_rds *r)
{
    CU(cudaMemset(r->d_chan_state.get(), 0, (r->taps - 1) * sizeof(float)));      // :209
    CU(cudaMemset(r->d_car_state.get(), 0, (r->taps - 1) * sizeof(float)));       // :216
    CU(cudaMemset(r->d_shift_state.get(), 0, std::max(1, r->delay) * sizeof(float)));   // :207
    CU(cudaMemcpy(r->d_pll_state.get(), kPllInitState, sizeof(kPllInitState), cudaMemcpyHostToDevice));   // :219-224
    return FMRX_OK;
}
}  // namespace

extern "C" int fmrx_rds_create(fmrx_rds **out, float bp_fs, int taps, int channel_delay, int device)
{
    if (!out || taps < 2 || taps > kMaxTaps || channel_delay < 0 || !(bp_fs > 0))
        return FMRX_ERR_ARG;
    *out = nullptr;
    const int rc = open_device(device);
    if (rc != FMRX_OK)
        return rc;
    std::unique_ptr<fmrx_rds> r(new (std::nothrow) fmrx_rds());
    if (!r)
        return FMRX_ERR_ALLOC;
    r->device = device;
    r->taps = taps;
    r->delay = channel_delay;
    r->fs = bp_fs;
    r->prm = make_pll_params(114000.0f, bp_fs, 0.5f, 0.0f, 0.01f);              // :256
    std::vector<float> ex(taps), ca(taps);
    fmrx_impulse_response_bpf(ex.data(), bp_fs, 54000.0f, 60000.0f, taps);      // :210
    fmrx_impulse_response_bpf(ca.data(), bp_fs, 113500.0f, 114500.0f, taps);    // :217
    CU(dalloc(r->d_extract, taps));
    CU(dalloc(r->d_carrier, taps));
    CU(dalloc(r->d_chan_state, taps - 1));
    CU(dalloc(r->d_car_state, taps - 1));
    CU(dalloc(r->d_shift_state, std::max(1, channel_delay)));
    CU(dalloc(r->d_pll_state, 8));
    CU(cudaMemcpy(r->d_extract.get(), ex.data(), taps * sizeof(float), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(r->d_carrier.get(), ca.data(), taps * sizeof(float), cudaMemcpyHostToDevice));
    const int rs = rds_reset_state(r.get());
    if (rs != FMRX_OK)
        return rs;
    *out = r.release();
    return FMRX_OK;
}

extern "C" int fmrx_rds_destroy(fmrx_rds *r)
{
    delete r;
    return FMRX_OK;
}

extern "C" int fmrx_rds_reset(fmrx_rds *r)
{
    if (!r)
        return FMRX_ERR_ARG;
    CU(cudaSetDevice(r->device));
    CU(cudaDeviceSynchronize());
    return rds_reset_state(r);
}

extern "C" int fmrx_rds_process(fmrx_rds *r, const float *demod, size_t n, float *mixer_out, float *channel_out,
                                float *carrier_out)
{
    if (!r || !demod || !mixer_out || n > 0x7fffffffu)
        return FMRX_ERR_ARG;
    // the reference's own code needs a block at least as long as its filters and its delay (:99-100, :263)
    if (n < static_cast<size_t>(r->taps - 1) || n < static_cast<size_t>(r->delay))
        return FMRX_ERR_ARG;
    CU(cudaSetDevice(r->device));
    if (n > r->cap) {
        r->cap = 0;
        CU(dalloc(r->d_buf, 6 * n));
        r->cap = n;
    }
    float *d_demod = r->d_buf.get(), *d_chan = d_demod + r->cap, *d_sq = d_chan + r->cap, *d_car = d_sq + r->cap,
          *d_trig = d_car + r->cap, *d_out = d_trig + r->cap;
    const int ni = static_cast<int>(n), T = r->taps;
    const size_t t1 = static_cast<size_t>(T - 1) * sizeof(float);
    CU(cudaMemcpy(d_demod, demod, n * sizeof(float), cudaMemcpyHostToDevice));
    CU(launch_resample(d_chan, ni, r->d_chan_state.get(), T - 1, d_demod, ni, r->d_extract.get(), T, 1, 1, 0));      // :244
    CU(cudaMemcpyAsync(r->d_chan_state.get(), d_demod + (n - (T - 1)), t1, cudaMemcpyDeviceToDevice, 0));      // filter.cpp:95-102
    CU(launch_square(d_sq, d_chan, n, 0));                                                               // :249-251
    CU(launch_resample(d_car, ni, r->d_car_state.get(), T - 1, d_sq, ni, r->d_carrier.get(), T, 1, 1, 0));           // :254
    CU(cudaMemcpyAsync(r->d_car_state.get(), d_sq + (n - (T - 1)), t1, cudaMemcpyDeviceToDevice, 0));
    if (carrier_out)         // (the band-passed carrier, before the PLL overwrites it with its NCO output)
        CU(cudaMemcpyAsync(carrier_out, d_car, n * sizeof(float), cudaMemcpyDeviceToHost, 0));
    PllArgs a{};
    a.pilot = d_car;
    a.pilot_stride = n;
    a.trig = d_trig;
    a.if_stride = n;
    a.if_off = 0;
    a.n_if = ni;
    a.state = r->d_pll_state.get();
    a.state_stride = 8;
    a.prm = r->prm;
    CU(launch_pll(a, 1, 0));                                                                             // :256
    CU(launch_rds_mix(d_out, d_trig, d_chan, r->d_shift_state.get(), r->delay, n, r->prm.scale, r->prm.adjust, 0));   // :259-263, :269
    if (r->delay)
        CU(cudaMemcpyAsync(r->d_shift_state.get(), d_chan + (n - r->delay), r->delay * sizeof(float), cudaMemcpyDeviceToDevice, 0));   // :265-266
    CU(cudaMemcpy(mixer_out, d_out, n * sizeof(float), cudaMemcpyDeviceToHost));
    if (channel_out)
        CU(cudaMemcpy(channel_out, d_chan, n * sizeof(float), cudaMemcpyDeviceToHost));
    return FMRX_OK;
}

extern "C" int fmrx_rds_pll_state(fmrx_rds *r, float out[6])
{
    if (!r || !out)
        return FMRX_ERR_ARG;
    CU(cudaSetDevice(r->device));
    float st[8];
    CU(cudaMemcpy(st, r->d_pll_state.get(), sizeof(st), cudaMemcpyDeviceToHost));
    std::memcpy(out, st, 6 * sizeof(float));
    return FMRX_OK;
}

// ---------------------------------------------------------------------------
// Spectrum tap: estimatePSD, src/fourier.cpp:35-117
// ---------------------------------------------------------------------------
extern "C" int fmrx_estimate_psd(float *freq, float *psd, const float *samples, size_t n, int freq_bins, float Fs)
{
    // (freq_bins <= 2048: the twiddle table and the window live in the default 48 KB of shared memory)
    if (!freq || !psd || !samples || freq_bins < 2 || freq_bins > 2048 || !(Fs > 0) || n / freq_bins < 1 || n / freq_bins > 0x7fffffffu)
        return FMRX_ERR_ARG;
    const int half = freq_bins / 2;
    const int n_seg = static_cast<int>(n / freq_bins);                   // :63 (samples beyond whole segments are ignored)
    const float df = Fs / freq_bins;                                     // :43
    for (int i = 0; i < half; i++)
        freq[i] = i * df;                                                // :50
    DevBuf d_x, d_p;
    const size_t used = static_cast<size_t>(n_seg) * freq_bins;
    CU(d_x.alloc(used * sizeof(float)));
    CU(d_p.alloc(half * sizeof(float)));
    CU(cudaMemcpy(d_x.p, samples, used * sizeof(float), cudaMemcpyHostToDevice));
    CU(launch_psd(d_p.as<float>(), d_x.as<float>(), n_seg, freq_bins, Fs, 0));
    CU(cudaMemcpy(psd, d_p.p, half * sizeof(float), cudaMemcpyDeviceToHost));
    return FMRX_OK;
}

// ---------------------------------------------------------------------------
// Band scan: Welch's averaged periodogram of the complex u8 IQ stream, and the station finder (include/fmrx.h)
// ---------------------------------------------------------------------------
// The handle keeps the stream's tail (pairs [n_seg*H, pairs), fewer than N) on the device.  A call first runs the at
// most two segments that start in that tail, assembled from the tail and the head of the new input, then the segments
// that lie wholly in the new input, straight from the caller's device buffer (fmrx_scan_process_device) or from
// device staging chunks (fmrx_scan_process).  Launches cover whole runs (scan_run_segments) counted from the call's
// first wholly-new segment, and the staging chunks are whole runs too, so both paths add the same partial sums in the
// same order.
struct fmrx_scan {
    int device = 0, n = 0;
    double fs = 0, win_sq = 0;                 // sum of the double window's squares
    stream_ptr st, cp;                         // compute, staging copies (host path)
    event_ptr ev_in, ev_out, ev_copied[2], ev_used[2];
    dptr<float> d_win;
    dptr<float2> d_tw;
    dptr<double> d_acc, d_partial;
    size_t partial_runs = 0;                   // capacity of d_partial in runs of N doubles
    dptr<uint8_t> d_tail[2], d_asm, d_stage[2];
    size_t stage_cap = 0;                      // bytes of each d_stage
    int cur = 0;                               // d_tail[cur] holds the tail
    uint64_t pairs = 0, n_seg = 0;

    ~fmrx_scan()
    {
        cudaSetDevice(device);
        cudaDeviceSynchronize();
    }
};

namespace {

constexpr size_t kScanPartialDoubles = size_t(1) << 24;   // 128 MB: the largest partial buffer (4096 runs at N = 4096)
constexpr size_t kScanStageBytes = size_t(1) << 26;       // per host-path staging buffer: 512 runs of 2^16 pairs

bool scan_n_ok(int n_fft) { return n_fft >= 256 && n_fft <= 16384 && (n_fft & (n_fft - 1)) == 0; }

// Segments [0, n_seg) of the pairs at iq (device), added to the accumulator on s->st.get() in launches of whole runs.
int scan_segments(fmrx_scan *s, const uint8_t *iq, uint64_t n_seg)
{
    const int N = s->n, H = N / 2, R = scan_run_segments(N);
    const uint64_t runs_total = (n_seg + R - 1) / R;
    const size_t max_runs = kScanPartialDoubles / N;
    const size_t want = static_cast<size_t>(std::min<uint64_t>(runs_total, max_runs));
    if (want > s->partial_runs) {
        s->partial_runs = 0;
        CU(dalloc_async(s->d_partial, want * N, s->st.get()));
        s->partial_runs = want;
    }
    const uint64_t per_launch = static_cast<uint64_t>(max_runs) * R;
    for (uint64_t j = 0; j < n_seg; j += per_launch) {
        const int k = static_cast<int>(std::min<uint64_t>(per_launch, n_seg - j));
        CU(launch_scan(iq + 2 * j * H, k, N, s->d_win.get(), s->d_tw.get(), s->d_partial.get(), s->d_acc.get(), s->st.get()));
    }
    return FMRX_OK;
}

// One call: `src` is a host pointer (host = true) or a device pointer ordered on s->st.
int scan_run(fmrx_scan *s, const uint8_t *src, uint64_t n, bool host)
{
    const uint64_t N = s->n, H = N / 2;
    const cudaMemcpyKind in_kind = host ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice;
    const uint64_t P = s->pairs, start = s->n_seg * H, tl = P - start, end = P + n;
    // 1. segments that start in the tail: at `start` and `start + H`, whole ones only
    uint64_t k_str = 0;
    while (k_str < 2 && start + k_str * H < P && start + k_str * H + N <= end)
        k_str++;
    if (k_str) {
        const uint64_t head = start + (k_str - 1) * H + N - P;
        CU(cudaMemcpyAsync(s->d_asm.get(), s->d_tail[s->cur].get(), 2 * tl, cudaMemcpyDeviceToDevice, s->st.get()));
        CU(cudaMemcpyAsync(s->d_asm.get() + 2 * tl, src, 2 * head, in_kind, s->st.get()));
        const int rc = scan_segments(s, s->d_asm.get(), k_str);
        if (rc != FMRX_OK)
            return rc;
    }
    // 2. segments wholly in the new input (none if a segment starting in the tail is still incomplete)
    const uint64_t next = start + k_str * H;
    uint64_t k_main = 0;
    if (next >= P && end - next >= N)
        k_main = (end - next - N) / H + 1;
    if (k_main) {
        const uint8_t *base = src + 2 * (next - P);
        if (!host) {
            const int rc = scan_segments(s, base, k_main);
            if (rc != FMRX_OK)
                return rc;
        } else {
            // whole runs per staging chunk, double-buffered: copies on s->cp under the kernels on s->st
            const uint64_t R = scan_run_segments(s->n);
            const uint64_t chunk = std::max<uint64_t>(1, kScanStageBytes / (2 * R * H)) * R;   // segments
            const size_t need = static_cast<size_t>(2 * ((std::min(chunk, k_main) - 1) * H + N));
            if (need > s->stage_cap) {
                s->stage_cap = 0;
                for (auto &q : s->d_stage)
                    CU(dalloc_async(q, need, s->st.get()));
                s->stage_cap = need;
            }
            CU(cudaEventRecord(s->ev_used[0].get(), s->st.get()));        // (the allocations above are ordered on s->st)
            CU(cudaEventRecord(s->ev_used[1].get(), s->st.get()));
            int b = 0;
            for (uint64_t j = 0; j < k_main; j += chunk, b ^= 1) {
                const uint64_t k = std::min(chunk, k_main - j);
                CU(cudaStreamWaitEvent(s->cp.get(), s->ev_used[b].get(), 0));
                CU(cudaMemcpyAsync(s->d_stage[b].get(), base + 2 * j * H, 2 * ((k - 1) * H + N), cudaMemcpyHostToDevice, s->cp.get()));
                CU(cudaEventRecord(s->ev_copied[b].get(), s->cp.get()));
                CU(cudaStreamWaitEvent(s->st.get(), s->ev_copied[b].get(), 0));
                const int rc = scan_segments(s, s->d_stage[b].get(), k);
                if (rc != FMRX_OK)
                    return rc;
                CU(cudaEventRecord(s->ev_used[b].get(), s->st.get()));
            }
        }
    }
    // 3. the new tail: pairs [n_seg*H, end), from the old tail and the new input
    s->n_seg += k_str + k_main;
    const uint64_t ns = s->n_seg * H;
    uint8_t *dst = s->d_tail[s->cur ^ 1].get();
    uint64_t a = 0;
    if (ns < P) {
        a = P - ns;
        CU(cudaMemcpyAsync(dst, s->d_tail[s->cur].get() + 2 * (ns - start), 2 * a, cudaMemcpyDeviceToDevice, s->st.get()));
    }
    const uint64_t from = ns > P ? ns - P : 0;
    if (n > from)
        CU(cudaMemcpyAsync(dst + 2 * a, src + 2 * from, 2 * (n - from), in_kind, s->st.get()));
    s->cur ^= 1;
    s->pairs = end;
    return FMRX_OK;
}

}  // namespace

extern "C" int fmrx_scan_create(fmrx_scan **out, int n_fft, double rf_fs, int device)
{
    if (!out || !scan_n_ok(n_fft) || !(rf_fs > 0) || !std::isfinite(rf_fs))
        return FMRX_ERR_ARG;
    *out = nullptr;
    const int rc = open_device(device);
    if (rc != FMRX_OK)
        return rc;
    std::unique_ptr<fmrx_scan> s(new (std::nothrow) fmrx_scan());
    if (!s)
        return FMRX_ERR_ALLOC;
    s->device = device;
    s->n = n_fft;
    s->fs = rf_fs;
    const int N = n_fft;
    CU(make_stream(s->st));
    CU(make_stream(s->cp));
    for (event_ptr *e : { &s->ev_in, &s->ev_out, &s->ev_copied[0], &s->ev_copied[1], &s->ev_used[0], &s->ev_used[1] })
        CU(make_event(*e));
    // the periodic Hann window and the twiddles, in double, rounded to float
    std::vector<float> win(N);
    std::vector<float2> tw(N / 2);
    const double two_pi = 2.0 * 3.14159265358979323846;
    s->win_sq = 0.0;
    for (int k = 0; k < N; k++) {
        const double w = 0.5 - 0.5 * std::cos(two_pi * k / N);
        win[k] = static_cast<float>(w);
        s->win_sq += w * w;
    }
    for (int k = 0; k < N / 2; k++)
        tw[k] = make_float2(static_cast<float>(std::cos(two_pi * k / N)), static_cast<float>(-std::sin(two_pi * k / N)));
    CU(dalloc(s->d_win, N));
    CU(dalloc(s->d_tw, N / 2));
    CU(dalloc(s->d_acc, N));
    CU(dalloc(s->d_tail[0], 2 * N));
    CU(dalloc(s->d_tail[1], 2 * N));
    CU(dalloc(s->d_asm, 3 * N));              // the tail and the head of a call: two segments, 3N/2 pairs
    CU(cudaMemcpy(s->d_win.get(), win.data(), N * sizeof(float), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(s->d_tw.get(), tw.data(), N / 2 * sizeof(float2), cudaMemcpyHostToDevice));
    CU(cudaMemset(s->d_acc.get(), 0, N * sizeof(double)));
    *out = s.release();
    return FMRX_OK;
}

extern "C" int fmrx_scan_destroy(fmrx_scan *s)
{
    delete s;
    return FMRX_OK;
}

extern "C" int fmrx_scan_reset(fmrx_scan *s)
{
    if (!s)
        return FMRX_ERR_ARG;
    CU(cudaSetDevice(s->device));
    CU(cudaStreamSynchronize(s->st.get()));
    CU(cudaMemset(s->d_acc.get(), 0, s->n * sizeof(double)));
    s->pairs = 0;
    s->n_seg = 0;
    return FMRX_OK;
}

extern "C" int fmrx_scan_process(fmrx_scan *s, const uint8_t *iq, size_t n_pairs)
{
    if (!s || (!iq && n_pairs))
        return FMRX_ERR_ARG;
    if (!n_pairs)
        return FMRX_OK;
    CU(cudaSetDevice(s->device));
    const int rc = scan_run(s, iq, n_pairs, true);
    CU(cudaStreamSynchronize(s->st.get()));    // the caller may reuse iq on return
    return rc;
}

extern "C" int fmrx_scan_process_device(fmrx_scan *s, const uint8_t *iq_dev, size_t n_pairs, void *stream)
{
    if (!s || (!iq_dev && n_pairs))
        return FMRX_ERR_ARG;
    if (!n_pairs)
        return FMRX_OK;
    CU(cudaSetDevice(s->device));
    cudaStream_t caller = static_cast<cudaStream_t>(stream);
    CU(cudaEventRecord(s->ev_in.get(), caller));
    CU(cudaStreamWaitEvent(s->st.get(), s->ev_in.get(), 0));
    const int rc = scan_run(s, iq_dev, n_pairs, false);
    CU(cudaEventRecord(s->ev_out.get(), s->st.get()));
    CU(cudaStreamWaitEvent(caller, s->ev_out.get(), 0));
    return rc;
}

extern "C" int fmrx_scan_read(fmrx_scan *s, double *psd, size_t n, uint64_t *n_segments)
{
    if (!s || !psd || n < static_cast<size_t>(s->n))
        return FMRX_ERR_ARG;
    CU(cudaSetDevice(s->device));
    CU(cudaStreamSynchronize(s->st.get()));
    CU(cudaMemcpy(psd, s->d_acc.get(), s->n * sizeof(double), cudaMemcpyDeviceToHost));
    const double norm = s->n_seg ? 1.0 / (static_cast<double>(s->n_seg) * s->fs * s->win_sq) : 0.0;
    for (int m = 0; m < s->n; m++)
        psd[m] = s->n_seg ? psd[m] * norm : 0.0;
    if (n_segments)
        *n_segments = s->n_seg;
    return FMRX_OK;
}

extern "C" int fmrx_find_stations(const double *psd, int n_fft, double rf_fs, double threshold_db, double channel_hz,
                                  fmrx_station *out, int max_out, int *n_found)
{
    if (!psd || !n_found || max_out < 0 || (!out && max_out) || !scan_n_ok(n_fft) || !(rf_fs > 0) ||
        !std::isfinite(rf_fs) || !std::isfinite(threshold_db) || !std::isfinite(channel_hz))
        return FMRX_ERR_ARG;
    if (threshold_db <= 0)
        threshold_db = 10.0;
    if (channel_hz <= 0)
        channel_hz = 200e3;
    const int N = n_fft;
    const double df = rf_fs / N;
    const double hh = std::floor(channel_hz / (2.0 * df) + 0.5);
    if (!(hh >= 1) || 2 * hh + 1 > N)
        return FMRX_ERR_ARG;
    const int h = static_cast<int>(hh);
    std::vector<double> sorted(psd, psd + N);
    std::sort(sorted.begin(), sorted.end());
    const double floor_ = sorted[static_cast<size_t>(std::floor(0.1 * (N - 1)))];
    const double thr = floor_ * std::pow(10.0, threshold_db / 10.0);
    struct Cand { int m; double mean; };
    std::vector<Cand> cand;
    for (int m = h; m <= N - 1 - h; m++) {
        double sum = 0.0;
        for (int k = m - h; k <= m + h; k++)
            sum += psd[k];
        const double mean = sum / (2 * h + 1);
        if (mean >= thr && mean > 0)
            cand.push_back({ m, mean });
    }
    std::sort(cand.begin(), cand.end(), [](const Cand &a, const Cand &b) {
        return a.mean != b.mean ? a.mean > b.mean : a.m < b.m;
    });
    std::vector<Cand> acc;
    for (const Cand &c : cand) {
        bool ok = true;
        for (const Cand &a : acc)
            if (std::abs(c.m - a.m) * df < channel_hz) {
                ok = false;
                break;
            }
        if (ok)
            acc.push_back(c);
    }
    std::vector<fmrx_station> st;
    for (const Cand &c : acc) {
        double sq = 0.0, sfq = 0.0, sp = 0.0;
        for (int k = c.m - h; k <= c.m + h; k++) {
            const double q = std::max(psd[k] - floor_, 0.0);
            sq += q;
            sfq += (k - N / 2) * df * q;
            sp += psd[k];
        }
        st.push_back({ sfq / sq, 10.0 * std::log10(sp * df), 10.0 * std::log10(c.mean / floor_) });
    }
    std::sort(st.begin(), st.end(), [](const fmrx_station &a, const fmrx_station &b) { return a.offset_hz < b.offset_hz; });
    *n_found = static_cast<int>(st.size());
    for (int i = 0; i < max_out && i < static_cast<int>(st.size()); i++)
        out[i] = st[i];
    return FMRX_OK;
}

// ---------------------------------------------------------------------------
// RDS decoder: constants and tables (include/fmrx.h, fmrx_set_rds), and the group summary
// ---------------------------------------------------------------------------

namespace fmrx {

RdsParams rds_params(int fs)
{
    RdsParams P{};
    P.fs = fs;
    P.D = fs == 288000 ? 12 : 10;
    P.fs2 = fs / P.D;
    P.L = static_cast<int>(P.fs2 / 2375.0 + 0.5);
    P.M = P.fs2 / 10;
    P.taps = 2 * static_cast<int>(63.0 * fs / 240000.0 + 0.5) + 1;
    const int g = std::gcd(57000, fs);
    P.P = fs / g;
    P.q = 57000 / g;
    const int g2 = std::gcd(2375, 2 * P.fs2);      // 1187.5 / fs2 = 2375 / (2 fs2)
    P.Q = 2 * P.fs2 / g2;
    P.q2 = 2375 / g2;
    return P;
}

void rds_tables(const RdsParams &P, float *taps, float2 *mix, double2 *bitphase)
{
    const double pi = 3.14159265358979323846;
    const int N = P.taps;
    const double fc = 2.0 * 4000.0 / P.fs;
    std::vector<double> h(N);
    double sum = 0.0;
    for (int n = 0; n < N; n++) {
        const double x = n - (N - 1) / 2.0;
        const double sinc = x == 0.0 ? 1.0 : std::sin(pi * fc * x) / (pi * fc * x);
        const double w = 0.42 - 0.5 * std::cos(2 * pi * n / (N - 1)) + 0.08 * std::cos(4 * pi * n / (N - 1));
        h[n] = fc * sinc * w;
        sum += h[n];
    }
    for (int n = 0; n < N; n++)
        taps[n] = static_cast<float>(h[n] / sum);
    for (int k = 0; k < P.P; k++) {
        const double a = 2 * pi * k / P.P;
        mix[k] = make_float2(static_cast<float>(std::cos(a)), -static_cast<float>(std::sin(a)));
    }
    for (int k = 0; k < P.Q; k++) {
        const double a = 2 * pi * k / P.Q;
        bitphase[k] = make_double2(std::cos(a), -std::sin(a));
    }
}

}  // namespace fmrx

extern "C" int fmrx_rds_summarise(const fmrx_rds_group *g, size_t n, fmrx_rds_info *out)
{
    if (!out || (n && !g))
        return FMRX_ERR_ARG;
    std::memset(out, 0, sizeof(*out));
    out->pty = out->tp = -1;
    std::memset(out->ps, ' ', 8);
    std::memset(out->rt, ' ', 64);
    std::vector<uint16_t> pi_seen;
    int ab = -1;
    for (size_t i = 0; i < n; i++) {
        const fmrx_rds_group &x = g[i];
        out->groups++;
        out->blocks_total += 4;
        for (int b = 0; b < 4; b++)
            out->blocks_valid += (x.valid >> b) & 1u;
        if ((x.valid & 1u) && !out->pi_valid) {
            if (std::find(pi_seen.begin(), pi_seen.end(), x.block[0]) != pi_seen.end()) {
                out->pi_valid = 1;
                out->pi = x.block[0];
            } else {
                pi_seen.push_back(x.block[0]);
            }
        }
        if (!(x.valid & 2u))
            continue;
        const uint16_t B = x.block[1];
        out->pty = (B >> 5) & 31;
        out->tp = (B >> 10) & 1;
        const int type = B >> 12, version_b = (B >> 11) & 1;
        if (type == 0 && (x.valid & 8u)) {
            const int seg = B & 3;
            out->ps[2 * seg] = static_cast<char>(x.block[3] >> 8);
            out->ps[2 * seg + 1] = static_cast<char>(x.block[3] & 0xFF);
            out->ps_seen |= static_cast<uint8_t>(1u << seg);
        } else if (type == 2) {
            const int flag = (B >> 4) & 1, seg = B & 15;
            if (version_b ? !(x.valid & 8u) : (x.valid & 12u) != 12u)
                continue;
            if (flag != ab) {
                if (ab >= 0) {
                    std::memset(out->rt, ' ', 64);
                    out->rt_seen = 0;
                }
                ab = flag;
            }
            if (version_b) {
                out->rt[2 * seg] = static_cast<char>(x.block[3] >> 8);
                out->rt[2 * seg + 1] = static_cast<char>(x.block[3] & 0xFF);
            } else {
                out->rt[4 * seg] = static_cast<char>(x.block[2] >> 8);
                out->rt[4 * seg + 1] = static_cast<char>(x.block[2] & 0xFF);
                out->rt[4 * seg + 2] = static_cast<char>(x.block[3] >> 8);
                out->rt[4 * seg + 3] = static_cast<char>(x.block[3] & 0xFF);
            }
            out->rt_seen |= static_cast<uint16_t>(1u << seg);
        }
    }
    out->ps[8] = 0;
    out->rt[64] = 0;
    for (int k = 0; k < 64; k++)
        if (out->rt[k] == 0x0D) {
            out->rt[k] = 0;
            break;
        }
    return FMRX_OK;
}
