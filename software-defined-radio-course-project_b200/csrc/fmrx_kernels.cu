// fmrx_kernels.cu -- hand-written sm_100a kernels of the FM receive chain.
//
//   K1 k_rf_demod      u8 IQ unpack + RF low-pass/decimate (I,Q) + FM discriminator
//                      (reference: src/iofunc.cpp:62-69, src/project.cpp:57-69,
//                       src/filter.cpp:84-92 with up=1, src/filter.cpp:110-132)
//   K2 k_bandpass_pair pilot and stereo-band band-pass FIRs (src/project.cpp:162,165)
//   K3 k_pll           PLL recurrence, one warp per capture (src/filter.cpp:157-171)
//   K4 k_audio         NCO cosine, mixer, mono+stereo polyphase low-pass with the
//                      shared-state block quirk, mono delay, L/R combine, s16 pack
//                      (src/filter.cpp:170,176-199, src/project.cpp:146-193)
//
// Data layout: every per-capture stream is contiguous ([capture][sample]); IF-rate
// arrays carry `if_off` samples of history in front of the chunk so that FIR taps
// that reach before the chunk start are plain negative indices.
//
// FIR arithmetic is acc = fadd(acc, fmul(c[k], x)) from +0 with k ascending --
// the reference's exact sequence -- so one MAC costs an FMUL and an FADD: the
// attainable ceiling of these kernels is half the FFMA peak by construction.
#include <cstddef>
#include <mutex>
#include <type_traits>

#include "fmrx_internal.h"
#ifdef FMRX_PLL_PROFILE   // development build: k_pll prints its cycle accounting for capture 0 of every launch
#include <cstdio>
#endif

namespace fmrx {

// Per-device launch configuration.  cudaFuncSetAttribute(MaxDynamicSharedMemorySize) applies to
// the CURRENT device only, and one process may hold pipelines on several devices
// (fmrx_config.device), created from several host threads: everything cached about a kernel's
// opt-in shared memory is keyed by the device ordinal and guarded by a mutex.
constexpr int kMaxDevices = 64;
struct DeviceCfg {
    size_t rf_smem[2][3] = {};             // k_rf_demod_win<10|4|9, untuned|tuned>: configured dynamic shared memory
    size_t audio_smem = 0;                 // k_audio
    size_t bp_smem = 0;                    // k_bandpass_pair
    size_t pll_ring_only = 0, pll_whole_sm = 0;
    int sm_count = 0;
};
static std::mutex g_cfg_mutex;
static DeviceCfg g_cfg[kMaxDevices];
static DeviceCfg *device_cfg()
{
    int dev = -1;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices)
        return nullptr;
    return &g_cfg[dev];
}

// ============================================================================
// K1: u8 unpack + RF FIR (decimating) + FM discriminator
// ============================================================================
//
// A tile computes RF_COMPUTED consecutive IF outputs; the first one is the
// discriminator's "previous sample" halo, so RF_COMPUTED-1 demod samples are
// produced.  The u8 IQ window of the tile is converted to float ONCE while it
// is staged into shared memory, de-interleaved into an I plane and a Q plane.

constexpr int RF_COMPUTED = 512;                        // IF outputs computed per tile
constexpr int RF_REAL = RF_COMPUTED - 1;                // 511 demod samples per tile

// ---- K1: register delay line over the RAW u8 tile (decimation known at compile time) ----------------
//
// Output n, tap k reads x[n*D - k].  A thread owns R = 4 consecutive outputs n..n+3, and output n+i at tap k reads
// exactly the sample output n read at tap k - i*D.  So only output n ("i = 0") loads from shared memory, one IQ
// pair per tap, into a circular register delay line of L = 3*D entries per plane; outputs n+1..n+3 take theirs from
// the line, D, 2D and 3D taps back.  The tap loop is unrolled over one trip round the line so that every line index
// is static.  Each accumulator still sees its products in ascending tap order.  T is padded to a multiple of L with
// zero taps: acc + 0*x is a bit-exact no-op for finite x.
//
// Round 2: the tile is staged as the RAW bytes it is (one aligned 32-bit global load and one 32-bit shared store per
// two IQ pairs; round 1 converted to two float planes while staging, which took 31 % of the kernel's instructions at
// 51 taps and four times the shared memory) and a pair is converted when the thread that owns it loads it: one
// 16-bit LDS, then per byte a byte-permute into the float 65536 + b/128 and one subtraction (bit-identical to
// (b - 128)/128, fmrx_device.cuh).  Per tap: 1 pair LDS + 4 conversion instructions + 1 broadcast tap LDS against
// 8 FMUL + 8 FADD.  The tile is padded by one 32-bit word per 4*D pairs so that the lane stride (4*D pairs + 1 word)
// is an odd number of words: conflict-free.

constexpr int RFW_THREADS = 128;
constexpr int RFW_R = 4;

template <int D> struct RfWin {
    static constexpr int L = (RFW_R - 1) * D;       // delay-line length
    static constexpr int SEG = RFW_R * D;           // pairs per thread = padding period (even for every D in use)
    static_assert(SEG % 2 == 0, "two pairs per staged word");
    static __host__ __device__ int tpad(int T) { return (T + L - 1) / L * L; }
    static __host__ __device__ int wp_max(int T) { return (RF_COMPUTED - 1) * D + T + (tpad(T) - T) + 1; }   // staged pairs (one more if the window starts on an odd pair)
    static __host__ __device__ int words(int T) { return (wp_max(T) + 1) / 2 + (wp_max(T) + 1) / SEG + 2; }  // 32-bit words of the padded tile
    static size_t smem_bytes(int T) { return sizeof(uint32_t) * (size_t)2 * words(T) + sizeof(float) * ((size_t)2 * RF_COMPUTED + tpad(T)); }   // two tiles
    // tuned: one float2 per staged pair, one float2 of padding per SEG pairs (lane stride SEG + 1 float2: conflict-free)
    static __host__ __device__ int words_tuned(int T) { return 2 * (wp_max(T) + wp_max(T) / SEG + 1); }
    static size_t smem_bytes_tuned(int T) { return sizeof(uint32_t) * (size_t)2 * words_tuned(T) + sizeof(float) * ((size_t)2 * RF_COMPUTED + tpad(T)); }
};

// Tuned K1 (fmrx_set_tuning): the tile is staged already mixed to the station, I' = i cos + q sin, Q' = q cos - i sin
// with (cos, sin) = cs[ph >> 16], ph = (uint32)(n * inc) at absolute pair n, as two floats per pair -- round 1's float
// staging -- and the delay line loads those floats instead of converting bytes.  Rotating at use instead would cost a
// table lookup per tap and thread.  The staging is plain loads (it computes), so there is no cp.async on this path.
__device__ __forceinline__ void rf_pair(uint32_t v, float &i, float &q)
{
    i = unpack_u8_byte<0>(v);
    q = unpack_u8_byte<1>(v);
}
__device__ __forceinline__ void rf_pair(float2 v, float &i, float &q)
{
    i = v.x;
    q = v.y;
}

// A CTA takes RFW_TILES_MAX (fewer on short chunks) consecutive tiles of one capture and keeps two raw tiles in shared
// memory: the bytes of tile i+1 arrive by cp.async (4 bytes per request: the tile starts on an arbitrary IQ pair, and
// the padded layout breaks 16-byte runs anyway) while tile i is computed.  Before this the kernel spent two thirds of
// its time at 51 taps waiting for the tile it was about to compute (ncu source view, profiles/r02_ncu_summary.md).
constexpr int RFW_TILES_MAX = 8;

template <int D, bool Tuned>
__global__ void __launch_bounds__(RFW_THREADS) k_rf_demod_win(const RfDemodArgs a, const int tiles_per_cta, const RfTuneArgs tu)
{
    using W = RfWin<D>;
    constexpr int L = W::L, SEG = W::SEG, R = RFW_R;
    using Elem = typename std::conditional<Tuned, float2, unsigned short>::type;   // one staged pair
    using Val = typename std::conditional<Tuned, float2, uint32_t>::type;
    constexpr int PADE = Tuned ? 1 : 2;     // padding elements per SEG staged pairs
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int T = a.T;
    const int Tpad = (T + L - 1) / L * L;
    const int words = Tuned ? W::words_tuned(T) : W::words(T);
    uint32_t *s_buf = reinterpret_cast<uint32_t *>(smem_raw);               // two tiles (raw: two pairs per word), padded
    float *o_i = reinterpret_cast<float *>(s_buf + 2 * words);              // [RF_COMPUTED]
    float *o_q = o_i + RF_COMPUTED;
    float *s_c = o_q + RF_COMPUTED;                                         // [Tpad]

    const int c = blockIdx.y;
    const int tid = threadIdx.x;
    const long long n_pairs = (long long)a.n_if * D;
    const uint8_t *iq = a.iq + (size_t)c * a.iq_stride;
    const uint8_t *hist = a.hist + (size_t)c * 2 * a.hist_pairs;
    const uint16_t *iq16 = reinterpret_cast<const uint16_t *>(iq);
    const uint16_t *hist16 = reinterpret_cast<const uint16_t *>(hist);
    const int padl0 = Tpad - T;
    const int n_tiles = (a.n_if + RF_REAL - 1) / RF_REAL;
    const int tile_lo = blockIdx.x * tiles_per_cta, tile_hi = min(n_tiles, tile_lo + tiles_per_cta);

    for (int k = tid; k < Tpad; k += RFW_THREADS)
        s_c[k] = (k < T) ? a.taps[k] : 0.0f;
    auto pair_at = [&](long long m) -> uint32_t {
        if (m >= 0)
            return m < n_pairs ? (uint32_t)iq16[m] : 0x8080u;      // (128,128) -> 0.0f, 0.0f
        const long long h = a.hist_pairs + m;
        return h >= 0 ? (uint32_t)hist16[h] : 0x8080u;
    };
    // Staged pair l' (0..Wp) of a tile is chunk-local pair m_first + l'; the window starts `padl` pairs in front of the
    // first sample a real tap reads (the padded taps read those; they only ever meet zero taps), one more if that makes
    // its first pair 4-byte aligned in global memory.  Word j holds pairs l' = 2j, 2j+1 and sits at j + j / (SEG/2).
    auto tile_padl = [&](int tile) {
        const long long m_base = (long long)(tile * RF_REAL - 1) * D - (T - 1);
        return padl0 + (int)((reinterpret_cast<uintptr_t>(iq16 + (m_base - padl0)) >> 1) & 1);
    };
    auto stage = [&](int tile, uint32_t *s_w) {
        const int padl = tile_padl(tile);
        const long long m_first = (long long)(tile * RF_REAL - 1) * D - (T - 1) - padl;
        const int Wp = (RF_COMPUTED - 1) * D + T + padl;
        if constexpr (Tuned) {
            float2 *s_f = reinterpret_cast<float2 *>(s_w);
            const RfTune cap = tu.cap[c];
            const long long n_first = cap.pair_offset + tu.pairs_run + m_first;    // absolute index of staged pair 0
            const uint32_t ph_first = (uint32_t)((unsigned long long)n_first * cap.inc);
            for (int l = tid; l < Wp; l += RFW_THREADS) {
                float xi, xq;
                rf_pair(pair_at(m_first + l), xi, xq);
                if (n_first + l >= 0) {      // the zero history in front of the stream's first pair is not rotated
                    const float2 cs = tu.cs[(ph_first + (uint32_t)l * cap.inc) >> 16];
                    const float ri = fadd(fmul(xi, cs.x), fmul(xq, cs.y));
                    xq = fsub(fmul(xq, cs.x), fmul(xi, cs.y));
                    xi = ri;
                }
                s_f[l + l / SEG] = make_float2(xi, xq);
            }
        } else {
            const int n_words = (Wp + 1) >> 1;
            for (int j = tid; j < n_words; j += RFW_THREADS) {
                const long long m0 = m_first + 2 * (long long)j;
                uint32_t *dst = s_w + j + j / (SEG / 2);
                if (m0 >= 0 && m0 + 1 < n_pairs) {
                    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((unsigned)__cvta_generic_to_shared(dst)), "l"(iq16 + m0) : "memory");
                } else {             // words that straddle the chunk (history in front, nothing behind): assembled pair by pair
                    *dst = pair_at(m0) | (pair_at(m0 + 1) << 16);
                }
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };

    if (tile_lo < tile_hi)
        stage(tile_lo, s_buf);
    for (int tile = tile_lo; tile < tile_hi; tile++) {
        uint32_t *s_w = s_buf + ((tile - tile_lo) & 1) * words;
        if (tile + 1 < tile_hi) {
            stage(tile + 1, s_buf + ((tile + 1 - tile_lo) & 1) * words);
            asm volatile("cp.async.wait_group 1;" ::: "memory");
        } else {
            asm volatile("cp.async.wait_group 0;" ::: "memory");
        }
        __syncthreads();

        const Elem *s_p = reinterpret_cast<const Elem *>(s_w);
        const int n0 = tile * RF_REAL;              // first demod sample of the tile
        const int padl = tile_padl(tile);
        // this thread: computed outputs o0..o0+3, o0 = 4 tid.  Output o0 at tap k reads staged pair tid*SEG + r0 - k,
        // r0 = T - 1 + padl (the same for every thread); pair l' sits at element l' + PADE (l' / SEG), i.e. for
        // l' = tid*SEG + e at tid*(SEG + PADE) + e + PADE (e / SEG)
        const int o0 = tid * R;
        const int r0 = T - 1 + padl;
        const Elem *tp = s_p + tid * (SEG + PADE);

        float di[L], dq[L];                         // delay lines: slot (k mod L) holds the sample of tap k
#pragma unroll
        for (int m = 1; m <= L; m++) {              // "taps" -m: the samples above tap 0's, for outputs o0+1..o0+3
            const int e = r0 + m;
            const Val v = tp[e + PADE * (e / SEG)];
            rf_pair(v, di[L - m], dq[L - m]);
        }
        float ai[R], aq[R];
#pragma unroll
        for (int i = 0; i < R; i++) {
            ai[i] = 0.0f;
            aq[i] = 0.0f;
        }
        for (int k0 = 0; k0 < Tpad; k0 += L) {
            // within a trip e = e_trip - j crosses at most one padding boundary: e / SEG = q - (j > rem)
            const int e_trip = r0 - k0;             // >= 0 by construction of padl
            const int q = e_trip / SEG, rem = e_trip - q * SEG;
            const Elem *tq = tp + e_trip + PADE * q;
#pragma unroll
            for (int j = 0; j < L; j++) {
                const Val v = tq[-j - (j > rem ? PADE : 0)];
                const float ck = s_c[k0 + j];
                const float old_i = di[j], old_q = dq[j];          // tap k - L: output 3's sample
                float xi, xq;
                rf_pair(v, xi, xq);
                di[j] = xi;
                dq[j] = xq;
                ai[0] = fadd(ai[0], fmul(ck, xi));
                aq[0] = fadd(aq[0], fmul(ck, xq));
                ai[1] = fadd(ai[1], fmul(ck, di[(j + L - D) % L]));
                aq[1] = fadd(aq[1], fmul(ck, dq[(j + L - D) % L]));
                ai[2] = fadd(ai[2], fmul(ck, di[(j + L - 2 * D) % L]));
                aq[2] = fadd(aq[2], fmul(ck, dq[(j + L - 2 * D) % L]));
                ai[3] = fadd(ai[3], fmul(ck, old_i));
                aq[3] = fadd(aq[3], fmul(ck, old_q));
            }
        }
#pragma unroll
        for (int i = 0; i < R; i++) {
            o_i[o0 + i] = ai[i];
            o_q[o0 + i] = aq[i];
        }
        __syncthreads();         // (also: every thread is done with this tile's bytes -- the next iteration stages over them)

        float *demod = a.demod + (size_t)c * a.if_stride + a.if_off;
#pragma unroll
        for (int r = 0; r < R; r++) {
            const int o = tid + r * RFW_THREADS;    // coalesced
            const int n = n0 - 1 + o;
            if (o >= 1 && n < a.n_if) {
                demod[n] = fm_discriminate(o_i[o], o_q[o], o_i[o - 1], o_q[o - 1]);
                if (a.i_ds) {
                    const size_t g = (size_t)c * a.stage_stride + a.stage_off + n;
                    a.i_ds[g] = o_i[o];
                    a.q_ds[g] = o_q[o];
                }
            }
        }
        __syncthreads();         // o_i / o_q are free again
    }
}

template <int D, bool Tuned> static cudaError_t launch_rf_demod_win(const RfDemodArgs &a, int n_captures, cudaStream_t s,
                                                                   const RfTuneArgs &tu)
{
    const size_t smem = Tuned ? RfWin<D>::smem_bytes_tuned(a.T) : RfWin<D>::smem_bytes(a.T);
    DeviceCfg *cfg = device_cfg();
    if (!cfg)
        return cudaErrorInvalidDevice;
    {
        std::lock_guard<std::mutex> lock(g_cfg_mutex);
        size_t &configured = cfg->rf_smem[Tuned][D == 10 ? 0 : D == 4 ? 1 : 2];
        if (smem > configured) {
            cudaError_t e = cudaFuncSetAttribute(k_rf_demod_win<D, Tuned>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess)
                return e;
            configured = smem;
        }
    }
    const int tiles = (a.n_if + RF_REAL - 1) / RF_REAL;
    // consecutive tiles per CTA (the next tile's bytes arrive while one is computed), fewer on short chunks so that
    // the grid still fills the machine
    int per = RFW_TILES_MAX;
    while (per > 1 && (long long)((tiles + per - 1) / per) * n_captures < 4 * 148)
        per >>= 1;
    dim3 grid((tiles + per - 1) / per, n_captures);
    k_rf_demod_win<D, Tuned><<<grid, RFW_THREADS, smem, s>>>(a, per, tu);
    return cudaGetLastError();
}

template <bool Tuned> static cudaError_t launch_rf_demod_d(const RfDemodArgs &a, int n_captures, cudaStream_t s, const RfTuneArgs &tu)
{
    // the reference's modes decimate by 10, 4 and 9 (src/project.cpp:327-362); fmrx_mode_table yields nothing else
    if (a.decim == 10)
        return launch_rf_demod_win<10, Tuned>(a, n_captures, s, tu);
    if (a.decim == 4)
        return launch_rf_demod_win<4, Tuned>(a, n_captures, s, tu);
    if (a.decim == 9)
        return launch_rf_demod_win<9, Tuned>(a, n_captures, s, tu);
    return cudaErrorInvalidValue;
}

cudaError_t launch_rf_demod(const RfDemodArgs &a, int n_captures, cudaStream_t s, const RfTuneArgs *tune)
{
    return tune ? launch_rf_demod_d<true>(a, n_captures, s, *tune) : launch_rf_demod_d<false>(a, n_captures, s, RfTuneArgs{});
}

// ============================================================================
// K2: pilot + stereo-band band-pass pair (no decimation)
// ============================================================================
// One staged demod tile feeds both filters.  A thread owns R = 8 consecutive outputs n..n+7; tap k of output
// n+i reads x[n + i - k], so over a group of four taps the eight outputs touch an 11-sample window that moves
// down by four samples per group: the window lives in a circular buffer of three register quads and every
// group brings in ONE new quad (an aligned LDS.128) plus the two filters' four taps (two broadcast LDS.128)
// for 64 FMUL + 64 FADD.  The tap loop is unrolled over one trip round the buffer (12 taps) so that every
// register index is static; T is padded to a multiple of 12 with zero taps (acc + 0*x is a bit-exact no-op for
// finite x; the IF arrays carry enough history in front for the extra reads).  Each accumulator still sees its
// products in ascending tap order (src/filter.cpp:84-92).  The tile is stored with one quad of padding after
// every 8 samples, so the lane stride of the quad loads is 48 bytes: conflict-free.

constexpr int BP_THREADS = 128;
constexpr int BP_R = 8;
constexpr int BP_TILE = BP_THREADS * BP_R;              // 1024 outputs per tile
constexpr int BP_UNROLL = 12;                           // taps per trip: three quads

static inline int bp_tpad(int T) { return (T + BP_UNROLL - 1) / BP_UNROLL * BP_UNROLL; }
// staged samples: outputs n0..n0+1023 need x[n0 - (Tpad-1) .. n0 + 1023], plus the front quad alignment
// samples staged in front of n0 (a multiple of 8): the Tpad - 1 the taps reach back, and the quad the loop loads past them
static inline int bp_front(int T) { return (bp_tpad(T) + 4 + 7) / 8 * 8; }
static inline size_t bp_smem_bytes(int T)
{
    const int staged = bp_front(T) + BP_TILE;            // a multiple of 8
    return sizeof(float) * ((size_t)staged / 8 * 12 + 2 * (size_t)bp_tpad(T));
}

__global__ void __launch_bounds__(BP_THREADS) k_bandpass_pair(const BandpassArgs a)
{
    extern __shared__ __align__(16) float smem[];
    const int T = a.T;
    const int Tpad = (T + BP_UNROLL - 1) / BP_UNROLL * BP_UNROLL;
    const int front = (Tpad + 4 + 7) / 8 * 8;
    const int staged = front + BP_TILE;
    float *s_x = smem;                           // [staged/8][12]: 8 samples + one quad of padding
    float *s_p = s_x + staged / 8 * 12;          // [Tpad] pilot taps
    float *s_c = s_p + Tpad;                     // [Tpad] channel taps

    const int c = blockIdx.y, tid = threadIdx.x;
    const int n0 = blockIdx.x * BP_TILE;
    const float *demod = a.demod + (size_t)c * a.if_stride + a.if_off;

    for (int k = tid; k < Tpad; k += BP_THREADS) {
        s_p[k] = k < T ? a.taps_pilot[k] : 0.0f;
        s_c[k] = k < T ? a.taps_chan[k] : 0.0f;
    }
    // staged sample l (0..staged) is x[n0 - front + l]; history in front of if_off is real data (or the zeros of a
    // fresh stream) as far back as the arrays go: -if_off
    for (int l = tid; l < staged; l += BP_THREADS) {
        const int n = n0 - front + l;
        s_x[l + (l >> 3) * 4] = (n < a.n_if && n >= -a.if_off) ? demod[n] : 0.0f;
    }
    __syncthreads();

    // this thread's outputs n0 + 8 tid + i.  Window quad q holds x[base - 4 q .. base - 4 q + 3] with
    // base = n0 + 8 tid + 4 (staged index front + 8 tid + 4): quads 0 and 1 are the thread's own 8 samples.
    const float4 *xq = reinterpret_cast<const float4 *>(s_x);
    // staged index of the first sample of quad q: l = front + 8 tid + 4 - 4 q, a multiple of 4; its float4 slot
    // is (l / 8) * 3 + (l % 8) / 4
    auto quad = [&](int q) -> float4 {
        const int l = front + 8 * tid + 4 - 4 * q;
        return xq[(l >> 3) * 3 + ((l >> 2) & 1)];
    };
    float4 w0 = quad(0), w1 = quad(1), w2 = quad(2);        // w0: x[n+4..n+7], w1: x[n..n+3], w2: x[n-4..n-1]
    float ap[BP_R], ac[BP_R];
#pragma unroll
    for (int i = 0; i < BP_R; i++) {
        ap[i] = 0.0f;
        ac[i] = 0.0f;
    }
    // One group of four taps k..k+3 with the window (hi, mid, lo) = samples x[m+4..m+7], x[m..m+3], x[m-4..m-1],
    // m = n - k: output i = 4 h + j (h = 0, 1) at tap k + t reads x[n + i - k - t] = x[m + i - t].
    auto group4 = [&](const float4 &hi, const float4 &mid, const float4 &lo, const float4 &cp, const float4 &cc) {
        const float xs[12] = { lo.x, lo.y, lo.z, lo.w, mid.x, mid.y, mid.z, mid.w, hi.x, hi.y, hi.z, hi.w };   // x[m-4 .. m+7]
        const float tp[4] = { cp.x, cp.y, cp.z, cp.w }, tc[4] = { cc.x, cc.y, cc.z, cc.w };
#pragma unroll
        for (int t = 0; t < 4; t++)
#pragma unroll
            for (int i = 0; i < BP_R; i++) {
                const float x = xs[4 + i - t];
                ap[i] = fadd(ap[i], fmul(tp[t], x));
                ac[i] = fadd(ac[i], fmul(tc[t], x));
            }
    };
    const float4 *pq = reinterpret_cast<const float4 *>(s_p);
    const float4 *cq = reinterpret_cast<const float4 *>(s_c);
    int q = 3;                                   // next quad to bring in
    for (int k = 0; k < Tpad; k += BP_UNROLL) {
        group4(w0, w1, w2, pq[k >> 2], cq[k >> 2]);
        w0 = quad(q++);                          // x[m-8 .. m-5] of the next group's m: the new "lo"
        group4(w1, w2, w0, pq[(k >> 2) + 1], cq[(k >> 2) + 1]);
        w1 = quad(q++);
        group4(w2, w0, w1, pq[(k >> 2) + 2], cq[(k >> 2) + 2]);
        w2 = quad(q++);
    }
    float *pilot = a.pilot + (size_t)c * a.pilot_stride;
    float *chan = a.chan + (size_t)c * a.if_stride + a.if_off;
    const int n = n0 + BP_R * tid;
    if (n + BP_R <= a.n_if && ((reinterpret_cast<uintptr_t>(pilot + n) | reinterpret_cast<uintptr_t>(chan + n)) & 15u) == 0) {
        reinterpret_cast<float4 *>(pilot + n)[0] = make_float4(ap[0], ap[1], ap[2], ap[3]);
        reinterpret_cast<float4 *>(pilot + n)[1] = make_float4(ap[4], ap[5], ap[6], ap[7]);
        reinterpret_cast<float4 *>(chan + n)[0] = make_float4(ac[0], ac[1], ac[2], ac[3]);
        reinterpret_cast<float4 *>(chan + n)[1] = make_float4(ac[4], ac[5], ac[6], ac[7]);
    } else {
#pragma unroll
        for (int i = 0; i < BP_R; i++)
            if (n + i < a.n_if) {
                pilot[n + i] = ap[i];
                chan[n + i] = ac[i];
            }
    }
}

cudaError_t launch_bandpass_pair(const BandpassArgs &a, int n_captures, cudaStream_t s)
{
    if (a.if_off < bp_front(a.T))                // the padded taps read this far in front of the chunk
        return cudaErrorInvalidValue;
    dim3 grid((a.n_if + BP_TILE - 1) / BP_TILE, n_captures);
    k_bandpass_pair<<<grid, BP_THREADS, bp_smem_bytes(a.T), s>>>(a);
    return cudaGetLastError();
}

// ============================================================================
// K3: PLL recurrence (src/filter.cpp:157-171)
// ============================================================================
// The recurrence is one dependent chain per capture, so its latency bounds the
// throughput of the whole receive chain; fmrx_pll_core.h holds the exact formulation of
// one step and the measurements behind it.  Evaluated as the reference writes it, a step
// is a sincos, two float products, an atan2 and the loop filter in sequence: ~300 cycles
// on this machine however it is arranged.  k_pll takes the sincos and the atan2 OFF the
// chain by speculating on values, with one CTA of twelve warps per capture (every warp
// SIMT-uniform or one-lane-per-item):
//
//   warp 9   the predictor.  The phase detector computes atan2(x*(-sin t), x*cos t), which
//            up to float rounding is wrap(pi*(x < 0) - t): with that, a step of the recurrence
//            is a handful of float operations (predictor_step), about half of what warp 0
//            needs.  The predictor runs ahead of warp 0 (restarted from the exact state
//            whenever a group of PLL_GROUP steps does not simply continue the one before)
//            and publishes its phaseEst of every step.  It is
//            never used for a result -- it says which float trigArg(u) will almost certainly
//            be: on a locked loop the exact trigArg is the predicted float grid point or a
//            neighbour (tests/test_pll_model.py::test_predictor_tracks_the_exact_recurrence).
//   warps 2,3,6,7,10,11   candidate tables.  trigArg(u) = fl32(w*trigOffset + phaseEst) lives
//            on the float grid of its binade.  For the three grid points G_c-1, G_c, G_c+1
//            around the predictor's, a quad of lanes evaluates everything that hangs off
//            trigArg(u): sin/cos (Cody-Waite + two polynomials), their float roundings, the
//            wrapped angle, the float products with pilot sample u+1, the FMA residuals and
//            the atan2 shortcut -- i.e. Kp*errorD, Ki*errorD of the NEXT sample under each
//            hypothesis, bit for bit what the sequential formulation computes.  Eight steps
//            per pass of a warp; one 32-byte table (PllRow) per step.
//   warp 0   the chain.  Per step: the loop filter of the next sample for the three
//            hypotheses (float additions that need the state but not the index), one FFMA
//            t = phaseEst/ulp - pi, two compares of t against the table's thresholds --
//            which of the three grid points trigArg(u) IS -- and two selects.  ~43 cycles,
//            bound by instruction issue, not latency.  Guards only accumulate; a block of 16
//            steps with a failed guard (table late or not this block's, grid point not among
//            the three, a candidate's own guard, sum too close to a rounding tie) is stepped
//            again the exact way (pll_block_exact).  A group that needs too many of those is
//            done again on the one-hypothesis scheme and the tables are retried with back-off;
//            a group whose trigArg leaves the binade of its grid is finished without tables
//            from the block at hand (pll_group_checked), no second pass.
//   warps 1,5   I/O.  One lane per sample: the coalesced pilot load, (double)x, the IEEE
//            reciprocal 1/x, the half-turn flag, w*trigOffset and its split on the float grid,
//            the predictor's constant, for the next group into a 2-group ring in shared
//            memory; and the coalesced store of the previous group's trigArg.
//   (warps 4, 8 share warp 0's scheduler and only take part in the barriers.)
//
// Hand-off is through shared memory rings with sequence stamps and bounded polling: the
// predictor's phaseEst records, the candidate tables, and one progress word warp 0 writes
// per block (flow control for both rings; also how a group is called off).  No barrier
// inside a group.  Only trigArg leaves the chain; the NCO output
// cos(trigArg*scale+adjust) is evaluated in K4.

constexpr int PLL_WARPS = 12;
constexpr int PLL_THREADS = 32 * PLL_WARPS;
constexpr int PLL_CAND_WARPS = 6;        // warps 2,3,6,7,10,11 (schedulers 2 and 3), eight steps each: one per quad of lanes
constexpr int PLL_BATCH = 8;             // steps per pass of a candidate warp
constexpr float PLL_ROW_INVALID = 0x1p100f;   // lq of a table nothing matches
constexpr int PLL_IO_WARPS = 2;          // warps 1, 5 (scheduler 1); warps 4 and 8 (warp 0's scheduler) only take part in the barriers
constexpr int PLL_PRED_WARP = 9;         // the run-ahead predictor (scheduler 1)
constexpr int PLL_GROUP = 2048;          // steps between checkpoints / barriers (a group's header, its two barriers and the hand-over
                                         // are ~3 500 cycles of cold serial code on warp 0: the longer the group the better)
constexpr int PLL_RING = 2 * PLL_GROUP;  // per-sample input ring: the group running and the next one
constexpr int kPllSpareSms = 32;         // SMs that must stay free for the FIR kernels before PLL CTAs claim whole SMs
constexpr int PLL_TABLES = 128;          // candidate tables in flight (a ring over the steps)
constexpr int PLL_PH_RING = 512;         // predicted-phaseEst records in flight
constexpr int PLL_TABLES1 = 256;         // one-hypothesis rows in flight (16 bytes each: the same shared memory as the tables)
constexpr int PLL_BATCH1 = 32;           // ... steps per pass of a candidate warp there: one per lane
constexpr int PLL_LEAD1 = 256;           // ... and how far its predictor may run ahead of warp 0
constexpr int PLL_PBLK = 16;             // ... steps per block of its predictor (one flow-control look, one |angle| test, one publication)
constexpr int PLL_EXACT_MAX1 = 16;       // exact blocks after which a one-hypothesis group is finished without tables
constexpr int PLL_HEAD = 48;             // steps of the NEXT group the predictor and the candidate warps do at the end of a group,
                                         // so that warp 0 finds its first tables waiting (multiple of 16)
constexpr int PLL_PRED_LEAD = 128;       // the predictor stays at most this far ahead of warp 0
constexpr int PLL_SPIN_LIMIT = 1 << 16;  // bounded polling (~1 ms): a bug must not hang the GPU
static_assert(PLL_TABLES % 16 == 0 && PLL_PH_RING % PLL_BATCH == 0, "no ring wraps inside a block of 16 steps or a batch of candidates");
static_assert(PLL_PRED_LEAD + PLL_TABLES <= PLL_PH_RING, "a record outlives every candidate that may still need it");
static_assert(PLL_LEAD1 + PLL_TABLES1 <= PLL_PH_RING && PLL_TABLES1 % PLL_BATCH1 == 0 && PLL_TABLES1 * 16 == PLL_TABLES * 32, "one-hypothesis rings");
constexpr int PLL_ABANDONED = -1;        // progress value: warp 0 gave the group up
constexpr int PLL_EXACT_MAX = PLL_GROUP / 128;  // exact blocks (an eighth of the group) after which a speculated group is given up
constexpr int PLL_BACKOFF_MAX = 64;      // groups between retries of the three-hypothesis tables after repeated failures
                                         // (they run on the one-hypothesis scheme meanwhile)

struct __align__(16) PllIn {             // off-chain inputs of one sample
    float x;
    float c3;                            // three-hypothesis predictor: pi*(x < 0) - (w*trigOffset before this step mod 2 pi); its errorD is wrap(c3 - phaseEst)
    double inv_x;                        // 1/(double)x, IEEE divide
    double v;                            // w * trigOffset after this step (:166-167)
    int vi;                              // rint(v/ulp) for the binade the slot was prepared in ...
    float vr;                            // ... and fl32(v/ulp - vi), |vr| <= 0.5
    pllcore::OneHypIn h1;                // one-hypothesis predictor: P, r, B, c (fmrx_pll_core.h), one LDS.128
};
static_assert(sizeof(PllIn) == 48 && offsetof(PllIn, c3) == 4 && offsetof(PllIn, vi) == 24 && offsetof(PllIn, h1) == 32, "k_pll addresses these fields by offset");
__device__ __forceinline__ double pll_turn(float x) { return x < 0.0f ? 2.0 : 0.0; }   // half a turn, in quadrants (-0.0f: none, as atan2 has it)

__device__ __forceinline__ unsigned smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void st_v4(void *p, int a, int b, int c, int d)
{
    asm volatile("st.volatile.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(smem_u32(p)), "r"(a), "r"(b), "r"(c), "r"(d)
                 : "memory");
}
__device__ __forceinline__ int4 ld_v4(const void *p)
{
    int4 v;
    asm volatile("ld.volatile.shared.v4.b32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
                 : "r"(smem_u32(p))
                 : "memory");
    return v;
}
__device__ __forceinline__ int2 ld_v2(const void *p)
{
    int2 v;
    asm volatile("ld.volatile.shared.v2.b32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(smem_u32(p)) : "memory");
    return v;
}
__device__ __forceinline__ double i2d(int hi, int lo) { return __hiloint2double(hi, lo); }

// ---- the table-speculated steps of one group (warp 0) --------------------------------
//
// One step: the loop filter (:163-164), the grid index of trigArg (:166-167), and the
// lookup of Kp*errorD, Ki*errorD of the next sample in the candidate table of that grid
// point.  No branches, no FP64 on the chain.  The grid index of trigArg(u) =
// fl32(v(u) + phaseEst) is had without leaving the FP32 pipe: with v(u)/ulp = vi + vr
// (integer + remainder, prepared per sample) and phaseEst/ulp = pi + t (pi = rint at the
// group start, so |t| stays small),
//     G = vi + pi + rint(t + vr),   t = fma(phaseEst, 1/ulp, -pi)  (one rounding).
// Error budget, in grid steps: t carries one rounding (<= 2^-24 |t|), vr one (<= 2^-25), their
// sum z one more (<= 2^-24 (|t| + 1/2)), and the reference's own double rounding of
// v + phaseEst moves the exact sum by < 2^-29: together < 2^-23 |t| + 2^-24 + 2^-29.  A z
// farther than 2^-22 * max(|t|, 4) from a tie therefore rounds the way the reference's sum
// does; closer ones (about two per million steps) fail the guard and the group is redone
// the exact way.
// The grid index of a trigArg from what warp 0 parks for it -- the bits of
// t = fma(phaseEst, 1/ulp, -pi): vi + pi + rint(t + vr) (:166-167), kbase = pi - bits(1.5 * 2^23).
__device__ __forceinline__ int parked_index(int t_bits, const PllIn &in, int kbase)
{
    return in.vi + kbase + __float_as_int(__fadd_rn(__fadd_rn(__int_as_float(t_bits), in.vr), 12582912.0f));
}

// pi of a block of 16 steps: rint(phaseEst/ulp) of the phaseEst the block starts from -- the exact one
// at the start of a group, the predictor's thereafter (any integer near phaseEst/ulp will do: it only
// keeps t = phaseEst/ulp - pi small; warp 0 and the candidate warps just have to use the same one).
__device__ __forceinline__ void block_pi(float ph, float inv_ulp_f, float &pi_f, int &kbase)
{
    const float pm = __fadd_rn(__fmul_rn(ph, inv_ulp_f), 12582912.0f);       // rint via 1.5 * 2^23
    pi_f = __fadd_rn(pm, -12582912.0f);
    kbase = __float_as_int(pm) - 0x4B400000 - 0x4B400000;
}

struct TableRun {
    float integ, ph, kpe, kie;       // in/out: loop filter state; Kp*errorD, Ki*errorD of the sample about to run
    float inv_ulp_f, pi_f;           // 1/ulp (a power of two); pi of the group's first block
    int kbase;                       // pi as an integer, less the bit pattern of 1.5 * 2^23 (of the block at hand, for pll_block_exact)
    int base, cnt;                   // first step and number of steps of the group
    unsigned in_base, tab_base, sg_base, prog_addr;   // shared-window addresses: ring {vi, vr}, tables, parked indices, progress word
    unsigned sph_base, kb_base;      // ... the predictor's records, the per-block kbase of the group (for the I/O warp)
    unsigned head_addr;              // ... the I/O warps' words about the head of the next group (pll_block_exact)
    int cont;                        // the group continues the one before: pi of its first block comes from the predictor too
#ifdef FMRX_PLL_PROFILE
    int prof_stamp, prof_c, prof_fatal_exact;
    int prof_tie, prof_range, prof_inv;      // why a block's guard failed: near a rounding tie, grid point not one of the three, no valid table
#endif
    int gi;                          // in: grid index of the trigArg before the group; out: of the last one
    int n_exact;                     // out: blocks of 16 that had to be stepped the exact way
    int fatal;                       // out: the group was not completed here: 1 too many exact blocks (the caller redoes the group),
                                     // 2 an exact block left the group's grid (the caller finishes it without tables, from t_stop)
    int t_stop;                      // out: steps of the group completed when it stopped
    // for the exact steps
    const PllIn *ring;               // the per-sample input ring
    pllcore::Consts k;
    double ulp;
    float toff_base;                 // trigOffset before the group
};

// A block of up to 16 steps the exact way (the checked single-warp step: sincos of the
// known trigArg on the chain, ~300 cycles per step; the reference's statements one by one
// where a guard of that fails), from the state before the block: the fall-back for a
// block in which a table was late, the grid point lay outside its table, a candidate's
// guard failed or the grid index was too close to a tie.  Parks the grid indices exactly
// as the table steps do, and hands back Kp*errorD, Ki*errorD of the sample after the
// block so that the table steps resume.  Returns false if trigArg left the binade the
// group's grid belongs to (the caller then redoes the whole group).
__device__ __noinline__ bool pll_block_exact(TableRun &r, int u0, int nsteps, const int lane)
{
    using namespace pllcore;
    const TrigK K = trig_constants();
    int gi = r.gi;
    Chain c;
    c.integ = r.integ;
    c.ph = r.ph;
    c.toff = fminf(r.toff_base + (float)(u0 - r.base), 16777216.0f);   // the counter saturates (:166)
    c.tad = p_mul((double)gi, r.ulp);
    c.fi = c.fq = 0.0f;
    chain_refresh(c);
    for (int j = 0; j < nsteps; j++) {
        if (c.binade == FMRX_DISARMED || c.ulp != r.ulp)
            return false;
        const int u = u0 + j;
        const PllIn i = r.ring[u & (PLL_RING - 1)];
        StepIn in;
        in.x = i.x;
        in.xd = (double)i.x;
        in.inv_x = i.inv_x;
        in.turn = pll_turn(i.x);
        in.v = i.v;
        if (!chain_step_fast(c, r.k, K, in))
            chain_step_generic(c, r.k, i.x);
        const int g = grid_index(grid_round(c.tad, c.inv_ulp));
        // parked like the table steps do: a float t with vi + pi + rint(t + vr) = the grid index
        asm volatile("st.shared.b32 [%0], %1;" ::"r"(r.sg_base + 4u * (unsigned)(u - r.base)),
                     "r"(__float_as_int(p_faddf((float)(g - i.vi - r.kbase - 0x4B400000), -i.vr))));
        gi = g;
    }
    if (c.binade == FMRX_DISARMED || c.ulp != r.ulp)
        return false;
    // Kp*errorD, Ki*errorD of the sample after the block, from the now known trigArg (the first sample of the next
    // group, at the very end of this one: the I/O warps say when that one is in the ring)
    if (u0 + nsteps == r.base + PLL_GROUP) {
        int a0 = 0, a1 = 0;
        for (int spin = 0; spin < PLL_SPIN_LIMIT; spin++) {
            asm volatile("ld.volatile.shared.b32 %0, [%1];" : "=r"(a0) : "r"(r.head_addr) : "memory");
            asm volatile("ld.volatile.shared.b32 %0, [%1];" : "=r"(a1) : "r"(r.head_addr + 4u) : "memory");
            if (a0 == u0 + nsteps && a1 == u0 + nsteps)
                break;
        }
        if (a0 != u0 + nsteps || a1 != u0 + nsteps)
            return false;
    }
    const PllIn nx = r.ring[(u0 + nsteps) & (PLL_RING - 1)];
    const Feedback f = make_feedback(K, c.tad, pll_turn(nx.x), nx.inv_x, nullptr, nullptr);
    bool ok = true;
    float ed = error_from_feedback(f, nx.x, (double)nx.x, ok);
    if (!ok) {           // the shortcut's guard: the reference's own atan2 of its own float products
        float fi, fq;
        chain_feedback(c, fi, fq);
        ed = p_d2f(atan2((double)p_fmulf(nx.x, -fq), (double)p_fmulf(nx.x, fi)));
    }
    r.kpe = p_fmulf(r.k.kp, ed);
    r.kie = p_fmulf(r.k.ki, ed);
    r.integ = c.integ;
    r.ph = c.ph;
    r.gi = gi;
    return true;
}

// A group without tables, in blocks of 16 from a checkpoint: the single-warp speculative
// step (sincos of the known trigArg on the chain, ~300 cycles) with the prepared inputs;
// a block in which one of its guards fails -- or during which the fast step is disarmed
// (irregular trigOffset, trigArg beyond the exact-reduction range) -- is stepped again
// with the checked step, which falls back to the reference's statements one by one.
// Parks the float trigArg of every step.
__device__ __noinline__ void pll_group_checked(pllcore::Chain &chain, const pllcore::Consts k, const PllIn *ring, int base, int t_begin, int cnt,
                                               bool regular, unsigned sg_base, bool park_ph)
{
    using namespace pllcore;
    const TrigK K = trig_constants();
    Chain ch = chain;
    for (int tb = t_begin; tb < cnt; tb += 16) {
        const int nb = min(16, cnt - tb);
        const Chain ckb = ch;
        bool okb = regular && ch.binade != FMRX_DISARMED;
        if (okb) {
            for (int t = tb; t < tb + nb; t++) {
                const PllIn i = ring[(base + t) & (PLL_RING - 1)];
                StepIn in;
                in.x = i.x;
                in.xd = (double)i.x;
                in.inv_x = i.inv_x;
                in.turn = pll_turn(i.x);
                in.v = i.v;
                okb &= chain_step_spec(ch, k, K, in);
                // (no "memory" clobber: nothing here reads s_g, and the next sample's inputs may be loaded early)
                asm volatile("st.shared.b32 [%0], %1;" ::"r"(sg_base + 4u * (unsigned)t),
                             "r"(park_ph ? __float_as_int(ch.ph) : __float_as_int(__double2float_rn(ch.tad))));
            }
        }
        if (!okb) {
            ch = ckb;
            for (int t = tb; t < tb + nb; t++) {
                const float ta = chain_step(ch, k, K, ring[(base + t) & (PLL_RING - 1)].x, nullptr);
                asm volatile("st.shared.b32 [%0], %1;" ::"r"(sg_base + 4u * (unsigned)t), "r"(park_ph ? __float_as_int(ch.ph) : __float_as_int(ta)) : "memory");
            }
        }
    }
    chain = ch;
}

// ---- the one-hypothesis steps of one group (warp 0) -----------------------------------
//
// fmrx_pll_core.h ("the one-hypothesis scheme") has the idea; here warp 0's part.  A row of step u holds
// Kp*errorD, Ki*errorD of sample u -- the EXACT phase detector, evaluated by a candidate lane for the trigArg
// the reference forms (:167) from the predictor's phaseEst of step u - 1 -- and the predictor's phaseEst of
// step u.  Warp 0 runs the loop filter (:163-164: three dependent float additions per step) and XORs its
// phaseEst with the predicted one.  Induction over a block of 16: the block starts from a phaseEst equal to
// the prediction (checked), so row u0 was computed for the true trigArg, so phaseEst(u0) is the reference's;
// if that equals the prediction again, row u0 + 1 was computed for the true trigArg, and so on.  A block with
// any mismatch (or a candidate's guard, or a row that is not this step's) is stepped again the exact way from
// its checkpoint, after which the comparison simply goes on: the predictor's trajectory and the exact one
// usually re-merge within a block or two (phaseEst's coarse rounding forgets small differences).
// The chain is three times faster than the predictor that feeds it, so unlike the table steps it WAITS for
// its rows.  Parks the bits of phaseEst per step; the I/O warps turn them into trigArg (:167) in parallel.
struct __align__(16) PllRow1 {
    float kpe, kie;                  // Kp*errorD, Ki*errorD of this step's sample
    int ph_bits;                     // the predictor's phaseEst after this step
    int stamp;                       // step + 1; -(step + 1) if a guard of the candidate failed (present, not usable)
};
static_assert(sizeof(PllRow1) == 16, "one LDS.128 per step");

struct OneRun {
    float integ, ph;                 // in/out: loop filter state
    int base, cnt;
    unsigned tab_base, sg_base, prog_addr;
    const PllIn *ring;
    pllcore::Consts k;
    float toff_base;                 // trigOffset before the group
    double tad0;                     // trigArg before the group (exact)
    int n_exact;                     // out: blocks stepped the exact way
    int done;                        // out: steps completed here (< cnt: the caller finishes the group without tables)
    int timed_out;                   // out: a row never came
};

// the chain state after `steps_done` steps of the group, from the loop filter state and the trigArg it implies
__device__ __forceinline__ void onehyp_chain_at(pllcore::Chain &c, float integ, float ph, float toff, double tad)
{
    using namespace pllcore;
    c.integ = integ;
    c.ph = ph;
    c.toff = toff;
    c.tad = tad;
    c.cr = c.sr = c.r = c.nd = c.ulp = c.inv_ulp = 0.0;
    c.cf = c.sf = 0.0f;
    c.binade = FMRX_DISARMED;
    if (fabs(tad) <= (double)FMRX_FAST_TRIG_MAX) {
        chain_refresh(c);
    } else {                             // beyond the exact-reduction range: the library functions (:168-169)
        c.fi = p_d2f(cos(tad));
        c.fq = p_d2f(sin(tad));
    }
}

__device__ __noinline__ void pll_block_exact1(OneRun &r, int u0, int nsteps, float &integ, float &ph)
{
    using namespace pllcore;
    const TrigK K = trig_constants();
    Chain c;
    const double tad = u0 == r.base ? r.tad0 : onehyp_trigarg(r.ring[(u0 - 1) & (PLL_RING - 1)].v, ph);
    onehyp_chain_at(c, integ, ph, fminf(r.toff_base + (float)(u0 - r.base), 16777216.0f), tad);
    for (int j = 0; j < nsteps; j++) {
        const PllIn i = r.ring[(u0 + j) & (PLL_RING - 1)];
        StepIn in;
        in.x = i.x;
        in.xd = (double)i.x;
        in.inv_x = i.inv_x;
        in.turn = pll_turn(i.x);
        in.v = i.v;
        if (c.binade == FMRX_DISARMED || !chain_step_fast(c, r.k, K, in))
            chain_step_generic(c, r.k, i.x);
        asm volatile("st.shared.b32 [%0], %1;" ::"r"(r.sg_base + 4u * (unsigned)(u0 + j - r.base)), "r"(__float_as_int(c.ph)) : "memory");
    }
    integ = c.integ;
    ph = c.ph;
}

__device__ __noinline__ void pll_onehyp_group(OneRun &r, const int lane)
{
    using namespace pllcore;
    float integ = r.integ, ph = r.ph;
    const int base = r.base, cnt = r.cnt;
    const unsigned tab_base = r.tab_base, sg_base = r.sg_base, prog_addr = r.prog_addr;
    int last_pred = __float_as_int(ph);          // the predictor starts the group from this very phaseEst
    int n_exact = 0, t = 0;
    bool timed_out = false;
    auto load_row = [&](unsigned addr) {
        int4 v;
        asm volatile("ld.volatile.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr) : "memory");
        return v;
    };
    for (; t < cnt; t += 16) {
        const int u0 = base + t, nb = min(16, cnt - t);
        // wait (bounded) for the block's last row: the candidate warps store a batch of 32 rows with one
        // instruction, so the block's other rows are there too (each row's own stamp is checked anyway)
        {
            const unsigned a_last = tab_base + (unsigned)((u0 + nb - 1) & (PLL_TABLES1 - 1)) * 16u + 12u;
            int z, spin = 0;
            do {
                asm volatile("ld.volatile.shared.b32 %0, [%1];" : "=r"(z) : "r"(a_last) : "memory");
            } while (z != u0 + nb && z != -(u0 + nb) && ++spin < PLL_SPIN_LIMIT);
            if (spin >= PLL_SPIN_LIMIT) {
                timed_out = true;
                break;
            }
        }
        const float integ0 = integ, ph0 = ph;
        int bad = __float_as_int(ph) ^ last_pred;
        const unsigned row0 = tab_base + (unsigned)(u0 & (PLL_TABLES1 - 1)) * 16u;     // rows do not wrap inside a block of 16
        if (nb == 16) {
            int park[16];
#pragma unroll
            for (int h = 0; h < 16; h += 8) {
                int4 rw[8];
#pragma unroll
                for (int j = 0; j < 8; j++)
                    rw[j] = load_row(row0 + (unsigned)(h + j) * 16u);
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    integ = p_faddf(integ, __int_as_float(rw[j].y));                               // :163
                    ph = p_faddf(ph, p_faddf(__int_as_float(rw[j].x), integ));                     // :164
                    bad |= (__float_as_int(ph) ^ rw[j].z) | (rw[j].w ^ (u0 + h + j + 1));
                    park[h + j] = __float_as_int(ph);
                }
                last_pred = rw[7].z;
            }
#pragma unroll
            for (int j = 0; j < 16; j += 4)
                asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(sg_base + 4u * (unsigned)(t + j)), "r"(park[j]), "r"(park[j + 1]),
                             "r"(park[j + 2]), "r"(park[j + 3])
                             : "memory");
        } else {
            for (int j = 0; j < nb; j++) {
                const int4 rw = load_row(row0 + (unsigned)j * 16u);
                integ = p_faddf(integ, __int_as_float(rw.y));
                ph = p_faddf(ph, p_faddf(__int_as_float(rw.x), integ));
                bad |= (__float_as_int(ph) ^ rw.z) | (rw.w ^ (u0 + j + 1));
                last_pred = rw.z;
                asm volatile("st.shared.b32 [%0], %1;" ::"r"(sg_base + 4u * (unsigned)(t + j)), "r"(__float_as_int(ph)) : "memory");
            }
        }
        if (bad) {
            integ = integ0;
            ph = ph0;
            pll_block_exact1(r, u0, nb, integ, ph);
            if (++n_exact > PLL_EXACT_MAX1) {        // the predictor has lost the trajectory for good: no more waiting for its rows
                t += nb;
                break;
            }
        }
        asm volatile("st.volatile.shared.b32 [%0], %1;" ::"r"(prog_addr), "r"(u0 + nb) : "memory");
    }
    r.integ = integ;
    r.ph = ph;
    r.n_exact = n_exact;
    r.done = min(t, cnt);
    r.timed_out = timed_out;
    (void)lane;
}

// A candidate table: what the next sample's phase detector gives for the three float-grid
// points around the predictor's trigArg of a step.  32 bytes, written by ONE store
// instruction of a candidate warp (four lanes, 8 bytes each), read by warp 0 as two
// 16-byte halves -- the half with the key and the block stamp FIRST, so that a half
// overwritten in between can only fail the check, never pass it.
// The stamp of a table: which block of 16 steps of the launch it is for (low 26 bits: a launch has
// fewer than 2^26 steps, fmrx_create sees to that) and the low 6 bits of the block pi its threshold
// was formed with -- warp 0 and the candidate warps each from their OWN pi, so a disagreement about
// pi (tests/pll_model.cpp, pll_model_stale_head) fails the stamp check instead of selecting a
// neighbouring hypothesis silently.  Never 0 (the stamp of an invalidated row).
__device__ __forceinline__ int pll_stamp(int u0, int kbase) { return (u0 + 1) ^ (kbase << 26); }

struct __align__(32) PllRow {
    float kpe0, kie0, kpe1, kie1;    // Kp*errorD, Ki*errorD of the next sample if trigArg is grid point G_c - 1, G_c
    float kpe2, kie2;                // ... G_c + 1
    float lp;                        // (n1 - 1/2) - vr, n1 = G_c - (vi + pi): trigArg IS G_c iff lp < t < lp + 1,
                                     // t = fma(phaseEst, 1/ulp, -pi) as warp 0 computes it (PLL_ROW_INVALID if a guard failed)
    int stamp;                       // pll_stamp(step & ~15, kbase of that block)
};

__device__ __noinline__ void pll_table_group(TableRun &r, const int lane)
{
    using namespace pllcore;
    float integ = r.integ, ph = r.ph, kpe = r.kpe, kie = r.kie;
    const float inv_ulp_f = r.inv_ulp_f;
    float pi_f = r.pi_f;
    int kbase = r.kbase;
    const int base = r.base, cnt = r.cnt;
    const unsigned sph_base = r.sph_base, kb_base = r.kb_base;
    const unsigned in_base = r.in_base, tab_base = r.tab_base, sg_base = r.sg_base, prog_addr = r.prog_addr;
    int bad = 0, gi = r.gi, n_exact = 0;
    float cmax = 0.0f;
    // (a, b) = t < lo ? (a0, b0) : t > hi ? (a2, b2) : (a1, b1), as selects on the data path (a predicated
    // instruction waits longer for its predicate than a select does)
    auto pick = [](float t, float lo, float hi, float a0, float a1, float a2, float b0, float b1, float b2, float &a, float &b) {
        asm("{ .reg .pred q0, q2;\n\t"
            "setp.lt.f32 q0, %2, %3;\n\t"
            "setp.gt.f32 q2, %2, %4;\n\t"
            "selp.f32 %0, %5, %6, q0;\n\t"
            "selp.f32 %1, %8, %9, q0;\n\t"
            "selp.f32 %0, %7, %0, q2;\n\t"
            "selp.f32 %1, %10, %1, q2; }"
            : "=&f"(a), "=&f"(b)
            : "f"(t), "f"(lo), "f"(hi), "f"(a0), "f"(a1), "f"(a2), "f"(b0), "f"(b1), "f"(b2));
    };
    // One step: from (integrator, phaseEst) after sample u and the table of step u to the state
    // after sample u+1 -- or, with `last`, to Kp*errorD, Ki*errorD of sample u+1 (what a block hands
    // to the next one and to the exact fall-back).
    //   - three hypotheses: trigArg(u) is grid point G_c-1, G_c, G_c+1; for each the loop filter
    //     (:163-164) of sample u+1 -- float additions that need the state but not the index;
    //   - which one: trigArg(u) is the float nearest w*trigOffset + phaseEst (:166-167), i.e. grid
    //     point vi + pi + rint(z), z = t + vr, t = fma(phaseEst, 1/ulp, -pi).  So G_c - 1 iff
    //     z < n1 - 1/2 iff t < lp, and G_c + 1 iff t > lp + 1: two compares of t against values
    //     ready long before; two selects pick the state.
    // On the dependent chain: one FFMA, a compare, two selects.  Returns the bits of t (parked:
    // the grid index is vi + pi + rint(t + vr)).
    // Guards (they only accumulate; the block is stepped again the exact way if one fails), on
    // q = t - (lp + 1/2) = z - n1 up to rounding:
    //   - the table is this block's (stamp);
    //   - |q| < 3/2: the grid point is one of the three;
    //   - q is clear of +-1/2 (a tie of the float rounding) by 2^-15.  The candidate warps only
    //     emit tables with |n1| <= 60, so |t| < 62, and the error budget in grid steps is: t
    //     <= 2^-24 |t|, vr 2^-25, the thresholds lp, lp + 1, lp + 1/2 <= 2^-24 (|n1| + 2) each, the
    //     reference's own double rounding of the sum < 2^-29 -- below 2^-24 * 320 < 2^-15.
    // All three are one test: | | |q| - 1/2 | - 1/2 | < 1/2 - 2^-15.
    auto step = [&](int4 ra, int4 rb, int stamp, bool last) -> int {
        const float kpe0 = __int_as_float(ra.x), kie0 = __int_as_float(ra.y), kpe1 = __int_as_float(ra.z), kie1 = __int_as_float(ra.w);
        const float kpe2 = __int_as_float(rb.x), kie2 = __int_as_float(rb.y);
        const float lp = __int_as_float(rb.z);
        const float hp = p_faddf(lp, 1.0f), lc = p_faddf(lp, 0.5f);
        const float tt = __fmaf_rn(ph, inv_ulp_f, -pi_f);
        if (!last) {
            const float i0 = p_faddf(integ, kie0), i1 = p_faddf(integ, kie1), i2 = p_faddf(integ, kie2);     // :163
            const float p0 = p_faddf(ph, p_faddf(kpe0, i0)), p1 = p_faddf(ph, p_faddf(kpe1, i1)), p2 = p_faddf(ph, p_faddf(kpe2, i2));   // :164
            pick(tt, lp, hp, i0, i1, i2, p0, p1, p2, integ, ph);
        } else {
            pick(tt, lp, hp, kpe0, kpe1, kpe2, kie0, kie1, kie2, kpe, kie);
        }
        bad |= rb.w ^ stamp;
        const float q = p_faddf(tt, -lc);
        cmax = fmaxf(cmax, fabsf(p_faddf(fabsf(p_faddf(fabsf(q), -0.5f)), -0.5f)));
        return __float_as_int(tt);
    };
    auto guards_failed = [&]() { return bad != 0 || !(cmax < 0.5f - 0x1p-15f); };
    auto load_vg = [&](unsigned addr) {
        int2 v;
        asm volatile("ld.shared.v2.b32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(addr));
        return v;
    };
    auto load_half = [&](unsigned addr) {
        int4 v;
        asm volatile("ld.volatile.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr) : "memory");
        return v;
    };
    // after a block: if a guard failed in it, the same block again, the exact way (rare)
    auto settle = [&](int u0, int nb, float integ0, float ph0, int gi0) -> bool {
        if (guards_failed()) {
#ifdef FMRX_PLL_PROFILE
            r.prof_stamp += bad != 0;
            r.prof_c += bad == 0;
            if (bad == 0) {
                if (!(cmax < 1e30f)) r.prof_inv++;
                else if (cmax > 0.5f) r.prof_range++;
                else r.prof_tie++;
            }
#endif
            r.kbase = kbase;
            r.integ = integ0;            // by value through r: nothing on the chain has its address taken
            r.ph = ph0;
            r.gi = gi0;
            n_exact++;
            if (!pll_block_exact(r, u0, nb, lane)) {
#ifdef FMRX_PLL_PROFILE
                r.prof_fatal_exact++;
                if (blockIdx.x == 0 && lane == 0)
                    printf("pll dbg fatal: group base %d block at %d (of %d) gi %d kbase %d\n", base, u0 - base, cnt, r.gi, r.kbase);
                __syncwarp();
#endif
                return false;
            }
            integ = r.integ;
            ph = r.ph;
            kpe = r.kpe;
            kie = r.kie;
            gi = r.gi;
        }
        bad = 0;
        cmax = 0.0f;
        return true;
    };
    auto load_rec = [&](int u) {      // the predictor's record of step u: {phaseEst, u + 1}
        int2 v;
        asm volatile("ld.volatile.shared.v2.b32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(sph_base + (unsigned)(u & (PLL_PH_RING - 1)) * 8u) : "memory");
        return v;
    };
    // pi of the block starting at step u0 > base: from the predictor's phaseEst of step u0 - 1.  The
    // record is fetched and turned into (pi, kbase) in the middle of the block before, beside the
    // chain.  No branch at the block boundary: if the record was not there yet (or is out of range)
    // the block keeps the previous pi and fails its guards.
    float pi_next = 0.0f;
    int kbase_next = 0, seq_next = 0;
    auto next_pi = [&](int u0) {
        const bool have = seq_next == u0 && fabsf(pi_next) < 2097152.0f;
        pi_f = have ? pi_next : pi_f;
        kbase = have ? kbase_next : kbase;
        bad |= (int)!have;
    };
    int t = 0;
    int fatal = 0;               // 1: too many exact blocks; 2: an exact block left the group's grid (r.integ, r.ph, r.gi: the state before it)
    const int n_full = cnt >> 4;
    if (r.cont) {        // (once per group: this one may wait for the load)
        const int2 rec = load_rec(base - 1);
        block_pi(__int_as_float(rec.x), inv_ulp_f, pi_next, kbase_next);
        seq_next = rec.y;
    } else {             // the first block of a group that starts afresh: pi from the exact phaseEst (header)
        pi_next = pi_f;
        kbase_next = kbase;
        seq_next = base;
    }
    for (int b = 0; b < n_full; b++, t += 16) {
        const int u0 = base + t;
        next_pi(u0);
        asm volatile("st.shared.b32 [%0], %1;" ::"r"(kb_base + 4u * (unsigned)(t >> 4)), "r"(kbase) : "memory");
        // the state before the block (after sample u0-1, with Kp*errorD, Ki*errorD of sample u0
        // pending), in case it has to be stepped the exact way
        const float integ0 = integ, ph0 = ph;
        const int gi0 = gi;
        integ = p_faddf(integ, kie);                                  // :163 of sample u0
        ph = p_faddf(ph, p_faddf(kpe, integ));                       // :164
        // neither the rings nor the tables wrap inside a block of 16 (all sizes are multiples
        // of 16 and u0 is one): addresses are base + constant
        const unsigned in_a0 = in_base + (unsigned)(u0 & (PLL_RING - 1)) * (unsigned)sizeof(PllIn);
        const unsigned tab_a0 = tab_base + (unsigned)(u0 & (PLL_TABLES - 1)) * (unsigned)sizeof(PllRow);
        const int stamp = pll_stamp(u0, kbase);
        int gis[16];
        // tables are fetched two steps ahead -- late enough for the candidate warps, early enough
        // to be off the chain; the half of a table with the stamp before its other half
        int4 rb0 = load_half(tab_a0 + 16u), ra0 = load_half(tab_a0);
        int4 rb1 = load_half(tab_a0 + (unsigned)sizeof(PllRow) + 16u), ra1 = load_half(tab_a0 + (unsigned)sizeof(PllRow));
        const int2 vg_last = load_vg(in_a0 + 15u * (unsigned)sizeof(PllIn));
#pragma unroll
        for (int j = 0; j < 16; j++) {
            int4 rb2 = rb1, ra2 = ra1;
            if (j + 2 < 16) {
                rb2 = load_half(tab_a0 + (unsigned)(j + 2) * (unsigned)sizeof(PllRow) + 16u);
                ra2 = load_half(tab_a0 + (unsigned)(j + 2) * (unsigned)sizeof(PllRow));
            }
            gis[j] = step(ra0, rb0, stamp, j == 15);
            ra0 = ra1; rb0 = rb1;
            ra1 = ra2; rb1 = rb2;
            if (j == 8) {            // the next block's pi (the predictor is normally far enough ahead by now)
                const int2 rec = load_rec(u0 + 15);
                block_pi(__int_as_float(rec.x), inv_ulp_f, pi_next, kbase_next);
                seq_next = rec.y;
            }
        }
        // the block's last grid index (:166-167): vi + pi + rint(t + vr)
        gi = vg_last.x + kbase + __float_as_int(p_faddf(p_faddf(__int_as_float(gis[15]), __int_as_float(vg_last.y)), 12582912.0f));
        // park the bits of the 16 t's for the I/O warp (every lane the same stores)
#pragma unroll
        for (int j = 0; j < 16; j += 4)
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(sg_base + 4u * (unsigned)(t + j)), "r"(gis[j]), "r"(gis[j + 1]),
                         "r"(gis[j + 2]), "r"(gis[j + 3])
                         : "memory");
        // (A row is read as two halves, stamp half first, so a row REPLACED between the two loads would pass the
        // check with another step's data.  The only writer that could do that is a candidate warp a whole ring
        // behind, storing the table of step u - PLL_TABLES late; it looks at warp 0's progress immediately before
        // its store and skips it if warp 0 has left its batch behind, and warp 0 cannot cover the 120 steps from
        // there to this row in the few cycles between that look and the store.  Reading the 16 stamps once more
        // here instead cost 7 cycles per step: the dependent LDS + vote sits on the block's critical path.)
        if (!settle(u0, 16, integ0, ph0, gi0)) {
            fatal = 2;
            break;
        }
        if (n_exact > PLL_EXACT_MAX) {
            fatal = 1;               // (more exact blocks than a group without tables costs: give the group up)
            break;
        }
        // progress: lets the candidate warps reuse the table rows of this block, the predictor run on
        asm volatile("st.volatile.shared.b32 [%0], %1;" ::"r"(prog_addr), "r"(u0 + 16) : "memory");
    }
    if (!fatal && t < cnt) {     // the short last block of a launch
        const int u0 = base + t, nb = cnt - t;
        next_pi(u0);
        asm volatile("st.shared.b32 [%0], %1;" ::"r"(kb_base + 4u * (unsigned)(t >> 4)), "r"(kbase) : "memory");
        const float integ0 = integ, ph0 = ph;
        const int gi0 = gi;
        integ = p_faddf(integ, kie);
        ph = p_faddf(ph, p_faddf(kpe, integ));
        for (int j = 0; j < nb; j++) {
            const int u = u0 + j;
            const unsigned row = tab_base + (unsigned)(u & (PLL_TABLES - 1)) * (unsigned)sizeof(PllRow);
            const int4 rb = load_half(row + 16u), ra = load_half(row);
            const int2 vg = load_vg(in_base + (unsigned)(u & (PLL_RING - 1)) * (unsigned)sizeof(PllIn));
            const int tb = step(ra, rb, pll_stamp(u0, kbase), j == nb - 1);
            gi = vg.x + kbase + __float_as_int(p_faddf(p_faddf(__int_as_float(tb), __int_as_float(vg.y)), 12582912.0f));
            asm volatile("st.shared.b32 [%0], %1;" ::"r"(sg_base + 4u * (unsigned)(t + j)), "r"(tb) : "memory");
        }
        fatal = settle(u0, nb, integ0, ph0, gi0) ? 0 : 2;
    }
    r.fatal = fatal;
    r.t_stop = t;
    r.n_exact = n_exact;
    if (fatal == 2)              // (r.integ, r.ph, r.gi: the state before the block that could not be done, as settle() left them)
        return;
    r.integ = integ;
    r.ph = ph;
    r.kpe = kpe;
    r.kie = kie;
    r.gi = gi;
}

__global__ void __launch_bounds__(PLL_THREADS) k_pll(const PllArgs a)
{
    using namespace pllcore;
    extern __shared__ __align__(16) unsigned char pll_dyn_smem[];
    PllIn *s_in = reinterpret_cast<PllIn *>(pll_dyn_smem);      // [PLL_RING]
    __shared__ __align__(16) int2 s_ph[PLL_PH_RING];  // {predicted phaseEst, step + 1}, written by the predictor warp
    __shared__ float s_hdr[3];                        // integrator, phaseEst at the start of the group (warp 0 -> predictor, I/O) and the
                                                      // mean slope of phaseEst over the group before (I/O: where phaseEst is heading)
    __shared__ double s_hdr_tad;                      // trigArg before the group (exact)
    __shared__ int s_kbase;                           // rint(phaseEst/ulp) at the start of the group, less the bits of 1.5 * 2^23
    __shared__ int s_kb_blk[2][PLL_GROUP / 16];       // kbase of every block of the group whose parked values are in s_g[.]
    __shared__ int s_prog;                            // steps of the capture warp 0 has completed (per block of 16), or PLL_ABANDONED
    __shared__ PllRow s_tab[PLL_TABLES];              // candidate tables, a ring over the steps (one-hypothesis groups: PLL_TABLES1 rows of 16 bytes)
    __shared__ __align__(16) int s_g[2][PLL_GROUP];                 // what warp 0 parks per step of the group (see s_spec), double-buffered
    __shared__ double s_grid[2];                      // ulp, 1/ulp of the current group
    __shared__ double s_prep_ulp[2];                  // ulp the ring slots of each group were prepared with
    __shared__ int s_head_ready[PLL_IO_WARPS];        // I/O warp w has prepared its share of the first 64 samples of the group starting HERE
                                                      // (the rest of that group is only touched behind the barrier that ends this one)
    __shared__ double s_ulp_hist[2];                  // ulp the parked grid indices of a group refer to
    __shared__ int s_spec[2];                         // what s_g holds: 0 float trigArg, 1 the bits of t (three-hypothesis steps), 2 the bits of phaseEst
    __shared__ int s_split[2];                        // ... kind 1: only the first s_split steps; float trigArg from there on
    __shared__ int s_flag[5];                         // [0] scheme of the group: 0 none, 3 three hypotheses, 1 one hypothesis; [1] error;
                                                      // [2] re-grid the group's ring slot first (binade change); [3] the group continues the one before (its head
                                                      // is already done); [4] this pass repeats the group of the pass before (its tables failed)
    __shared__ int s_redo;                            // warp 0, at the end of a pass: do this group again (on the one-hypothesis scheme)

    const int c = blockIdx.x;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const float *p = a.pilot + (size_t)c * a.pilot_stride;
    float *tr = a.trig + (size_t)c * a.if_stride + a.if_off;
    float *st = a.state + 8 * (size_t)c;
    const int n = a.n_if;

    Consts k;
    k.kp = a.prm.kp;
    k.ki = a.prm.ki;
    k.w = a.prm.w;
    const TrigK &K = a.kconst;       // kernel-parameter constant bank: direct DFMA operands

    // every warp derives the (uniform) start of the trigOffset sequence itself
    const float toff0 = st[5];
    const bool regular = toff_is_regular(toff0);
    const int t0 = regular ? (int)toff0 : 0;
    // roles by scheduler (warp & 3): 0 = the chain (warp 0; warps 4, 8 idle), 1 = I/O and the predictor, 2 and 3 = candidates
    const int role = warp & 3;
    const int io_id = warp >> 2;                          // 0, 1 for warps 1, 5 (2: warp 9, the predictor)
    const int cand_id = (warp >> 2) * 2 + role - 2;       // 0..5 for warps 2, 3, 6, 7, 10, 11

    // I/O warp: one lane per sample, off-chain inputs of the samples of a group into the ring.  The one-hypothesis
    // inputs extrapolate phaseEst from e_ph, its value before step e_base, with e_slope per step.
    auto prepare_one = [&](int u, float e_slope, float e_ph, int e_base) {
        {
            const float pvv = (u < n) ? p[u] : 1.0f;
            const float pnx = (u + 1 < n) ? p[u + 1] : 1.0f;
            PllIn in;
            in.x = pvv;
            in.inv_x = 1.0 / (double)pvv;                                // IEEE divide
            const float toff = (float)min(t0 + u + 1, 16777216);         // exact: <= 2^24
            in.v = __dmul_rn(k.w, (double)toff);
            // v on the float grid of the current binade: integer part and remainder
            const double qv = grid_round(in.v, s_grid[1]);
            in.vi = grid_index(qv);
            in.vr = __double2float_rn(__fma_rn(in.v, s_grid[1], -p_add(qv, -FMRX_RINT_MAGIC)));
            in.c3 = predictor_c(k, pvv, (float)min(t0 + u, 16777216));      // trigOffset BEFORE this step
            in.h1 = onehyp_inputs(in.v, e_ph, e_slope, u + 1 - e_base, pnx);
            s_in[u & (PLL_RING - 1)] = in;
        }
    };
    auto prepare = [&](int base, float e_slope, float e_ph, int e_base) {
        for (int j = 32 * io_id; j < PLL_GROUP; j += 32 * PLL_IO_WARPS)
            prepare_one(base + j + lane, e_slope, e_ph, e_base);
        if (lane == 0 && io_id == 0)
            s_prep_ulp[(base / PLL_GROUP) & 1] = s_grid[0];
    };
    // the first samples of the NEXT group are read before the barrier that ends this one (by the predictor and the
    // candidate warps doing its head, by an exact block at the very end of this group): wait for the I/O warps' word
    auto head_ready = [&](int next_base) -> bool {
        for (int spin = 0; spin < PLL_SPIN_LIMIT; spin++) {
            int a0, a1;
            asm volatile("ld.volatile.shared.b32 %0, [%1];" : "=r"(a0) : "r"(smem_u32(&s_head_ready[0])) : "memory");
            asm volatile("ld.volatile.shared.b32 %0, [%1];" : "=r"(a1) : "r"(smem_u32(&s_head_ready[1])) : "memory");
            if (a0 == next_base && a1 == next_base)
                return true;
        }
        return false;
    };

    for (int i = threadIdx.x; i < PLL_PH_RING; i += PLL_THREADS)
        s_ph[i] = make_int2(0, 0);
    for (int i = threadIdx.x; i < PLL_TABLES; i += PLL_THREADS) {
        s_tab[i].lp = PLL_ROW_INVALID;
        s_tab[i].stamp = 0;
        s_tab[i].kie0 = 0.0f;            // (the stamp word of the one-hypothesis row in the table's first half)
    }
    if (threadIdx.x == 0) {
        s_flag[1] = 0;
        s_redo = 0;
        s_head_ready[0] = s_head_ready[1] = -1;
    }
    // warp 0 owns the recurrence state
    Chain ch;
    bool stale = false;              // ch's sincos leftovers lag behind ch.tad (after speculative groups)
    bool have_ed = false;            // kpe_next/kie_next below belong to the next sample
    float kpe_next = 0.0f, kie_next = 0.0f;
    bool dead = false;               // a hand-off timed out: stay on the checked path
    int backoff = 0, skip = 0;       // after a failed table group: `skip` groups without the tables, then retry
    int prev_scheme = 0;
    float ph_hdr_prev = 0.0f;        // phaseEst at the start of the group before (lane 0 of warp 0)
    int n_groups = 0, n_redone = 0, n_exact = 0, prev_exact = 0;
    float pred_integ = 0.0f, pred_ph = 0.0f;          // the predictor's state (warp 9)
#ifdef FMRX_PLL_PROFILE
    long long prof_steps_cyc = 0, prof_wait = 0, prof_pre = 0, prof_one_cyc = 0;
    long long prof_t_end = 0, prof_bar2 = 0, prof_hdr = 0, prof_bar1 = 0, prof_post = 0, prof_post2 = 0, prof_c1 = 0;    // warp 0: where a group's time outside its steps goes
    const long long prof_k0 = clock64();
    int prof_steps = 0, prof_n_stamp = 0, prof_n_c = 0, prof_n_fe = 0, prof_n_fm = 0;
    int prof_n_tie = 0, prof_n_range = 0, prof_n_inv = 0;
    int prof_one_steps = 0, prof_one_groups = 0, prof_one_exact = 0, prof_one_short = 0, prof_checked = 0;
    __shared__ int s_prof[8];        // candidate warps: why a table was not emitted
    __shared__ long long s_prof1[8]; // one-hypothesis groups: [0] predictor cycles waiting for warp 0, [1] predictor cycles stepping, [2] predictor blocks
                                     // redone with the reduction, [3] candidate pass cycles (warp 2), [4] passes, [5] candidate cycles waiting for records
    if (threadIdx.x < 8) {
        s_prof[threadIdx.x] = 0;
        s_prof1[threadIdx.x] = 0;
    }
#endif
    if (warp == 0) {
        ch.integ = st[0];
        ch.ph = st[1];
        ch.fi = st[2];
        ch.fq = st[3];
        ch.toff = toff0;
        chain_load(ch, k);
        if (lane == 0) {
            s_grid[0] = ch.ulp;
            s_grid[1] = ch.inv_ulp;
        }
    }
    __syncthreads();
    if (role == 1 && io_id < PLL_IO_WARPS) {
        prepare(0, st[0], st[1], 0);
    }
    __syncthreads();

    for (int base = 0, g = 0; base < n;) {
        const int cnt = min(PLL_GROUP, n - base);
        Chain ck;
        // ---- group header (warp 0) ----
#ifdef FMRX_PLL_PROFILE
        const long long prof_h0 = clock64();
        if (warp == 0 && prof_t_end)
            prof_bar2 += prof_h0 - prof_t_end;
#endif
        if (warp == 0) {
            ck = ch;
            const bool again = s_redo != 0;          // (uniform: written before the barrier that ended the last pass)
            // (disarmed: a state whose feedback pair does not belong to its trigArg -- a hand-made one -- or a
            // trigArg of 0 or beyond 2^24: the checked step sorts that out)
            const bool usable = regular && !dead && ch.binade != FMRX_DISARMED && fabs(ch.tad) <= (double)FMRX_FAST_TRIG_MAX;
            // The hypotheses of a three-hypothesis step are NEIGHBOURING float-grid points of trigArg, which presumes
            // that phaseEst moves on a grid at least as fine.  Where the reference hands the PLL if_fs*interp (modes
            // 2/3) phaseEst cancels w*trigOffset, trigArg is a small difference of large floats and its possible values
            // lie a whole phaseEst spacing (thousands of its own grid steps) apart: there -- and while the tables are
            // backing off after a failure, e.g. on a loop that locks onto nothing -- the one-hypothesis scheme runs.
            // (Tables also serve the regime past trigOffset == 2^24, where trigArg freezes on two grid points
            // and the loop dithers across a float rounding boundary: tests/test_gpu_operators.py::
            // test_pll_long_run_past_counter_saturation and the >= 70 s pipeline runs of tests/test_gpu_long_runs.py.)
            const bool can3 = usable && !again && skip == 0 && (double)fabsf(ch.ph) < ch.ulp * 16777216.0;
            // the group's ring slot was prepared while the group before ran, with ITS grid: after a binade change
            // (vi, vr) are re-made for the new one before anything else happens (below, all warps)
            const bool regrid = can3 && s_prep_ulp[g & 1] != ch.ulp;
            const int scheme = can3 ? 3 : usable ? 1 : 0;
            // the group before ran on tables to its end and hardly needed the exact step: predictor and
            // candidates did our head, and the predictor carries on from its own state (otherwise it
            // restarts from the exact one: it may have drifted)
            const bool cont = scheme == 3 && prev_scheme == 3 && have_ed && prev_exact <= 2 && !regrid;
#ifdef FMRX_PLL_PROFILE
            prof_post += clock64() - prof_h0;        // (header, first part: copy and decisions)
#endif
            if (scheme != prev_scheme || again) {
                // the other scheme's rows (and records) share the rings: nothing of them may be taken for this group's
                for (int i = lane; i < PLL_TABLES; i += 32) {
                    s_tab[i].lp = PLL_ROW_INVALID;
                    s_tab[i].stamp = 0;
                    s_tab[i].kie0 = 0.0f;
                }
                for (int i = lane; i < PLL_PH_RING; i += 32)
                    s_ph[i] = make_int2(0, 0);
            } else if (scheme == 3 && !cont && base > 0) {
                // ... and then the head that the group before prepared must go: its tables carry this
                // group's stamps and its records this group's sequence numbers, but their block pi came
                // from the OLD predictor run, while warp 0 now takes pi of the first block from the exact
                // phaseEst -- where the two differ (phaseEst/ulp near a half-integer: a loop sitting on a
                // rounding boundary, e.g. past counter saturation) the thresholds select a neighbouring
                // hypothesis without any guard noticing (reproduced on the host: tests/pll_model.cpp,
                // pll_model_stale_head).  Everyone is behind the barrier that ended the last group.
                for (int i = lane; i < PLL_HEAD; i += 32) {
                    s_tab[(base + i) & (PLL_TABLES - 1)].lp = PLL_ROW_INVALID;
                    s_tab[(base + i) & (PLL_TABLES - 1)].stamp = 0;
                    s_ph[(base + i) & (PLL_PH_RING - 1)] = make_int2(0, 0);
                }
            }
            if (lane == 0) {
                s_flag[0] = scheme;
                s_flag[2] = regrid;
                s_grid[0] = ch.ulp;
                s_grid[1] = ch.inv_ulp;
                s_flag[3] = cont;
                s_flag[4] = again;
                s_kbase = __float_as_int(p_faddf(p_fmulf(ch.ph, (float)ch.inv_ulp), 12582912.0f)) - 0x4B400000 - 0x4B400000;
                s_hdr[0] = ch.integ;
                s_hdr[1] = ch.ph;
                // where phaseEst is heading: its mean slope over the group before (at the start of a launch: the
                // integrator, which is that slope on a loop at rest -- but e.g. in modes 2/3 the phase detector's
                // output has a mean of its own, and 3000 steps ahead the difference is whole turns)
                if (!again) {
                    s_hdr[2] = g > 0 ? p_fmulf(p_faddf(ch.ph, -ph_hdr_prev), 1.0f / PLL_GROUP) : ch.integ;
                    ph_hdr_prev = ch.ph;
                }
                s_hdr_tad = ch.tad;
                s_prog = base;
            }
        }
#ifdef FMRX_PLL_PROFILE
        const long long prof_h1 = clock64();
#endif
        __syncthreads();
#ifdef FMRX_PLL_PROFILE
        if (warp == 0) {
            prof_hdr += prof_h1 - prof_h0;
            prof_bar1 += clock64() - prof_h1;
        }
#endif
        if (s_flag[2]) {         // (uniform)
            const double iu = s_grid[1];
            for (int j = threadIdx.x; j < PLL_GROUP; j += PLL_THREADS) {
                PllIn &in = s_in[(base + j) & (PLL_RING - 1)];
                const double qv = grid_round(in.v, iu);
                in.vi = grid_index(qv);
                in.vr = __double2float_rn(__fma_rn(in.v, iu, -p_add(qv, -FMRX_RINT_MAGIC)));
            }
            if (threadIdx.x == 0)
                s_prep_ulp[g & 1] = s_grid[0];
            __syncthreads();
        }
        const int scheme = s_flag[0];
        const bool spec = scheme == 3;
        const bool again = s_flag[4] != 0;
        const double ulp = s_grid[0], inv_ulp = s_grid[1];
#ifdef FMRX_PLL_PROFILE
        const long long prof_ga = clock64();
#endif

        if (warp == 0) {
            // ================= the chain =================
            if (lane == 0)
                s_redo = 0;          // (every warp read it after the barrier that ended the last pass)
            if (!again)
                n_groups++;
            bool good = scheme != 0;
            bool redo = false;
            bool regridded = false;  // a table group that ended without tables after a binade change
            int split = 0;           // three-hypothesis groups: steps parked as bits of t; the rest (after a binade change) as float trigArg
            int parked = 0;          // what s_g holds at the end (s_spec)
            if (scheme == 3) {
                float integ = ch.integ, ph = ch.ph;
                float kpe = kpe_next, kie = kie_next;        // Kp*errorD, Ki*errorD of the sample about to run
                if (!have_ed) {      // first group, or after a checked group: from the known trigArg
                    const PllIn i0 = s_in[base & (PLL_RING - 1)];
                    const Feedback f0 = make_feedback(K, ch.tad, pll_turn(i0.x), i0.inv_x, nullptr, nullptr);
                    const float ed = error_from_feedback(f0, i0.x, (double)i0.x, good);
                    kpe = p_fmulf(k.kp, ed);
                    kie = p_fmulf(k.ki, ed);
                }
                const float inv_ulp_f = (float)inv_ulp;                          // a power of two
                float pi_f = 0.0f;
                int cu_base = 0;
                // centre pi on the current phaseEst
                auto recentre = [&]() {
                    const float pm = p_faddf(p_fmulf(ph, inv_ulp_f), 12582912.0f);   // rint via 1.5*2^23
                    pi_f = p_faddf(pm, -12582912.0f);
                    cu_base = __float_as_int(pm) - 0x4B400000 - 0x4B400000;
                    good &= fabsf(pi_f) < 2097152.0f;                              // |phaseEst/ulp| < 2^21
                };
                recentre();
                // wait (bounded) for the first tables of the group; afterwards the candidate
                // warps run ahead and a late table only clears `good`
#ifdef FMRX_PLL_PROFILE
                const long long prof_w0 = clock64();
                prof_pre += prof_w0 - prof_ga;
#endif
                {   // lane t watches table t
                    const bool need = lane < 16 && lane < cnt;           // the first block's tables
                    int spin = 0;
                    for (;;) {
                        const int z = ld_v4(&s_tab[(base + (lane & 15)) & (PLL_TABLES - 1)].kpe2).w;      // the stamp
                        if (__all_sync(0xffffffffu, !need || (z & 0x3ffffff) == base + 1) || ++spin >= PLL_SPIN_LIMIT)
                            break;
                    }
                    if (spin >= PLL_SPIN_LIMIT) {
                        dead = true;
                        good = false;
                        if (lane == 0)
                            s_flag[1] = 1;
                    }
                }
#ifdef FMRX_PLL_PROFILE
                prof_wait += clock64() - prof_w0;
#endif
                // the steps themselves: a separately compiled function, so that its instruction
                // schedule -- which IS the step time -- does not move when anything else in this
                // kernel changes
                TableRun r;
                r.integ = integ;
                r.ph = ph;
                r.kpe = kpe;
                r.kie = kie;
                r.inv_ulp_f = inv_ulp_f;
                r.pi_f = pi_f;
                r.kbase = cu_base;
                r.base = base;
                r.cnt = cnt;
                r.in_base = smem_u32(&s_in[0]) + (unsigned)offsetof(PllIn, vi);   // {vi, vr} of a slot
                r.tab_base = smem_u32(&s_tab[0]);
                r.sg_base = smem_u32(&s_g[g & 1][0]);
                r.prog_addr = smem_u32(&s_prog);
                r.sph_base = smem_u32(&s_ph[0]);
                r.kb_base = smem_u32(&s_kb_blk[g & 1][0]);
                r.head_addr = smem_u32(&s_head_ready[0]);
                r.cont = s_flag[3];
#ifdef FMRX_PLL_PROFILE
                r.prof_stamp = r.prof_c = r.prof_fatal_exact = 0;
                r.prof_tie = r.prof_range = r.prof_inv = 0;
#endif
                r.gi = __double2int_rn(p_mul(ch.tad, inv_ulp));                  // exact: trigArg is on the grid
                r.n_exact = 0;
                r.fatal = 0;
                r.ring = s_in;
                r.k = k;
                r.ulp = ulp;
                r.toff_base = ch.toff;
                if (good) {
                    __syncwarp();
#ifdef FMRX_PLL_PROFILE
                    const long long prof_c0 = clock64();
#endif
                    pll_table_group(r, lane);
#ifdef FMRX_PLL_PROFILE
                    prof_c1 = clock64();
                    prof_steps_cyc += prof_c1 - prof_c0;
                    prof_steps += cnt;
                    prof_n_stamp += r.prof_stamp;
                    prof_n_c += r.prof_c;
                    prof_n_fe += r.prof_fatal_exact;
                    prof_n_tie += r.prof_tie;
                    prof_n_range += r.prof_range;
                    prof_n_inv += r.prof_inv;
                    prof_n_fm += r.fatal && !r.prof_fatal_exact;
#endif
                    good = r.fatal == 0;
                    n_exact += r.n_exact;
                    prev_exact = r.n_exact;
                }
                if (good && r.fatal == 0)
                    split = cnt;
                if (r.fatal == 2) {
                    // trigArg left the binade the group's grid belongs to (in mode 0 it grows with w*trigOffset: some
                    // twenty times per capture, most of them in its first seconds).  The blocks before are done and
                    // parked; the rest of the group goes without tables from the state before the block at hand --
                    // no second pass -- and the next group starts afresh on the new grid (its ring slot is
                    // re-gridded in its header pass).
                    asm volatile("st.volatile.shared.b32 [%0], %1;" ::"r"(smem_u32(&s_prog)), "r"(PLL_ABANDONED) : "memory");
                    split = r.t_stop;
                    onehyp_chain_at(ch, r.integ, r.ph, (float)min(t0 + base + r.t_stop, 16777216), p_mul((double)r.gi, ulp));
                    pll_group_checked(ch, k, s_in, base, r.t_stop, cnt, regular, smem_u32(&s_g[g & 1][0]), false);
                    stale = false;
                    have_ed = false;
                    parked = 1;
                    regridded = true;        // (prev_scheme = 0 below: nothing of this group's head work is taken over)
                } else if (good) {
                    ch.integ = r.integ;
                    ch.ph = r.ph;
                    ch.toff = (float)min(t0 + base + cnt, 16777216);
                    ch.tad = p_mul((double)r.gi, ulp);
                    stale = true;
                    have_ed = true;
                    kpe_next = r.kpe;
                    kie_next = r.kie;
                    backoff = 0;
                    parked = 1;
                } else {
                    // the predictor and the candidate warps stop working on this group; it is done again, on the
                    // one-hypothesis scheme, and the tables rest for a while
                    asm volatile("st.volatile.shared.b32 [%0], %1;" ::"r"(smem_u32(&s_prog)), "r"(PLL_ABANDONED) : "memory");
                    n_redone++;
                    backoff = min(backoff < 4 ? backoff + 1 : 2 * backoff, PLL_BACKOFF_MAX);       // 1, 2, 3, 4, 8, 16, ...
                    skip = backoff;
                    ch = ck;
                    have_ed = false;
                    redo = !dead;
                    if (!redo) {         // a hand-off timed out: no second pass, the group goes without tables right here
                        if (stale) {
                            chain_refresh(ch);
                            stale = false;
                        }
                        pll_group_checked(ch, k, s_in, base, 0, cnt, regular, smem_u32(&s_g[g & 1][0]), false);
                    }
                }
            } else if (scheme == 1) {
                if (skip > 0 && !again)
                    skip--;
                OneRun r;
                r.integ = ch.integ;
                r.ph = ch.ph;
                r.base = base;
                r.cnt = cnt;
                r.tab_base = smem_u32(&s_tab[0]);
                r.sg_base = smem_u32(&s_g[g & 1][0]);
                r.prog_addr = smem_u32(&s_prog);
                r.ring = s_in;
                r.k = k;
                r.toff_base = ch.toff;
                r.tad0 = ch.tad;
                r.n_exact = 0;
                r.done = 0;
                r.timed_out = 0;
                __syncwarp();
#ifdef FMRX_PLL_PROFILE
                const long long prof_c0 = clock64();
#endif
                pll_onehyp_group(r, lane);
#ifdef FMRX_PLL_PROFILE
                prof_one_cyc += clock64() - prof_c0;
                prof_one_steps += r.done;
                prof_one_groups++;
                prof_one_exact += r.n_exact;
                prof_one_short += r.done < cnt;
#endif
                n_exact += r.n_exact;
                if (r.timed_out) {
                    dead = true;
                    if (lane == 0)
                        s_flag[1] = 1;
                }
                // the state after r.done steps; what is left of the group (the predictor lost the trajectory) goes without tables
                const int last = base + r.done - 1;
                const double tad = r.done ? onehyp_trigarg(s_in[last & (PLL_RING - 1)].v, r.ph) : ch.tad;
                if (r.done < cnt) {
                    asm volatile("st.volatile.shared.b32 [%0], %1;" ::"r"(smem_u32(&s_prog)), "r"(PLL_ABANDONED) : "memory");
                    onehyp_chain_at(ch, r.integ, r.ph, (float)min(t0 + base + r.done, 16777216), tad);
                    pll_group_checked(ch, k, s_in, base, r.done, cnt, regular, smem_u32(&s_g[g & 1][0]), true);
                    stale = false;
                } else {
                    ch.integ = r.integ;
                    ch.ph = r.ph;
                    ch.toff = (float)min(t0 + base + cnt, 16777216);
                    ch.tad = tad;
                    stale = true;
                    if (fabs(tad) <= (double)FMRX_FAST_TRIG_MAX)
                        chain_arm(ch);           // the binade may have changed (the header wants ulp and binade)
                    else
                        onehyp_chain_at(ch, r.integ, r.ph, ch.toff, tad), stale = false;
                }
                have_ed = false;
                parked = 2;
            } else {
                if (skip > 0)
                    skip--;
                if (stale) {         // bring the sincos leftovers up to date with ch.tad
                    chain_refresh(ch);
                    stale = false;
                }
                // the group without tables (a separately compiled function, like the table steps)
#ifdef FMRX_PLL_PROFILE
                prof_checked++;
#endif
                pll_group_checked(ch, k, s_in, base, 0, cnt, regular, smem_u32(&s_g[g & 1][0]), false);
                have_ed = false;
                parked = 0;
            }
            prev_scheme = redo || regridded ? 0 : scheme;
            if (lane == 0) {
                s_spec[g & 1] = parked;
                s_split[g & 1] = split;
                s_ulp_hist[g & 1] = ulp;
                s_redo = redo;
            }
#ifdef FMRX_PLL_PROFILE
            prof_t_end = clock64();
            if (prof_c1)
                prof_post2 += prof_t_end - prof_c1;
            prof_c1 = 0;
#endif
        } else if (role >= 2) {
            // ================= candidate tables =================
            if (scheme == 3) {
                // A warp evaluates eight consecutive steps at once, one per quad of lanes: lane 4*s + j
                // takes step base + 8*cand_id + s (mod 8*PLL_CAND_WARPS) and the grid point G_c - 1 + j
                // around the predictor's trigArg of that step (j = 3 is idle work: SIMT).
                const int sq = lane >> 2, jq = lane & 3;
                const unsigned prog_a = smem_u32(&s_prog);
                auto progress = [&]() {
                    int v;
                    asm volatile("ld.volatile.shared.b32 %0, [%1];" : "=r"(v) : "r"(prog_a) : "memory");
                    return v;
                };
                // steps [first, end): this group's (less its head if the group before did it) and the head
                // of the next one; batch q = step / 8 belongs to warp q mod PLL_CAND_WARPS
                const bool cont = s_flag[3] != 0;
                const int first = base + (cont ? PLL_HEAD : 0);
                const int end = base + cnt + (base + cnt + PLL_HEAD <= n ? PLL_HEAD : 0);
                const int q0 = first / PLL_BATCH;
                bool head_seen = false;
                for (int ub8 = first + ((cand_id - q0 % PLL_CAND_WARPS + PLL_CAND_WARPS) % PLL_CAND_WARPS) * PLL_BATCH; ub8 < end;
                     ub8 += PLL_BATCH * PLL_CAND_WARPS) {
                    if (!head_seen && cnt == PLL_GROUP && ub8 + PLL_BATCH >= base + cnt) {      // samples of the next group from here on
                        if (!head_ready(base + PLL_GROUP)) {
                            s_flag[1] = 1;
                            break;
                        }
                        head_seen = true;
                    }
                    const bool live = ub8 + sq < end;
                    const int u = ub8 + (live ? sq : 0);
                    const double v = s_in[u & (PLL_RING - 1)].v;
                    const int vi = s_in[u & (PLL_RING - 1)].vi;
                    const float vr = s_in[u & (PLL_RING - 1)].vr;
                    const PllIn nx = s_in[(u + 1) & (PLL_RING - 1)];     // the sample the result is for
                    // the predictor publishes in order: once the last record of the batch is there, all are
                    const int last = min(ub8 + PLL_BATCH - 1, end - 1);
                    int prog = 0, spin = 0;
                    for (;; spin++) {
                        const int seq = ld_v2(&s_ph[last & (PLL_PH_RING - 1)]).y;
                        if (seq - (last + 1) >= 0 || spin >= PLL_SPIN_LIMIT)
                            break;
                        if ((spin & 7) == 7 && (prog = progress()) == PLL_ABANDONED)
                            break;
                    }
                    if (prog == PLL_ABANDONED)
                        break;
                    if (spin >= PLL_SPIN_LIMIT) {
                        s_flag[1] = 1;
                        break;
                    }
                    const int2 pr = ld_v2(&s_ph[u & (PLL_PH_RING - 1)]);
                    // pi of the block these eight steps belong to: as warp 0 takes it
                    const int ub = ub8 & ~15;
                    int kb = s_kbase;
                    bool have_pi = true;
                    if (ub != base || cont) {
                        const int2 rb = ld_v2(&s_ph[(ub - 1) & (PLL_PH_RING - 1)]);
                        float pif;
                        block_pi(__int_as_float(rb.x), (float)inv_ulp, pif, kb);
                        have_pi = rb.y == ub;
                    }
                    // (a record that is not this step's: the warp fell a whole ring behind -- no table then)
                    const bool have = pr.y == u + 1 && have_pi;
                    // this lane's grid point: G_c - 1 + j
                    const int gc = grid_index(grid_round(p_add(v, (double)__int_as_float(pr.x)), inv_ulp));
                    const int gl = gc - 1 + jq;
                    const double tad = p_mul((double)gl, ulp);                        // exact
                    const Feedback f = make_feedback(K, tad, pll_turn(nx.x), nx.inv_x, nullptr, nullptr);
                    // the float grid of the binade is only right strictly inside it
                    const int ag = gl < 0 ? -gl : gl;
                    bool ok = have && ag > (1 << 23) && ag < (1 << 24);
#ifdef FMRX_PLL_PROFILE
                    const bool prof_ok_b = ok;
#endif
                    const float ed = error_from_feedback(f, nx.x, (double)nx.x, ok);  // :159-161 of sample u+1
                    // the table is good if the guards of its three grid points held
                    const int n1 = gc - (vi + kb) - 0x4B400000;                       // G_c - (vi + pi): small
#ifdef FMRX_PLL_PROFILE
                    if (live && jq < 3 && blockIdx.x == 0) {
                        if (!(pr.y == u + 1)) atomicAdd(&s_prof[0], 1);
                        else if (!have_pi) atomicAdd(&s_prof[1], 1);
                        else if (!prof_ok_b) atomicAdd(&s_prof[2], 1);
                        else if (!ok) atomicAdd(&s_prof[fabs(f.phi) >= FMRX_SEAM_PHI_MAX ? 3 : 4], 1);
                        else if (!(n1 >= -60 && n1 <= 60)) atomicAdd(&s_prof[5], 1);
                        else atomicAdd(&s_prof[6], 1);
                    }
#endif
                    ok = ok && n1 >= -60 && n1 <= 60;
                    const unsigned oks = __ballot_sync(0xffffffffu, ok || jq == 3);
                    const bool valid = ((oks >> (4 * sq)) & 7u) == 7u;
                    // the rows still hold the tables of steps u - PLL_TABLES: wait until warp 0 is past them
                    for (spin = 0; (prog = progress()) != PLL_ABANDONED && prog - (ub8 + PLL_BATCH - PLL_TABLES) < 0 && spin < PLL_SPIN_LIMIT;
                         spin++)
                        ;
                    if (prog == PLL_ABANDONED)
                        break;
                    if (spin >= PLL_SPIN_LIMIT) {
                        s_flag[1] = 1;
                        break;
                    }
                    // one store instruction writes the eight tables: 8 bytes per lane, 32 per quad
                    // (a warp that fell so far behind that warp 0 has already left this batch behind -- it
                    // stepped those blocks the exact way -- must not store: the rows may by now belong to the
                    // steps one ring further on)
                    if (live && prog - (ub8 + PLL_BATCH) < 0) {
                        const int lo = jq < 3 ? __float_as_int(p_fmulf(k.kp, ed))
                                              : __float_as_int(valid ? p_faddf(p_faddf((float)n1, -0.5f), -vr) : PLL_ROW_INVALID);
                        const int hi = jq < 3 ? __float_as_int(p_fmulf(k.ki, ed)) : pll_stamp(u & ~15, kb);
                        asm volatile("st.volatile.shared.v2.b32 [%0], {%1, %2};" ::"r"(smem_u32(&s_tab[u & (PLL_TABLES - 1)]) + 8u * (unsigned)jq),
                                     "r"(lo), "r"(hi)
                                     : "memory");
                    }
                }
            } else if (scheme == 1) {
                // One-hypothesis rows, one step per lane: the exact phase detector of sample u for the trigArg the
                // reference forms (:167) from the predictor's phaseEst of step u - 1 (the group's first step: from the
                // exact trigArg in the header).  Batch q of 32 steps belongs to warp q mod PLL_CAND_WARPS.
                const unsigned prog_a = smem_u32(&s_prog);
                auto progress = [&]() {
                    int v;
                    asm volatile("ld.volatile.shared.b32 %0, [%1];" : "=r"(v) : "r"(prog_a) : "memory");
                    return v;
                };
                const int end = base + cnt;
                for (int ub = base + cand_id * PLL_BATCH1; ub < end; ub += PLL_BATCH1 * PLL_CAND_WARPS) {
                    const bool live = ub + lane < end;
                    const int u = live ? ub + lane : end - 1;
                    const int last = min(ub + PLL_BATCH1 - 1, end - 1);
                    int prog = 0, spin = 0;
#ifdef FMRX_PLL_PROFILE
                    const long long cw0 = clock64();
#endif
                    for (;; spin++) {
                        const int seq = ld_v2(&s_ph[last & (PLL_PH_RING - 1)]).y;
                        if (seq == last + 1 || spin >= PLL_SPIN_LIMIT)
                            break;
                        if ((spin & 7) == 7 && (prog = progress()) == PLL_ABANDONED)
                            break;
                    }
                    if (prog == PLL_ABANDONED)
                        break;
                    if (spin >= PLL_SPIN_LIMIT) {
                        s_flag[1] = 1;
                        break;
                    }
#ifdef FMRX_PLL_PROFILE
                    const long long cw1 = clock64();
#endif
                    const int2 cur = ld_v2(&s_ph[u & (PLL_PH_RING - 1)]);
                    bool ok = cur.y == u + 1;
                    double tad = s_hdr_tad;
                    if (u != base) {
                        const int2 prv = ld_v2(&s_ph[(u - 1) & (PLL_PH_RING - 1)]);
                        ok = ok && prv.y == u;
                        tad = onehyp_trigarg(s_in[(u - 1) & (PLL_RING - 1)].v, __int_as_float(prv.x));
                    }
                    const float x = s_in[u & (PLL_RING - 1)].x;
                    const double inv_x = s_in[u & (PLL_RING - 1)].inv_x;
                    ok = ok && fabs(tad) <= (double)FMRX_FAST_TRIG_MAX;
                    const Feedback f = make_feedback(K, ok ? tad : 0.0, pll_turn(x), inv_x, nullptr, nullptr);
                    const float ed = error_from_feedback(f, x, (double)x, ok);        // :159-161 of sample u
                    // the rows still hold steps u - PLL_TABLES1: wait until warp 0 is past them
                    for (spin = 0; (prog = progress()) != PLL_ABANDONED && prog - (ub + PLL_BATCH1 - PLL_TABLES1) < 0 && spin < PLL_SPIN_LIMIT; spin++)
                        ;
                    if (prog == PLL_ABANDONED)
                        break;
                    if (spin >= PLL_SPIN_LIMIT) {
                        s_flag[1] = 1;
                        break;
                    }
                    if (live)
                        st_v4(reinterpret_cast<PllRow1 *>(&s_tab[0]) + (u & (PLL_TABLES1 - 1)), __float_as_int(p_fmulf(k.kp, ed)),
                              __float_as_int(p_fmulf(k.ki, ed)), cur.x, ok ? u + 1 : -(u + 1));
#ifdef FMRX_PLL_PROFILE
                    if (lane == 0 && blockIdx.x == 0 && cand_id == 0) {
                        s_prof1[3] += clock64() - cw1;
                        s_prof1[4] += 1;
                        s_prof1[5] += cw1 - cw0;
                    }
#endif
                }
            }
        } else if (warp == PLL_PRED_WARP) {
            // ================= the run-ahead predictor =================
            if (scheme == 3) {
                // The same recurrence with the phase detector replaced by what it computes up to
                // rounding (fmrx_pll_core.h, predictor_step): nine dependent float operations per
                // step, so it runs about twice as fast as warp 0 can consume tables, and its phaseEst
                // stays within a grid step or two of the exact one for the whole group (it restarts
                // from the exact state at every group).  It is only ever used to CENTRE the tables.
                // a group that continues the one before finds its head done and the predictor's state
                // where that left it (it needs no restart: tests/test_pll_model.py runs it for 20 s)
                const bool cont = s_flag[3] != 0;
                if (!cont) {
                    pred_integ = s_hdr[0];
                    pred_ph = s_hdr[1];
                }
                float integ = pred_integ, ph = pred_ph;
                const unsigned prog_a = smem_u32(&s_prog);
                const unsigned ph_a = smem_u32(&s_ph[0]);
                const unsigned c_a = smem_u32(&s_in[0]) + (unsigned)offsetof(PllIn, c3);
                int prog = base;
                const int t_end = cnt + (base + cnt + PLL_HEAD <= n ? PLL_HEAD : 0);
                for (int t = cont ? PLL_HEAD : 0; t < t_end; t += 16) {
                    const int u0 = base + t;
                    if (t == PLL_GROUP && !head_ready(base + PLL_GROUP)) {      // the head of the next group starts here
                        s_flag[1] = 1;
                        break;
                    }
                    int spin = 0;                // stay within PLL_PRED_LEAD of warp 0
                    do {
                        asm volatile("ld.volatile.shared.b32 %0, [%1];" : "=r"(prog) : "r"(prog_a) : "memory");
                    } while (prog != PLL_ABANDONED && u0 - prog > PLL_PRED_LEAD - 16 && ++spin < PLL_SPIN_LIMIT);
                    if (prog == PLL_ABANDONED || spin >= PLL_SPIN_LIMIT)
                        break;
                    // the 16 c's of the block first (they do not wrap inside it), then the dependent steps
                    const unsigned c_a0 = c_a + (unsigned)(u0 & (PLL_RING - 1)) * (unsigned)sizeof(PllIn);
                    const unsigned ph_a0 = ph_a + (unsigned)(u0 & (PLL_PH_RING - 1)) * 8u;
                    float cs[16];
#pragma unroll
                    for (int j = 0; j < 16; j++)
                        asm volatile("ld.shared.b32 %0, [%1];" : "=f"(cs[j]) : "r"(c_a0 + (unsigned)j * (unsigned)sizeof(PllIn)));
#pragma unroll
                    for (int j = 0; j < 16; j++) {
                        predictor_step(k, cs[j], integ, ph);         // steps past the end of a short last block are never used
                        asm volatile("st.volatile.shared.v2.b32 [%0], {%1, %2};" ::"r"(ph_a0 + (unsigned)j * 8u), "r"(__float_as_int(ph)),
                                     "r"(u0 + j + 1)
                                     : "memory");
                    }
                }
                pred_integ = integ;
                pred_ph = ph;
            } else if (scheme == 1) {
                // The recurrence in the reference's own operation order with the phase detector replaced by
                // wrap(pi*(x < 0) - trigArg) in float (fmrx_pll_core.h, onehyp_predictor_step): FMUL + 8 dependent
                // FADD per step.  Restarted from the exact state at every group; its phaseEst of every step is what
                // the candidate lanes evaluate the exact phase detector for and what warp 0 compares its own with.
                float integ = s_hdr[0], ph = s_hdr[1];
                float ang = onehyp_first_angle(s_in[base & (PLL_RING - 1)].x, s_hdr_tad);
                int careful = 0;             // blocks still to run with the angle reduction on the chain
                const unsigned prog_a = smem_u32(&s_prog);
                const unsigned ph_a = smem_u32(&s_ph[0]);
                const unsigned h_a = smem_u32(&s_in[0]) + (unsigned)offsetof(PllIn, h1);
                const bool short_form = onehyp_short_ok(s_hdr_tad, s_hdr[1]);   // trigArg small, phaseEst's grid coarse: the six-operation step

                int prog = base;             // warp 0's progress as last seen: a block old (the load is issued a block ahead, its latency off this warp's path)
                for (int t = 0; t < cnt; t += PLL_PBLK) {
                    const int u0 = base + t;
                    int spin = 0;                // stay within PLL_LEAD1 of warp 0
#ifdef FMRX_PLL_PROFILE
                    const long long pw0 = clock64();
#endif
                    while (prog != PLL_ABANDONED && u0 - prog > PLL_LEAD1 - PLL_PBLK && ++spin < PLL_SPIN_LIMIT)
                        asm volatile("ld.volatile.shared.b32 %0, [%1];" : "=r"(prog) : "r"(prog_a) : "memory");
#ifdef FMRX_PLL_PROFILE
                    const long long pw1 = clock64();
                    if (lane == 0 && blockIdx.x == 0)
                        s_prof1[0] += pw1 - pw0;
#endif
                    if (prog == PLL_ABANDONED || spin >= PLL_SPIN_LIMIT)
                        break;
                    int prog_next;               // (consumed at the top of the next block)
                    asm volatile("ld.volatile.shared.b32 %0, [%1];" : "=r"(prog_next) : "r"(prog_a) : "memory");
                    const unsigned h_a0 = h_a + (unsigned)(u0 & (PLL_RING - 1)) * (unsigned)sizeof(PllIn);
                    const unsigned ph_a0 = ph_a + (unsigned)(u0 & (PLL_PH_RING - 1)) * 8u;
                    // (loading the NEXT block's inputs here, under this block's steps, was tried: 5 % slower -- the 32 more
                    // live registers cost the schedule more than the exposed LDS latency)
                    OneHypIn hs[PLL_PBLK];
#pragma unroll
                    for (int j = 0; j < PLL_PBLK; j++)
                        asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];"
                                     : "=f"(hs[j].P), "=f"(hs[j].r), "=f"(hs[j].B), "=f"(hs[j].c)
                                     : "r"(h_a0 + (unsigned)j * (unsigned)sizeof(PllIn)));
                    // a block of steps without the angle reduction; if an angle left [-pi, pi] (P lost track of phaseEst by
                    // whole turns, or a loop far from lock), the block again with it -- and straight away for the next
                    // blocks, trying the unreduced step again every eighth block.  (Steps past the end of a short last
                    // group are never used.)
                    const float ang0 = ang, integ0 = integ, ph0 = ph;
                    float phs[PLL_PBLK];
                    bool reduce = careful > 0;
                    if (!reduce) {
                        float amax = fabsf(ang);
                        if (short_form) {
                            float crs[PLL_PBLK];
#pragma unroll
                            for (int j = 0; j < PLL_PBLK; j++)
                                crs[j] = p_faddf(hs[j].c, -hs[j].r);
#pragma unroll
                            for (int j = 0; j < PLL_PBLK; j++) {
                                ang = onehyp_predictor_step_short(k, hs[j].P, crs[j], ang, integ, ph);
                                phs[j] = ph;
                                if (j < PLL_PBLK - 1)
                                    amax = fmaxf(amax, fabsf(ang));
                            }
                        } else {
#pragma unroll
                            for (int j = 0; j < PLL_PBLK; j++) {
                                ang = onehyp_predictor_step(k, hs[j], ang, integ, ph);
                                phs[j] = ph;
                                if (j < PLL_PBLK - 1)
                                    amax = fmaxf(amax, fabsf(ang));
                            }
                        }
                        reduce = !(amax <= FMRX_ONEHYP_PI);
                        if (reduce)
                            careful = 8;
                    } else {
                        careful--;
                    }
                    if (reduce) {
                        ang = ang0;
                        integ = integ0;
                        ph = ph0;
                        if (!(fabsf(ang) <= FMRX_ONEHYP_PI))
                            ang = p_faddf(ang, -p_fmulf(6.2831855f, p_faddf(p_faddf(p_fmulf(ang, 0.15915494f), 12582912.0f), -12582912.0f)));
#pragma unroll
                        for (int j = 0; j < PLL_PBLK; j++) {
                            ang = onehyp_predictor_step_reduced(k, hs[j], ang, integ, ph);
                            phs[j] = ph;
                        }
                    }
#pragma unroll
                    for (int j = 0; j < PLL_PBLK; j++)
                        asm volatile("st.volatile.shared.v2.b32 [%0], {%1, %2};" ::"r"(ph_a0 + (unsigned)j * 8u), "r"(__float_as_int(phs[j])),
                                     "r"(u0 + j + 1)
                                     : "memory");
#ifdef FMRX_PLL_PROFILE
                    if (lane == 0 && blockIdx.x == 0) {
                        s_prof1[1] += clock64() - pw1;
                        s_prof1[2] += reduce;
                    }
#endif
                    prog = prog_next;
                }
            }
        } else if (role == 1 && io_id < PLL_IO_WARPS) {
            // ================= I/O =================
            if (!again) {            // (a pass that repeats a group has nothing new to load or store)
                // Sample by sample: the trigArg of the group before (always complete) out of its ring slot, then the
                // inputs of the NEXT group into the same slot (the ring holds two groups).  Prepared with the grid of
                // the group running now: after a binade change only the group that was prepared with the old grid goes
                // without tables.
                const int pb = base - PLL_GROUP, pg = (g - 1) & 1;
                const int kind_g = g > 0 ? s_spec[pg] : 0, split = g > 0 ? s_split[pg] : 0;
                for (int j = lane + 32 * io_id; j < PLL_GROUP; j += 32 * PLL_IO_WARPS) {
                    if (g > 0) {
                        const PllIn &in = s_in[(pb + j) & (PLL_RING - 1)];
                        const int w = s_g[pg][j];
                        const int kind = kind_g == 1 && j >= split ? 0 : kind_g;
                        tr[pb + j] = kind == 1   ? __double2float_rn(p_mul((double)parked_index(w, in, s_kb_blk[pg][j >> 4]), s_ulp_hist[pg]))
                                     : kind == 2 ? __double2float_rn(onehyp_trigarg(in.v, __int_as_float(w)))
                                                 : __int_as_float(w);
                    }
                    prepare_one(base + PLL_GROUP + j, s_hdr[2], s_hdr[1], base);
                    if (j < 32 * PLL_IO_WARPS) {         // the head of the next group is there: say so (see head_ready)
                        __syncwarp();
                        if (lane == 0) {
                            __threadfence_block();
                            asm volatile("st.volatile.shared.b32 [%0], %1;" ::"r"(smem_u32(&s_head_ready[io_id])), "r"(base + PLL_GROUP) : "memory");
                        }
                    }
                }
                if (lane == 0 && io_id == 0)
                    s_prep_ulp[(g + 1) & 1] = s_grid[0];
            }
        }
        __syncthreads();
        if (!s_redo) {
            base += PLL_GROUP;
            g++;
        }
    }
    // the last group's trigArg
    if (warp == 1 && n > 0) {
        const int g = (n - 1) / PLL_GROUP, pb = g * PLL_GROUP, pg = g & 1;
        const int kind_g = s_spec[pg], split = s_split[pg];
        for (int j = lane; pb + j < n && j < PLL_GROUP; j += 32) {
            const PllIn &in = s_in[(pb + j) & (PLL_RING - 1)];
            const int w = s_g[pg][j];
            const int kind = kind_g == 1 && j >= split ? 0 : kind_g;
            tr[pb + j] = kind == 1   ? __double2float_rn(p_mul((double)parked_index(w, in, s_kb_blk[pg][j >> 4]), s_ulp_hist[pg]))
                         : kind == 2 ? __double2float_rn(onehyp_trigarg(in.v, __int_as_float(w)))
                                     : __int_as_float(w);
        }
    }
    if (warp == 0 && lane == 0) {
        if (stale)
            chain_refresh(ch);
        float fi, fq;
        chain_feedback(ch, fi, fq);
        st[0] = ch.integ;
        st[1] = ch.ph;
        st[2] = fi;
        st[3] = fq;
        st[5] = ch.toff;
#ifdef FMRX_PLL_PROFILE
        if (c == 0)
            printf("pll dbg why: blocks near a tie %d, grid point not among the three %d, no valid table %d | candidate lanes: record late %d, no block pi %d, binade edge %d, phi at the seam %d, cross/dot %d, |n1| > 60 %d, ok %d\n",
                   prof_n_tie, prof_n_range, prof_n_inv, s_prof[0], s_prof[1], s_prof[2], s_prof[3], s_prof[4], s_prof[5], s_prof[6]);
        if (c == 0)
            printf("pll dbg: groups %d exact blocks %d (stamp/pi %d, guard %d) redone %d (exact step left the grid %d, too many exact blocks %d) | %.1f cyc/step over %d table steps | kernel %.1f cyc/step; per group: before wait %.0f, wait for tables %.0f, steps %.0f, rest %.0f\n",
                   n_groups, n_exact, prof_n_stamp, prof_n_c, n_redone, prof_n_fe, prof_n_fm, prof_steps ? (double)prof_steps_cyc / prof_steps : 0.0, prof_steps, (double)(clock64() - prof_k0) / n,
                   (double)prof_pre / n_groups, (double)prof_wait / n_groups, (double)prof_steps_cyc / n_groups,
                   (double)(clock64() - prof_k0 - prof_pre - prof_wait - prof_steps_cyc) / n_groups);
        if (c == 0)
            printf("pll dbg group overhead (cycles per group, warp 0): waiting at the end-of-group barrier %.0f, header %.0f (its decisions %.0f), waiting at the header barrier %.0f, after the table steps %.0f\n",
                   (double)prof_bar2 / n_groups, (double)prof_hdr / n_groups, (double)prof_post / n_groups, (double)prof_bar1 / n_groups, (double)prof_post2 / n_groups);
        if (c == 0)
            printf("pll dbg one-hypothesis: groups %d (cut short %d), %.1f cyc/step over %d steps, exact blocks %d | groups without tables %d | predictor: %.1f cyc/step stepping, %.1f waiting for warp 0, %lld blocks of 8 reduced | candidate warp 2: %lld passes, %.0f cyc each, %.0f waiting for records\n",
                   prof_one_groups, prof_one_short, prof_one_steps ? (double)prof_one_cyc / prof_one_steps : 0.0, prof_one_steps, prof_one_exact, prof_checked,
                   prof_one_steps ? (double)s_prof1[1] / prof_one_steps : 0.0, prof_one_steps ? (double)s_prof1[0] / prof_one_steps : 0.0, s_prof1[2],
                   s_prof1[4], s_prof1[4] ? (double)s_prof1[3] / s_prof1[4] : 0.0, s_prof1[4] ? (double)s_prof1[5] / s_prof1[4] : 0.0);
#endif
        st[6] = (float)(n_groups + 1000 * min(n_exact, 999));     // diagnostics of the last launch
        st[7] = s_flag[1] ? -1.0f : (float)n_redone;
        if (n > 0)
            st[4] = nco_from_trig(__double2float_rn(ch.tad), a.prm.scale, a.prm.adjust);   // :173
    }
}

cudaError_t launch_pll(const PllArgs &a_in, int n_captures, cudaStream_t s)
{
    PllArgs a = a_in;
    a.kconst = pllcore::trig_constants();
    // The chain warp's step time is pure issue-to-issue latency, and any other CTA resident
    // on the same SM (the FIR kernels of the neighbouring chunks run concurrently on the
    // other two streams) steals issue slots and shared-memory bandwidth from it: with 301
    // taps that costs the PLL 34 % (profiles/r01_pll_sm_isolation.txt).  While there are SMs
    // to spare, a PLL CTA therefore claims the whole shared memory of its SM, which keeps
    // every other CTA off it.  With more captures than that leaves SMs for, it only asks
    // for the ring it needs and shares.
    DeviceCfg *cfg = device_cfg();
    if (!cfg)
        return cudaErrorInvalidDevice;
    size_t ring_only, whole_sm;
    int sm_count;
    {
        std::lock_guard<std::mutex> lock(g_cfg_mutex);
        if (cfg->pll_ring_only == 0) {
            int dev = 0, optin = 0, sms = 0;
            cudaFuncAttributes fa;
            cudaError_t e = cudaGetDevice(&dev);
            if (e == cudaSuccess)
                e = cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
            if (e == cudaSuccess)
                e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
            if (e == cudaSuccess)
                e = cudaFuncGetAttributes(&fa, k_pll);
            if (e != cudaSuccess)
                return e;
            const size_t need = sizeof(PllIn) * PLL_RING;
            size_t all = (size_t)optin > fa.sharedSizeBytes ? (size_t)optin - fa.sharedSizeBytes : 0;
            if (all < need)
                all = need;
            e = cudaFuncSetAttribute(k_pll, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)all);
            if (e != cudaSuccess)
                return e;
            cfg->pll_whole_sm = all;
            cfg->pll_ring_only = need;
            cfg->sm_count = sms;
        }
        ring_only = cfg->pll_ring_only;
        whole_sm = cfg->pll_whole_sm;
        sm_count = cfg->sm_count;
    }
    const bool isolate = n_captures + kPllSpareSms <= sm_count;
    k_pll<<<n_captures, PLL_THREADS, isolate ? whole_sm : ring_only, s>>>(a);
    return cudaGetLastError();
}

// ============================================================================
// K4: NCO + mixer + mono/stereo polyphase low-pass + delay + combine + pack
// ============================================================================
// One CTA per tile of kAudioTile audio frames of one block of one capture.
// With r = IF index relative to the block start, output n of the block uses
// taps t=0..T-1 at r = floor(n*D/U) - t with coefficient h[(n*D)%U + t*U]
// (src/filter.cpp:85-87).  The reference keeps ONE state vector for the mono
// and the stereo low-pass (src/project.cpp:114,146,172), so for r < 0
//   mono   reads the PREVIOUS block's mixer output (continuous index r), and
//   stereo reads THIS block's demod tail, demod[B + r].
// The 5-frame mono delay (src/project.cpp:153-159) is mono(n-5) on the
// continuous frame index; the 5 frames before a tile are recomputed here.

__global__ void __launch_bounds__(kAudioTile) k_audio(const AudioArgs a, const int span)
{
    extern __shared__ float smem[];
    const int T = a.T, U = a.U, D = a.D, B = a.if_per_block, NA = a.audio_per_block;
    float *s_dem = smem;                     // [span]
    float *s_mix = s_dem + span;             // [span]
    float *s_tail = s_mix + span;            // [T]   demod[B-(T-1) .. B)
    float *s_mono = s_tail + T;              // [kAudioTile + kMonoDelay]
    float *s_cf = s_mono + kAudioTile + kMonoDelay;   // [T] the taps, when every frame has the same phase (U == 1: modes 0, 1)

    const int c = blockIdx.y, tid = threadIdx.x;
    const int tiles_per_block = NA / kAudioTile;
    const int b_local = blockIdx.x / tiles_per_block;
    const int n_lo = (blockIdx.x % tiles_per_block) * kAudioTile;

    const size_t cap = (size_t)c * a.if_stride;
    const long long blk0 = (long long)a.if_off + (long long)b_local * B;   // array index of r = 0
    const float *demod = a.demod + cap;
    const float *chan = a.chan + cap;
    const float *trig = a.trig + cap;

    const int q_first = (n_lo >= kMonoDelay) ? ((n_lo - kMonoDelay) * D) / U
                                             : ((NA - kMonoDelay) * D) / U - B;
    const int r_min = q_first - (T - 1);
    // the last tile of a block also stages the block's final samples (no audio frame of
    // this block uses them, but the stage taps cover the whole block)
    const int r_max = (n_lo + kAudioTile >= NA) ? B - 1 : ((n_lo + kAudioTile - 1) * D) / U;
    // IF samples this tile "owns" for the optional nco/mixer stage taps: those past the
    // previous tile's last staged sample
    const int own_lo = n_lo ? ((n_lo - 1) * D) / U + 1 : 0;
    const int own_hi = r_max + 1;
    const int q_lo = (n_lo * D) / U;          // newest sample of the tile's first frame
    const int count = r_max - r_min + 1;

    for (int i = tid; i < count; i += kAudioTile) {
        const int r = r_min + i;
        const long long g = blk0 + r;
        const float ch = chan[g];
        const float nco = nco_from_trig(trig[g], a.scale, a.adjust);     // src/filter.cpp:170
        const float mx = mix2(ch, nco);                                   // src/filter.cpp:182
        s_dem[i] = demod[g];
        s_mix[i] = mx;
        if (a.nco && r >= own_lo && r < own_hi) {
            const size_t sg = (size_t)c * a.if_stage_stride + a.if_stage_off + (size_t)b_local * B + r;
            a.nco[sg] = nco;
            a.mixer[sg] = mx;
        }
    }
    const bool need_tail = (q_lo - (T - 1)) < 0;
    if (need_tail)
        for (int i = tid; i < T - 1; i += kAudioTile)
            s_tail[i] = demod[blk0 + B - (T - 1) + i];
    if (U == 1)
        for (int i = tid; i < T; i += kAudioTile)
            s_cf[i] = a.coef_pm[i];
    __syncthreads();

    // this thread's frame
    const int n = n_lo + tid;
    float am = 0.0f, as = 0.0f;
    {
        const int nd = n * D;
        const int q = nd / U;
        const float *cf = U == 1 ? s_cf : a.coef_pm + (size_t)(nd % U) * T;
        // taps 0..q reach samples of this block (r >= 0); only the first frames of a block go on into the quirk:
        // mono takes the previous block's MIXER tail, stereo this block's DEMOD tail (src/project.cpp:114,146,172)
        const int t_in = min(T, q + 1);
        const float *xd = s_dem + (q - r_min), *xm = s_mix + (q - r_min);
        for (int t = 0; t < t_in; t++) {
            const float cv = cf[t];
            am = fadd(am, fmul(cv, xd[-t]));
            as = fadd(as, fmul(cv, xm[-t]));
        }
        for (int t = t_in; t < T; t++) {
            const float cv = cf[t];
            am = fadd(am, fmul(cv, xm[-t]));
            as = fadd(as, fmul(cv, s_tail[T - 1 + q - t]));
        }
    }
    s_mono[tid + kMonoDelay] = am;
    if (tid < kMonoDelay) {
        // frames n_lo-5 .. n_lo-1: always plain demod taps (previous block when n_lo == 0)
        int nd, q;
        if (n_lo >= kMonoDelay) {
            nd = (n_lo - kMonoDelay + tid) * D;
            q = nd / U;
        } else {
            nd = (NA - kMonoDelay + tid) * D;
            q = nd / U - B;
        }
        const float *cf = a.coef_pm + (size_t)(nd % U) * T;
        float ae = 0.0f;
        for (int t = 0; t < T; t++)
            ae = fadd(ae, fmul(cf[t], s_dem[q - t - r_min]));
        s_mono[tid] = ae;
    }
    __syncthreads();

    const float ms = s_mono[tid];                              // mono(n - 5)
    const float left = fmul(fadd(ms, as), 0.5f);               // src/filter.cpp:196
    const float right = fmul(fsub(ms, as), 0.5f);              // src/filter.cpp:197
    const size_t frame = (size_t)b_local * NA + n;
    uint32_t *pcm32 = reinterpret_cast<uint32_t *>(a.pcm + (size_t)c * a.pcm_stride);
    pcm32[frame] = pcm_s16(right) | (pcm_s16(left) << 16);     // R first (src/project.cpp:183-191)

    if (a.mono) {
        const size_t sg = (size_t)c * a.au_stage_stride + a.au_stage_off + frame;
        a.mono[sg] = am;
        a.mono_shift[sg] = ms;
        a.stereo[sg] = as;
        a.left[sg] = left;
        a.right[sg] = right;
    }
}

static inline int audio_span(int T, int U, int D)
{
    return (int)(((long long)(kAudioTile + kMonoDelay) * D + U - 1) / U) + T + 2;
}

int audio_smem_bytes(int T, int U, int D)
{
    return (int)sizeof(float) * (2 * audio_span(T, U, D) + 2 * T + kAudioTile + kMonoDelay);
}

cudaError_t launch_audio(const AudioArgs &a, int n_captures, cudaStream_t s)
{
    const int tiles = a.n_blocks * (a.audio_per_block / kAudioTile);
    dim3 grid(tiles, n_captures);
    k_audio<<<grid, kAudioTile, audio_smem_bytes(a.T, a.U, a.D), s>>>(a, audio_span(a.T, a.U, a.D));
    return cudaGetLastError();
}

// ============================================================================
// Operator kernels (one reference operator each; device pointers)
// ============================================================================

__global__ void k_u8_to_f32(const uint8_t *raw, size_t n, float *out)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n)
        out[i] = unpack_u8(raw[i]);
}

cudaError_t launch_u8_to_f32(const uint8_t *raw, size_t n, float *out, cudaStream_t s)
{
    if (n == 0)
        return cudaSuccess;
    k_u8_to_f32<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(raw, n, out);
    return cudaGetLastError();
}

// src/filter.cpp:84-92, one thread per kept output.
__global__ void k_resample(float *out, int n_out, const float *state, int state_len,
                           const float *in, const float *coeff, int taps, int up, int down)
{
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= n_out)
        return;
    const long long nd = (long long)n * down;
    float acc = 0.0f;
    for (int k = (int)(nd % up); k < taps; k += up) {
        const long long j = (nd - k) / up;
        float x;
        if (j >= 0) {
            x = in[j];
        } else {
            const long long sj = state_len + j;
            x = (sj >= 0) ? state[sj] : 0.0f;
        }
        acc = fadd(acc, fmul(coeff[k], x));
    }
    out[n] = acc;
}

cudaError_t launch_resample(float *out, int n_out, const float *state, int state_len,
                            const float *in, int n_in, const float *coeff, int taps,
                            int up, int down, cudaStream_t s)
{
    (void)n_in;
    if (n_out == 0)
        return cudaSuccess;
    k_resample<<<(n_out + 127) / 128, 128, 0, s>>>(out, n_out, state, state_len, in, coeff, taps,
                                                   up, down);
    return cudaGetLastError();
}

__global__ void k_fmdemod(float *out, const float *i_ds, const float *q_ds, int n, float prev_i,
                          float prev_q)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n)
        return;
    const float pi_ = k ? i_ds[k - 1] : prev_i;
    const float pq_ = k ? q_ds[k - 1] : prev_q;
    out[k] = fm_discriminate(i_ds[k], q_ds[k], pi_, pq_);
}

cudaError_t launch_fmdemod(float *out, const float *i_ds, const float *q_ds, int n, float prev_i,
                           float prev_q, cudaStream_t s)
{
    if (n == 0)
        return cudaSuccess;
    k_fmdemod<<<(n + 255) / 256, 256, 0, s>>>(out, i_ds, q_ds, n, prev_i, prev_q);
    return cudaGetLastError();
}

__global__ void k_nco(float *out, const float *trig, size_t n, float scale, float adjust)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n)
        out[i] = nco_from_trig(trig[i], scale, adjust);
}

cudaError_t launch_nco(float *out, const float *trig, size_t n, float scale, float adjust,
                       cudaStream_t s)
{
    if (n == 0)
        return cudaSuccess;
    k_nco<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(out, trig, n, scale, adjust);
    return cudaGetLastError();
}

__global__ void k_mixer(float *out, const float *x, const float *y, size_t n)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n)
        out[i] = mix2(x[i], y[i]);
}

cudaError_t launch_mixer(float *out, const float *x, const float *y, size_t n, cudaStream_t s)
{
    if (n == 0)
        return cudaSuccess;
    k_mixer<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(out, x, y, n);
    return cudaGetLastError();
}

__global__ void k_lr_extract(float *left, float *right, const float *mono, const float *stereo,
                             size_t n)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        const float m = mono[i], s = stereo[i];
        left[i] = fmul(fadd(m, s), 0.5f);
        right[i] = fmul(fsub(m, s), 0.5f);
    }
}

cudaError_t launch_lr_extract(float *left, float *right, const float *mono, const float *stereo,
                              size_t n, cudaStream_t s)
{
    if (n == 0)
        return cudaSuccess;
    k_lr_extract<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(left, right, mono, stereo, n);
    return cudaGetLastError();
}

__global__ void k_pcm_pack(int16_t *pcm, const float *left, const float *right, size_t n)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        pcm[2 * i] = (int16_t)pcm_s16(right[i]);
        pcm[2 * i + 1] = (int16_t)pcm_s16(left[i]);
    }
}

cudaError_t launch_pcm_pack(int16_t *pcm, const float *left, const float *right, size_t n,
                            cudaStream_t s)
{
    if (n == 0)
        return cudaSuccess;
    k_pcm_pack<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(pcm, left, right, n);
    return cudaGetLastError();
}

// ---- the reference's RDS sketch (src/project.cpp:200-271): the two element-wise steps between the operators ----

// :249-251 channel_squared[i] = channel_data[i] * channel_data[i]
__global__ void k_square(float *out, const float *x, size_t n)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n)
        out[i] = fmul(x[i], x[i]);
}

cudaError_t launch_square(float *out, const float *x, size_t n, cudaStream_t s)
{
    if (n == 0)
        return cudaSuccess;
    k_square<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(out, x, n);
    return cudaGetLastError();
}

// :170 (the PLL's ncoOut from its trigArg), :259-263 (the channel delayed by `delay` samples, the first ones from the
// carried state) and :269 / filter.cpp:182 (mixer): out[i] = 2 * (nco[i] * channel_shift[i])
__global__ void k_rds_mix(float *out, const float *trig, const float *chan, const float *shift_state, int delay, size_t n,
                          float scale, float adjust)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        const float nco = nco_from_trig(trig[i], scale, adjust);
        const float c = i >= (size_t)delay ? chan[i - delay] : shift_state[i];
        out[i] = mix2(nco, c);
    }
}

cudaError_t launch_rds_mix(float *out, const float *trig, const float *chan, const float *shift_state, int delay, size_t n,
                           float scale, float adjust, cudaStream_t s)
{
    if (n == 0)
        return cudaSuccess;
    k_rds_mix<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(out, trig, chan, shift_state, delay, n, scale, adjust);
    return cudaGetLastError();
}

// ---- spectrum tap: the reference's estimatePSD (src/fourier.cpp:35-117) ---------------------------------------
// Hann-windowed segments of freq_bins samples, the DFT of each (:14-22), power (4/(Fs N)) |X|^2 in dB, mean over the
// segments.  The reference accumulates its DFT in complex<float> with libm's cosf/sinf; here the window and the
// windowed samples are the reference's floats and everything behind them is double (twiddles from a shared table,
// index (j m) mod N kept incrementally), so the result is the same estimate to the reference's own float accuracy --
// a diagnostic, compared with a tolerance, not a parity-critical path.  One CTA per frequency bin; its threads take
// the segments round robin.
__global__ void __launch_bounds__(128) k_psd(float *psd, const float *samples, int n_seg, int N, float Fs)
{
    extern __shared__ __align__(16) double2 s_tw[];      // [N] e^{-2 pi i r / N}
    float *s_hann = reinterpret_cast<float *>(s_tw + N); // [N]
    __shared__ double s_red[128];
    const int m = blockIdx.x, tid = threadIdx.x;
    for (int r = tid; r < N; r += blockDim.x) {
        double sn, cs;
        sincospi(-2.0 * (double)r / (double)N, &sn, &cs);
        s_tw[r] = make_double2(cs, sn);
        const double h = sin((double)r * 3.14159265358979323846 / (double)N);       // :55
        s_hann[r] = (float)(h * h);
    }
    __syncthreads();
    double acc = 0.0;
    for (int sgm = tid; sgm < n_seg; sgm += blockDim.x) {
        const float *x = samples + (size_t)sgm * N;
        double re = 0.0, im = 0.0;
        int r = 0;
        for (int j = 0; j < N; j++) {
            const double w = (double)fmul(x[j], s_hann[j]);                          // :79 (float product)
            const double2 t = s_tw[r];
            re = __fma_rn(w, t.x, re);
            im = __fma_rn(w, t.y, im);
            r += m;
            r -= r >= N ? N : 0;
        }
        const double p = (4.0 / ((double)Fs * (double)N)) * (re * re + im * im);    // :94
        acc += 10.0 * log10(p);                                                      // :97
    }
    s_red[tid] = acc;
    __syncthreads();
    for (int st = 64; st > 0; st >>= 1) {
        if (tid < st)
            s_red[tid] += s_red[tid + st];
        __syncthreads();
    }
    if (tid == 0)
        psd[m] = (float)(s_red[0] / (double)n_seg);                                  // :110
}

cudaError_t launch_psd(float *psd, const float *samples, int n_seg, int freq_bins, float Fs, cudaStream_t s)
{
    if (freq_bins < 2 || n_seg < 1)
        return cudaSuccess;
    const size_t smem = (size_t)freq_bins * (sizeof(double2) + sizeof(float));
    k_psd<<<freq_bins / 2, 128, smem, s>>>(psd, samples, n_seg, freq_bins, Fs);
    return cudaGetLastError();
}

}  // namespace fmrx
