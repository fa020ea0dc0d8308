// fmrx_rds_dec.cu -- the RDS decoder of the fused pipeline (fmrx_set_rds; definition in include/fmrx.h and
// DESIGN.md 7.5, float64 oracle in tests/rds_oracle.py).  Two kernels per chunk, enqueued on the front stream after
// K2, so that K3 never waits for them:
//   k_rds_baseband : demod -> 57 kHz mix (exact phase table) -> decimating low-pass FIR -> biphase matched filter y[m],
//                    for the kept outputs only.  Feed-forward: one CTA per tile of y, independent of every other.
//   k_rds_bits     : one warp per capture at the bit rate: window sums c_w, timing, sampling, differential decision,
//                    block sync, groups into the capture's ring.
// Not bit-exact with anything (the oracle is float64), so contraction is allowed here; same bytes and the same
// split give the same bits (no atomics, fixed summation orders).
#include <cstdint>

#include "fmrx.h"
#include "fmrx_internal.h"

namespace fmrx {

namespace {

constexpr int kTileY = 128;     // y outputs per CTA of k_rds_baseband
constexpr int kBaseThreads = 128;

__constant__ uint16_t c_rds_h[26] = { 0x200, 0x100, 0x080, 0x040, 0x020, 0x010, 0x008, 0x004, 0x002,
                                      0x001, 0x2DC, 0x16E, 0x0B7, 0x287, 0x39F, 0x313, 0x355, 0x376,
                                      0x1BB, 0x201, 0x3DC, 0x1EE, 0x0F7, 0x2A7, 0x38F, 0x31B };
// syndromes of the offset words A, B, C, D, C' (IEC 62106 Annex B)
__constant__ uint16_t c_rds_syn[5] = { 0x3D8, 0x3D4, 0x25C, 0x258, 0x3CC };

__device__ __forceinline__ long long floor_div(long long a, long long b)
{
    const long long q = a / b;
    return (a % b != 0 && ((a < 0) != (b < 0))) ? q - 1 : q;
}
__device__ __forceinline__ long long ceil_div(long long a, long long b) { return -floor_div(-a, b); }

__device__ __forceinline__ float demod_at(const RdsBasebandArgs &a, int c, long long k)
{
    // k: sample index relative to the chunk's first; the decoder keeps its own tail of the last dtail_len samples
    return k >= 0 ? a.demod[static_cast<size_t>(c) * a.if_stride + a.if_off + k]
                  : a.dtail[static_cast<size_t>(c) * a.dtail_len + a.dtail_len + k];
}

__global__ void __launch_bounds__(kBaseThreads) k_rds_baseband(RdsBasebandArgs a)
{
    extern __shared__ float2 sm[];
    const RdsParams &P = a.prm;
    const int ci = blockIdx.y;
    const int c = a.caps[ci];
    const long long n0 = a.if_run + a.state[c].n_offset;          // the capture's n of the chunk's first sample
    const long long m_lo = ceil_div(n0, P.D), m_hi = ceil_div(n0 + a.n_if, P.D);
    const long long m0 = m_lo + static_cast<long long>(blockIdx.x) * kTileY;
    if (m0 >= m_hi)
        return;
    const int ny = static_cast<int>(m_hi - m0 < kTileY ? m_hi - m0 : kTileY);
    const int nu = ny + 2 * P.L - 1;                                 // u[m0-2L+1 .. m0+ny-1]
    const long long u0 = m0 - 2 * P.L + 1;
    const long long nz0 = u0 * P.D - (P.taps - 1);                   // first IF sample read
    const int nz = (nu - 1) * P.D + P.taps;
    float2 *z = sm;                    // [nz]
    float2 *u = sm + nz;               // [nu]
    for (int i = threadIdx.x; i < nz; i += blockDim.x) {
        const long long n = nz0 + i;
        const float d = demod_at(a, c, n - n0);
        const int k = static_cast<int>((static_cast<long long>(P.q) * (((n % P.P) + P.P) % P.P)) % P.P);
        const float2 e = a.mix[k];
        z[i] = make_float2(d * e.x, d * e.y);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < nu; i += blockDim.x) {
        const float2 *zp = z + i * P.D + P.taps - 1;
        float re = 0.f, im = 0.f;
        for (int t = 0; t < P.taps; t++) {
            const float h = a.taps[t];
            re = fmaf(h, zp[-t].x, re);
            im = fmaf(h, zp[-t].y, im);
        }
        u[i] = make_float2(re, im);
    }
    __syncthreads();
    float2 *y = a.ybuf + static_cast<size_t>(c) * a.ybuf_len + a.ytail_len + (m0 - m_lo);
    for (int r = threadIdx.x; r < ny; r += blockDim.x) {
        const float2 *up = u + r + 2 * P.L - 1;
        float pr = 0.f, pi = 0.f, nr = 0.f, ni = 0.f;
        for (int i = 0; i < P.L; i++) {
            pr += up[-i].x;
            pi += up[-i].y;
        }
        for (int i = P.L; i < 2 * P.L; i++) {
            nr += up[-i].x;
            ni += up[-i].y;
        }
        y[r] = make_float2(pr - nr, pi - ni);
    }
}

// ---- bit rate ------------------------------------------------------------------------------------------------------

__device__ double tau_at(const RdsDecState &s, double t, long long W, int M)
{
    const long long a = static_cast<long long>(floor((t - 0.5 * M) / M));
    if (a < s.w_first)
        return s.tau[s.w_first & 3];
    if (a >= W - 1)
        return s.tau[(W - 1) & 3];
    const double f = (t - (static_cast<double>(a) * M + 0.5 * M)) / M;
    const double ta = s.tau[a & 3], tb = s.tau[(a + 1) & 3];
    return ta + (tb - ta) * f;
}

__device__ int syndrome(uint32_t word)
{
    int s = 0;
    for (int i = 0; i < 26; i++)
        if ((word >> (25 - i)) & 1u)
            s ^= c_rds_h[i];
    return s;
}

__device__ void emit_group(RdsDecState &s, fmrx_rds_group *ring)
{
    if (!s.cur.valid)
        return;
    ring[s.written % kRdsRing] = s.cur;
    s.written++;
}

__device__ void start_group(RdsDecState &s, long long first_bit)
{
    first_bit = first_bit < 1 ? 1 : first_bit;   // a group that began before the decoder's first bit takes its instant
    s.cur.if_index = static_cast<uint64_t>(s.t_ring[first_bit & (kRdsBitRing - 1)]);
    for (int b = 0; b < 4; b++)
        s.cur.block[b] = 0;
    s.cur.valid = 0;
    s.cur.c_prime = 0;
    s.cur.reserved = 0;
}

// one decided bit through block synchronisation and group assembly (tests/rds_oracle.py: BlockSync.push)
__device__ void push_bit(RdsDecState &s, int bit, long long if_index, fmrx_rds_group *ring)
{
    s.reg = (s.reg << 1) | static_cast<unsigned long long>(bit);
    s.nbits++;
    s.t_ring[s.nbits & (kRdsBitRing - 1)] = if_index;
    const uint32_t word = static_cast<uint32_t>(s.reg & 0x3FFFFFFull);
    const int syn = syndrome(word);
    if (!s.synced) {
        if (s.nbits < 26)
            return;
        for (int x = 0; x < 5; x++) {
            if (syn != c_rds_syn[x])
                continue;
            const int p = x == 4 ? 2 : x;                 // C' stands where C does
            if (s.last_hit[(p + 3) & 3] == s.nbits - 26) {
                s.synced = 1;
                s.pos = p;
                s.in_block = 0;
                s.bad = 0;
                start_group(s, s.nbits - 26 * p - 25);
                if (p > 0) {
                    const uint32_t prev = static_cast<uint32_t>((s.reg >> 26) & 0x3FFFFFFull);
                    s.cur.block[p - 1] = static_cast<uint16_t>(prev >> 10);
                    s.cur.valid |= static_cast<uint8_t>(1u << (p - 1));
                    if (p - 1 == 2 && syndrome(prev) == c_rds_syn[4])
                        s.cur.c_prime = 1;
                }
                s.cur.block[p] = static_cast<uint16_t>(word >> 10);
                s.cur.valid |= static_cast<uint8_t>(1u << p);
                if (x == 4)
                    s.cur.c_prime = 1;
                if (p == 3)
                    emit_group(s, ring);
            } else {
                s.last_hit[p] = s.nbits;
            }
            break;
        }
        return;
    }
    if (++s.in_block < 26)
        return;
    s.in_block = 0;
    s.pos = (s.pos + 1) & 3;
    const int p = s.pos;
    if (p == 0)
        start_group(s, s.nbits - 25);
    bool ok = syn == c_rds_syn[p];
    if (p == 2 && syn == c_rds_syn[4]) {
        ok = true;
        s.cur.c_prime = 1;
    }
    s.cur.block[p] = static_cast<uint16_t>(word >> 10);
    if (ok) {
        s.cur.valid |= static_cast<uint8_t>(1u << p);
        s.bad = 0;
    } else {
        s.bad++;
    }
    if (p == 3)
        emit_group(s, ring);
    if (s.bad >= 8) {
        s.synced = 0;
        for (int k = 0; k < 4; k++)
            s.last_hit[k] = kRdsNoHit;
    }
}

__global__ void __launch_bounds__(32) k_rds_bits(RdsBitsArgs a)
{
    __shared__ RdsDecState s;
    const RdsParams &P = a.prm;
    const int c = a.caps[blockIdx.x];
    const int lane = threadIdx.x;
    RdsDecState *gs = a.state + c;
    {
        const int *src = reinterpret_cast<const int *>(gs);
        int *dst = reinterpret_cast<int *>(&s);
        for (int i = lane; i < static_cast<int>(sizeof(RdsDecState) / 4); i += 32)
            dst[i] = src[i];
    }
    __syncwarp();
    const long long n0 = a.if_run + s.n_offset;
    const long long m_lo = ceil_div(n0, P.D), m_hi = ceil_div(n0 + a.n_if, P.D);
    const long long m_base = m_lo - a.ytail_len;                      // the m of ybuf[c][0]
    float2 *y = a.ybuf + static_cast<size_t>(c) * a.ybuf_len;
    fmrx_rds_group *ring = a.ring + static_cast<size_t>(c) * kRdsRing;
    const int M = P.M;
    const double sps = static_cast<double>(P.fs2) / 1187.5;
    const long long W_end = floor_div(m_hi, M);                       // windows complete after this chunk
    for (long long w = s.w_next; w < W_end; w++) {
        // c_w = sum |y[m]|^2 e^{-2 pi i m 1187.5/fs2}: lane l takes m = wM + l + 32k in ascending k, then a fixed tree
        double re = 0.0, im = 0.0;
        for (int k = lane; k < M; k += 32) {
            const long long m = w * M + k;
            const float2 v = y[m - m_base];
            const double p = static_cast<double>(v.x) * v.x + static_cast<double>(v.y) * v.y;
            const double2 e = a.bitphase[static_cast<int>((m % P.Q) * P.q2 % P.Q)];
            re += p * e.x;
            im += p * e.y;
        }
        for (int o = 16; o > 0; o >>= 1) {
            re += __shfl_xor_sync(0xffffffffu, re, o);
            im += __shfl_xor_sync(0xffffffffu, im, o);
        }
        if (lane == 0) {
            const double raw = -atan2(im, re) / (2.0 * 3.14159265358979323846);
            if (w == s.w_first) {
                s.tau[w & 3] = raw;
            } else {
                const double prev = s.tau[(w - 1) & 3];
                double d = raw - prev;
                d -= ceil(d - 0.5);
                s.tau[w & 3] = prev + d;
            }
            const long long W = w + 1;
            for (;;) {
                const double t0 = s.have_prev ? s.t_prev + sps : static_cast<double>(s.j) * sps;
                const double t1 = (static_cast<double>(s.j) + tau_at(s, t0, W, M)) * sps;
                const double t = (static_cast<double>(s.j) + tau_at(s, t1, W, M)) * sps;
                if (t >= static_cast<double>(W - 1) * M)
                    break;
                const long long i = static_cast<long long>(floor(t));
                const double f = t - static_cast<double>(i);
                float2 y0 = make_float2(0.f, 0.f), y1 = y0;
                if (i >= 0 && i >= m_base)
                    y0 = y[i - m_base];
                if (i + 1 >= 0 && i + 1 >= m_base)
                    y1 = y[i + 1 - m_base];
                const double sr = y0.x * (1.0 - f) + y1.x * f, si = y0.y * (1.0 - f) + y1.y * f;
                if (s.have_prev) {
                    const double r = sr * s.s_prev.x + si * s.s_prev.y;     // Re(s_j conj(s_{j-1}))
                    push_bit(s, r < 0.0 ? 1 : 0, static_cast<long long>(floor(t * P.D + 0.5)), ring);
                }
                s.s_prev = make_double2(sr, si);
                s.t_prev = t;
                s.have_prev = 1;
                s.j++;
            }
        }
        __syncwarp();
    }
    if (lane == 0)
        s.w_next = s.w_next > W_end ? s.w_next : W_end;
    __syncwarp();
    // the last ytail_len samples move to the front for the next chunk (forward copy: reads stay ahead of writes)
    const long long n_new = m_hi - m_lo;
    for (int i0 = 0; i0 < a.ytail_len; i0 += 32) {
        const int i = i0 + lane;
        float2 v = make_float2(0.f, 0.f);
        if (i < a.ytail_len)
            v = y[i + n_new];
        __syncwarp();
        if (i < a.ytail_len)
            y[i] = v;
        __syncwarp();
    }
    {
        const int *src = reinterpret_cast<const int *>(&s);
        int *dst = reinterpret_cast<int *>(gs);
        for (int i = lane; i < static_cast<int>(sizeof(RdsDecState) / 4); i += 32)
            dst[i] = src[i];
    }
}

}  // namespace

int rds_baseband_smem(const RdsParams &P)
{
    const int nu = kTileY + 2 * P.L - 1;
    return static_cast<int>(((nu - 1) * P.D + P.taps + nu) * sizeof(float2));
}

cudaError_t launch_rds(const RdsBasebandArgs &b, const RdsBitsArgs &r, int n_caps, cudaStream_t s)
{
    const long long max_y = (static_cast<long long>(b.n_if) + b.prm.D - 1) / b.prm.D + 1;
    const dim3 grid(static_cast<unsigned>((max_y + kTileY - 1) / kTileY), static_cast<unsigned>(n_caps));
    k_rds_baseband<<<grid, kBaseThreads, rds_baseband_smem(b.prm), s>>>(b);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess)
        return e;
    k_rds_bits<<<n_caps, 32, 0, s>>>(r);
    return cudaGetLastError();
}

}  // namespace fmrx
