// fmrx_scan.cu -- band scan: Welch's averaged periodogram of the complex u8 IQ stream (include/fmrx.h, fmrx_scan_*).
//
// k_scan_welch<LOG2N>: CTA r of a launch takes the run of segments [r*R, r*R + R) of the launch (R = scan_run_segments:
// a function of N only, so that the same segments always form the same runs whatever the chunking of the host path).
// It reads the run's pairs from HBM once: the first segment's N pairs, then N/2 new pairs per segment, the overlapping
// half staying in shared memory.  Per segment: bytes -> (b-128)/128 (exact), times the float window, into shared memory
// in bit-reversed order; log2(N) radix-2 DIT stages with float twiddles; |X|^2 in double, added in segment order to
// per-thread registers (thread t owns the FFT bins t + i*T).  The CTA writes its run's sums to partial[r][N], in
// fft-shifted order.  k_scan_reduce then adds partial[0], partial[1], ... in that order to the handle's accumulator:
// no atomics, so the same bytes and the same calls give the same bits.
#include <cstdint>
#include <cuda_runtime.h>

#include "fmrx_internal.h"

namespace fmrx {
namespace {

template <int LOG2N> struct ScanShape {
    static constexpr int N = 1 << LOG2N;
    static constexpr int H = N / 2;
    // threads per CTA: 8 bins per thread up to N = 8192, 16 at N = 16384 (1024 threads)
    static constexpr int T = N / 8 < 128 ? 128 : (N / 8 > 1024 ? 1024 : N / 8);
    static constexpr int BPT = N / T;
};

template <int LOG2N>
__global__ void __launch_bounds__(ScanShape<LOG2N>::T)
k_scan_welch(const uint8_t *__restrict__ iq, int n_seg, int run, const float *__restrict__ win,
             const float2 *__restrict__ tw, double *__restrict__ partial)
{
    using S = ScanShape<LOG2N>;
    constexpr int N = S::N, H = S::H, T = S::T, BPT = S::BPT;
    extern __shared__ __align__(16) unsigned char smem[];
    float2 *buf = reinterpret_cast<float2 *>(smem);                  // N complex
    uchar2 *raw = reinterpret_cast<uchar2 *>(smem + N * sizeof(float2));   // N pairs: half q of the stream at slot q&1
    const int tid = threadIdx.x;
    const int j0 = blockIdx.x * run;
    const int j1 = min(n_seg, j0 + run);

    double acc[BPT];
#pragma unroll
    for (int i = 0; i < BPT; i++)
        acc[i] = 0.0;

    for (int j = j0; j < j1; j++) {
        // the halves j and j+1 of the stream (H pairs each) form segment j; load what is not yet resident
        for (int q = (j == j0 ? j : j + 1); q <= j + 1; q++) {
            const uint8_t *p = iq + static_cast<size_t>(q) * H * 2;
            uchar2 *dst = raw + (q & 1) * H;
            for (int k = tid; k < H; k += T)
                dst[k] = make_uchar2(p[2 * k], p[2 * k + 1]);
        }
        __syncthreads();
        for (int k = tid; k < N; k += T) {
            const uchar2 b = raw[((j + (k >= H)) & 1) * H + (k & (H - 1))];
            const float w = __ldg(win + k);
            const float xi = (static_cast<float>(b.x) - 128.0f) / 128.0f;
            const float xq = (static_cast<float>(b.y) - 128.0f) / 128.0f;
            buf[__brev(static_cast<unsigned>(k)) >> (32 - LOG2N)] = make_float2(xi * w, xq * w);
        }
        __syncthreads();
        // radix-2 decimation in time: at half-span s, butterfly b joins i = 2s*(b/s) + b%s and i+s with tw[(b%s)*N/(2s)]
#pragma unroll 1
        for (int ls = 0; ls < LOG2N; ls++) {
            const int s = 1 << ls;
            for (int b = tid; b < H; b += T) {
                const int pos = b & (s - 1);
                const int i = ((b >> ls) << (ls + 1)) + pos;
                const float2 w = __ldg(tw + (pos << (LOG2N - 1 - ls)));
                const float2 u = buf[i], v = buf[i + s];
                const float tr = v.x * w.x - v.y * w.y;
                const float ti = v.x * w.y + v.y * w.x;
                buf[i] = make_float2(u.x + tr, u.y + ti);
                buf[i + s] = make_float2(u.x - tr, u.y - ti);
            }
            __syncthreads();
        }
#pragma unroll
        for (int i = 0; i < BPT; i++) {
            const float2 x = buf[tid + i * T];
            const double re = x.x, im = x.y;
            acc[i] += re * re + im * im;
        }
        // (the next segment's first write to buf follows a __syncthreads, after every thread has read its bins)
    }
    double *out = partial + static_cast<size_t>(blockIdx.x) * N;
#pragma unroll
    for (int i = 0; i < BPT; i++)
        out[(tid + i * T + H) & (N - 1)] = acc[i];                   // fft-shifted: DC at N/2
}

__global__ void k_scan_reduce(double *__restrict__ acc, const double *__restrict__ partial, int n_runs, int n)
{
    const int m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= n)
        return;
    double a = acc[m];
    for (int r = 0; r < n_runs; r++)
        a += partial[static_cast<size_t>(r) * n + m];
    acc[m] = a;
}

template <int LOG2N>
cudaError_t launch_welch(const uint8_t *iq, int n_seg, const float *win, const float2 *tw, double *partial,
                         cudaStream_t s)
{
    using S = ScanShape<LOG2N>;
    const int smem = S::N * (sizeof(float2) + sizeof(uchar2));
    if (smem > 48 * 1024) {
        const cudaError_t e = cudaFuncSetAttribute(k_scan_welch<LOG2N>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess)
            return e;
    }
    const int run = scan_run_segments(S::N);
    const int grid = (n_seg + run - 1) / run;
    k_scan_welch<LOG2N><<<grid, S::T, smem, s>>>(iq, n_seg, run, win, tw, partial);
    return cudaGetLastError();
}

}  // namespace

int scan_run_segments(int n_fft)
{
    // 2^16 pairs of new input per run (8 segments at N = 16384, 512 at N = 256): enough work to amortise the first
    // segment's extra half, and about 2200 runs (CTAs) for a 60 s capture at 2.4 Msps
    const int r = (1 << 17) / n_fft;
    return r < 1 ? 1 : r;
}

cudaError_t launch_scan(const uint8_t *iq, int n_seg, int n_fft, const float *win, const float2 *tw, double *partial,
                        double *acc, cudaStream_t s)
{
    if (n_seg <= 0)
        return cudaSuccess;
    cudaError_t e;
    switch (n_fft) {
    case 256: e = launch_welch<8>(iq, n_seg, win, tw, partial, s); break;
    case 512: e = launch_welch<9>(iq, n_seg, win, tw, partial, s); break;
    case 1024: e = launch_welch<10>(iq, n_seg, win, tw, partial, s); break;
    case 2048: e = launch_welch<11>(iq, n_seg, win, tw, partial, s); break;
    case 4096: e = launch_welch<12>(iq, n_seg, win, tw, partial, s); break;
    case 8192: e = launch_welch<13>(iq, n_seg, win, tw, partial, s); break;
    case 16384: e = launch_welch<14>(iq, n_seg, win, tw, partial, s); break;
    default: return cudaErrorInvalidValue;
    }
    if (e != cudaSuccess)
        return e;
    const int run = scan_run_segments(n_fft);
    const int n_runs = (n_seg + run - 1) / run;
    k_scan_reduce<<<(n_fft + 255) / 256, 256, 0, s>>>(acc, partial, n_runs, n_fft);
    return cudaGetLastError();
}

}  // namespace fmrx
