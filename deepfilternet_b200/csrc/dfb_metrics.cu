// dfb_metrics.cu -- batched speech-quality metrics of (clean, degraded) pairs on the device (sm_100a): STOI, SI-SDR,
// segmental SNR, LLR and WSS with the semantics of the reference's evaluation code:
//   STOI   df/stoi.py:163-231 (resample to 10 kHz, remove_silent_frames :35-110, 512-point STFT, 15 third-octave bands,
//          30-frame segments, normalise, clip, correlate)
//   SI-SDR df/evaluation_utils.py:599-619 si_sdr_speechmetrics
//   SSNR   df/sepm.py:28-51 SNRseg; LLR :200-277 lpcoeff + llr; WSS :280-487 findLocPeaks + wss (all at 16 kHz)
// Utterance b of a padded batch is scored on its first len[b] samples exactly as if it were scored alone.
//
// Kernels (grid y / x = utterance; every per-utterance quantity comes from the host-computed Utt geometry):
//   k_resample (dfb_dsp.cu)  ragged rows to 10 kHz (STOI) and 16 kHz (sepm family)
//   k_sisdr          one block per utterance: fp64 sums x.x, x.y, y.y -> SI-SDR
//   k_stoi_energy    one warp per 256-sample frame: frame energy in dB (silent-frame detection)
//   k_stoi_select    one block per utterance: frames within 40 dB of the loudest, compacted in order (kept-frame list)
//   k_stoi_bands     one warp per STFT frame of the overlap-added kept frames: 512-point real FFT (runtime mixed-radix
//                    FFT of dfb_fft.cuh), 15 third-octave band magnitudes of both signals
//   k_stoi_corr      one block per utterance: the 30-frame segment correlations, mean
//   k_sepm_frames    one warp per 30 ms frame: segmental SNR (fp64), LPC autocorrelation + Levinson (fp64) and the LLR
//                    quadratic forms, 1024-point real FFT -> 25 critical-band log energies (fp64) -> WSS frame distortion
//   k_sepm_reduce    one block per utterance: mean (SSNR) and the mean of the 95 % smallest frames (LLR, WSS) by a
//                    radix select of the order statistic
#include <algorithm>
#include <cmath>
#include <cstring>
#include <vector>

#include "dfb_common.cuh"
#include "dfb_fft.cuh"

namespace dfb {
namespace {

constexpr double kDblEps = 2.220446049250313e-16;   // np.finfo(np.float64).eps
constexpr float kFltEps = 1.1920928955078125e-07f;  // np.finfo(np.float32).eps

// STOI (df/stoi.py:177-184)
constexpr int kStoiFs = 10000, kStoiFrame = 256, kStoiHop = 128, kStoiM = 256 /* 512-point real FFT */, kStoiBands = 15,
              kStoiSeg = 30;
constexpr int kStoiWarps = 8;
// sepm family at 16 kHz (sepm.py: frameLen 0.03, overlap 0.75, n_fft = 2^ceil(log2(2 winlength)), P = 16 above 10 kHz)
constexpr int kSepmFs = 16000, kSepmWin = 480, kSepmHop = 120, kSepmM = 512 /* 1024-point real FFT */, kCrit = 25, kLpc = 16;
constexpr int kSepmWarps = 4;
constexpr int kMaxCf = 512;   // non-zero critical-band filter taps (357 for the 25 bands at 16 kHz)

// per-utterance geometry, computed on the host from the lengths
struct Utt {
    int64_t len;      // samples at the input rate
    int64_t l10;      // at 10 kHz: ceil(len * 10000 / sr)
    int64_t l16;      // at 16 kHz
    int pad_front;    // remove_silent_frames: pad = 256 - l10 % 256 split front / end (stoi.py:59-61)
    int pad_end;
    int nw;           // 256 / 128 frames of the padded 10 kHz signal
    int nf;           // 30 ms frames scored by SNRseg / llr / wss: floor(l16 / 120) - 4, 0 below 600 samples
};
// result of the silent-frame removal of one utterance
struct StoiInfo {
    int K;     // kept frames
    int n;     // samples of the overlap-added signal after the end trims
    int trim;  // samples trimmed at the front
    int J;     // STFT frames (0: fewer than 512 samples, STOI is NaN)
};
struct StoiBands { int lo[kStoiBands], hi[kStoiBands]; };   // thirdoct (stoi.py:113-141): bins [lo, hi) of band m
struct CritTable { int lo[kCrit], cnt[kCrit], off[kCrit]; double v[kMaxCf]; };   // non-zero taps of sepm's crit_filter

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_sumf(float v) {
#pragma unroll
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
// block-wide sum (blockDim.x a multiple of 32, <= 1024); every thread gets the result
__device__ double block_sum(double v, double *s_red) {
    v = warp_sum(v);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    __syncthreads();
    if (lane == 0) s_red[warp] = v;
    __syncthreads();
    v = lane < nw ? s_red[lane] : 0.0;
    return warp_sum(v);
}

// twiddles of the M-point complex transform (e^{-2 pi i k / M}) and of the real split (e^{-2 pi i k / 2M}, k <= M/2)
__device__ void make_twiddles(float2 *tw, float2 *tws, int M) {
    for (int k = threadIdx.x; k < M; k += blockDim.x) {
        double s, c;
        sincospi(2.0 * k / M, &s, &c);
        tw[k] = make_float2((float)c, (float)-s);
    }
    for (int k = threadIdx.x; k <= M / 2; k += blockDim.x) {
        double s, c;
        sincospi((double)k / M, &s, &c);
        tws[k] = make_float2((float)c, (float)-s);
    }
}

// |X[k]|^2 of the 2M-point real signal packed into a[n] = (x[2n], x[2n+1]) for k in [0, M] (k = M into P[M] only when
// nyquist), by the warp; b is scratch, the power lands in whichever buffer the FFT did not end in (returned)
__device__ __forceinline__ float *warp_power(float2 *a, float2 *b, const float2 *tw, const float2 *tws, int M, int lane,
                                             bool nyquist) {
    const float2 *Z = warp_fft_any<false>(a, b, tw, M, lane);
    float *P = reinterpret_cast<float *>(Z == a ? b : a);
    for (int k = lane; k <= M / 2; k += 32) {
        float2 xk, xnk;
        rfft_split(Z[k], Z[(M - k) % M], tws[k], xk, xnk);
        const float pk = xk.x * xk.x + xk.y * xk.y, pnk = xnk.x * xnk.x + xnk.y * xnk.y;
        P[k] = pk;
        if (2 * k != M && (k > 0 || nyquist)) P[M - k] = pnk;
    }
    __syncwarp();
    return P;
}

// ------------------------------------------------------------------------------------------------ SI-SDR ----
// si_sdr_speechmetrics on float32 inputs (eps = float32 eps): a = (eps + x.y) / (x.x + eps), Sss = a^2 x.x,
// Snn = |y - a x|^2 = y.y - 2 a x.y + a^2 x.x, 10 log10((eps + Sss) / (eps + Snn)); sums in fp64.  grid B, block 512.
__global__ void __launch_bounds__(512) k_sisdr(const float *__restrict__ x, const float *__restrict__ y, int64_t T,
                                               const Utt *__restrict__ utt, float *__restrict__ out, int ncol, int col) {
    __shared__ double s_red[32];
    const int b = blockIdx.x;
    const int64_t L = utt[b].len;
    const float *xb = x + (int64_t)b * T, *yb = y + (int64_t)b * T;
    double sxx = 0, sxy = 0, syy = 0;
    for (int64_t i = threadIdx.x; i < L; i += blockDim.x) {
        const double u = __ldg(xb + i), v = __ldg(yb + i);
        sxx = fma(u, u, sxx);
        sxy = fma(u, v, sxy);
        syy = fma(v, v, syy);
    }
    sxx = block_sum(sxx, s_red);
    sxy = block_sum(sxy, s_red);
    syy = block_sum(syy, s_red);
    if (threadIdx.x == 0) {
        const double eps = kFltEps;
        const double a = (eps + sxy) / (sxx + eps);
        const double sss = a * a * sxx, snn = fmax(syy - 2.0 * a * sxy + a * a * sxx, 0.0);
        out[(int64_t)b * ncol + col] = (float)(10.0 * log10((eps + sss) / (eps + snn)));
    }
}

// -------------------------------------------------------------------------------------------------- STOI ----
// w[i] = torch.hann_window(258, periodic=False)[1 + i] (stoi.py:69-70, :147)
__device__ __forceinline__ float stoi_win(int i) { return (float)(0.5 - 0.5 * cospi(2.0 * (i + 1) / 257.0)); }

// sample p of the padded 10 kHz signal (remove_silent_frames zero-pads pad_front / pad_end samples)
__device__ __forceinline__ float stoi_padded(const float *row, int64_t l10, int pad_front, int64_t p) {
    const int64_t i = p - pad_front;
    return (i >= 0 && i < l10) ? __ldg(row + i) : 0.f;
}

// frame energies 20 log10(|w x_i| / sqrt(256) + eps) (stoi.py:75); grid (ceil(nw_max / kStoiWarps), B)
__global__ void __launch_bounds__(32 * kStoiWarps) k_stoi_energy(const float *__restrict__ x10, int64_t T10,
                                                               const Utt *__restrict__ utt, float *__restrict__ energy,
                                                               int nw_max) {
    const int b = blockIdx.y, lane = threadIdx.x & 31, i = blockIdx.x * kStoiWarps + (threadIdx.x >> 5);
    const Utt u = utt[b];
    if (i >= u.nw) return;
    const float *row = x10 + (int64_t)b * T10;
    float e = 0.f;
    for (int t = lane; t < kStoiFrame; t += 32) {
        const float v = stoi_win(t) * stoi_padded(row, u.l10, u.pad_front, (int64_t)i * kStoiHop + t);
        e = fmaf(v, v, e);
    }
    e = warp_sumf(e);
    if (lane == 0) energy[(int64_t)b * nw_max + i] = 20.f * log10f(sqrtf(e) / 16.f + (float)kDblEps);
}

// frames with energy above max - 40 dB, in order (stoi.py:78-82), and the length bookkeeping of the overlap-add and the
// end trims (:84-108).  grid B, block 256.
__global__ void __launch_bounds__(256) k_stoi_select(const float *__restrict__ energy, int nw_max, const Utt *__restrict__ utt,
                                                     int *__restrict__ kidx, StoiInfo *__restrict__ info) {
    __shared__ float s_max[8];
    __shared__ int s_cnt[8];
    __shared__ int s_base;
    const int b = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const Utt u = utt[b];
    const float *e = energy + (int64_t)b * nw_max;
    float mx = -INFINITY;
    for (int i = threadIdx.x; i < u.nw; i += blockDim.x) mx = fmaxf(mx, e[i]);
#pragma unroll
    for (int o = 16; o; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if (lane == 0) s_max[warp] = mx;
    if (threadIdx.x == 0) s_base = 0;
    __syncthreads();
    mx = s_max[0];
    for (int w = 1; w < 8; w++) mx = fmaxf(mx, s_max[w]);
    const float thr = mx - 40.f;
    int *kb = kidx + (int64_t)b * nw_max;
    for (int i0 = 0; i0 < u.nw; i0 += blockDim.x) {
        const int i = i0 + threadIdx.x;
        const bool keep = i < u.nw && thr - e[i] < 0.f;
        const unsigned bal = __ballot_sync(0xffffffffu, keep);
        if (lane == 0) s_cnt[warp] = __popc(bal);
        __syncthreads();
        int base = s_base;
        for (int w = 0; w < warp; w++) base += s_cnt[w];
        if (keep) kb[base + __popc(bal & ((1u << lane) - 1))] = i;
        __syncthreads();
        if (threadIdx.x == 0) for (int w = 0; w < 8; w++) s_base += s_cnt[w];
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const int K = s_base;
        const bool first = thr - e[0] < 0.f, last = thr - e[u.nw - 1] < 0.f;
        StoiInfo r;
        r.K = K;
        r.trim = first ? u.pad_front : 0;
        r.n = (K - 1) * kStoiHop + kStoiFrame - r.trim - (last ? u.pad_end : 0);
        r.J = r.n >= 2 * kStoiM ? 1 + (r.n - kStoiFrame) / kStoiHop : 0;
        info[b] = r;
    }
}

// One warp per STFT frame j of the silence-free signal (stoi.py:_stft, 256-sample hann frames, hop 128, 512-point FFT,
// normalised by the window sum): band magnitudes sqrt(sum_{k in band} |X_k|^2) of both signals -> xb / yb
// [B][nw_max][16].  Sample q of the silence-free signal is the overlap-add of the kept frames divided by the overlap-add
// of the window (stoi.py:84-100).  grid (ceil(nw_max / kStoiWarps), B), dynamic smem 2 M float2 per warp.
__global__ void __launch_bounds__(32 * kStoiWarps) k_stoi_bands(const float *__restrict__ x10, const float *__restrict__ y10,
                                                              int64_t T10, const Utt *__restrict__ utt,
                                                              const StoiInfo *__restrict__ info, const int *__restrict__ kidx,
                                                              int nw_max, StoiBands bands, float *__restrict__ xb,
                                                              float *__restrict__ yb) {
    extern __shared__ __align__(16) float2 s_buf[];
    __shared__ float2 s_tw[kStoiM], s_tws[kStoiM / 2 + 1];
    __shared__ float s_win[kStoiFrame];
    __shared__ StoiBands s_bands;
    if (threadIdx.x == 0) s_bands = bands;
    make_twiddles(s_tw, s_tws, kStoiM);
    for (int i = threadIdx.x; i < kStoiFrame; i += blockDim.x) s_win[i] = stoi_win(i);
    __syncthreads();
    const int b = blockIdx.y, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int j = blockIdx.x * kStoiWarps + warp;
    const StoiInfo inf = info[b];
    if (j >= inf.J) return;
    const Utt u = utt[b];
    const int *kb = kidx + (int64_t)b * nw_max;
    float2 *A = s_buf + (size_t)warp * 2 * kStoiM, *Bf = A + kStoiM;
    constexpr float kInvWsum2 = 1.f / (128.5f * 128.5f);   // the window sums to 128.5
    for (int s = 0; s < 2; s++) {
        const float *row = (s ? y10 : x10) + (int64_t)b * T10;
        auto sample = [&](int t) -> float {   // windowed sample t of STFT frame j
            const int64_t q = (int64_t)j * kStoiHop + t + inf.trim;
            const int c = (int)(q / kStoiHop), o = (int)(q - (int64_t)c * kStoiHop);
            float num = 0.f, den = 0.f;
            if (c < inf.K) {
                const float w = s_win[o];
                num += w * stoi_padded(row, u.l10, u.pad_front, (int64_t)kb[c] * kStoiHop + o);
                den += w;
            }
            if (c >= 1) {
                const float w = s_win[o + kStoiHop];
                num += w * stoi_padded(row, u.l10, u.pad_front, (int64_t)kb[c - 1] * kStoiHop + o + kStoiHop);
                den += w;
            }
            return s_win[t] * (num / den);
        };
        for (int n = lane; n < kStoiM; n += 32)
            A[n] = n < kStoiFrame / 2 ? make_float2(sample(2 * n), sample(2 * n + 1)) : make_float2(0.f, 0.f);
        __syncwarp();
        const float *P = warp_power(A, Bf, s_tw, s_tws, kStoiM, lane, true);
        float *dst = (s ? yb : xb) + ((int64_t)b * nw_max + j) * 16;
        if (lane < kStoiBands) {
            float acc = 0.f;
            for (int k = s_bands.lo[lane]; k < s_bands.hi[lane]; k++) acc += P[k] * kInvWsum2;
            dst[lane] = sqrtf(acc);
        }
        __syncwarp();
    }
}

// Segment correlations (stoi.py:208-230): per segment s and band m the L = min(J, 30) frames starting at s (one segment
// of all J frames when J <= 30); out = sum of correlations / (15 * segments).  grid B, block 256.
__global__ void __launch_bounds__(256) k_stoi_corr(const StoiInfo *__restrict__ info, const float *__restrict__ xb,
                                                   const float *__restrict__ yb, int nw_max, float *__restrict__ out,
                                                   int ncol, int col) {
    __shared__ double s_red[32];
    const int b = blockIdx.x;
    const int J = info[b].J;
    if (J == 0) {
        if (threadIdx.x == 0) out[(int64_t)b * ncol + col] = NAN;
        return;
    }
    const int nseg = J > kStoiSeg ? J - kStoiSeg + 1 : 1, L = J > kStoiSeg ? kStoiSeg : J;
    const float clip = (float)(1.0 + 5.623413251903491), eps = (float)kDblEps;   // 1 + 10^(-beta / 20), beta = -15
    const float invL = 1.f / (float)L;
    double acc = 0.0;
    for (int it = threadIdx.x; it < nseg * kStoiBands; it += blockDim.x) {
        const int s = it / kStoiBands, m = it - s * kStoiBands;
        const float *xp = xb + ((int64_t)b * nw_max + s) * 16 + m, *yp = yb + ((int64_t)b * nw_max + s) * 16 + m;
        float xv[kStoiSeg], yv[kStoiSeg];
        float nx = 0.f, ny = 0.f;
#pragma unroll
        for (int i = 0; i < kStoiSeg; i++) {
            xv[i] = i < L ? xp[i * 16] : 0.f;
            yv[i] = i < L ? yp[i * 16] : 0.f;
            nx = fmaf(xv[i], xv[i], nx);
            ny = fmaf(yv[i], yv[i], ny);
        }
        const float g = sqrtf(nx) / (sqrtf(ny) + eps);
        float mx = 0.f, my = 0.f;
#pragma unroll
        for (int i = 0; i < kStoiSeg; i++) {
            yv[i] = fminf(yv[i] * g, xv[i] * clip);
            mx += xv[i];
            my += yv[i];
        }
        mx *= invL;
        my *= invL;
        float sx = 0.f, sy = 0.f;
#pragma unroll
        for (int i = 0; i < kStoiSeg; i++) {
            xv[i] = i < L ? xv[i] - mx : 0.f;
            yv[i] = i < L ? yv[i] - my : 0.f;
            sx = fmaf(xv[i], xv[i], sx);
            sy = fmaf(yv[i], yv[i], sy);
        }
        const float ix = 1.f / (sqrtf(sx) + eps), iy = 1.f / (sqrtf(sy) + eps);
        float c = 0.f;
#pragma unroll
        for (int i = 0; i < kStoiSeg; i++) c = fmaf(xv[i] * ix, yv[i] * iy, c);
        acc += c;
    }
    acc = block_sum(acc, s_red);
    if (threadIdx.x == 0) out[(int64_t)b * ncol + col] = (float)(acc / (double)(kStoiBands * nseg));
}

// ------------------------------------------------------------------------------------------ sepm family ----
// sepm's window: 0.5 (1 - cos(2 pi n / 481)), n = 1 .. 480
__device__ __forceinline__ double sepm_win(int i) { return 0.5 * (1.0 - cospi(2.0 * (i + 1) / (kSepmWin + 1.0))); }

// sepm.lpcoeff (sepm.py:200-243) from the autocorrelation R[0..16] (fp64 Levinson-Durbin, by one thread): lp[0..16] =
// the float32 lpparams [1, -a]; a / ap are 16-entry work arrays (shared memory, so that nothing is indexed in registers)
__device__ void levinson(const double *R, double *lp, double *a, double *ap) {
    double E = R[0];
    for (int i = 0; i < kLpc; i++) a[i] = 1.0;
    for (int i = 0; i < kLpc; i++) {
        double sum = 0.0;
        for (int j = 0; j < i; j++) sum += a[j] * R[i - j];
        const double rc = (R[i + 1] - sum) / fmax(E, kDblEps);
        for (int j = 0; j < i; j++) ap[j] = a[j];
        a[i] = rc;
        for (int j = 0; j < i; j++) a[j] = ap[j] - rc * ap[i - 1 - j];
        E = (1.0 - rc * rc) * E;
    }
    lp[0] = 1.0;
    for (int i = 0; i < kLpc; i++) lp[i + 1] = (double)(float)(-a[i]);
}

// One warp per 30 ms frame i < nf (hop 120): seg[b][i] (SNRseg, sepm.py:45-47, before the clamp of the mean),
// llr[b][i] (log of the LPC residual ratio, :257-270), wss[b][i] (weighted spectral slope distance, :433-481).
// grid (ceil(nf_max / kSepmWarps), B); dynamic smem: per warp 2 x 480 double (windowed frames) + 2 x 512 float2 (FFT).
struct SepmWarpSmem {
    double wx[kSepmWin], wy[kSepmWin];
    float2 fa[kSepmM], fb[kSepmM];
    double R[2][kLpc + 1], A[2][kLpc + 1], work[2][2][kLpc];
    double logE[2][kCrit];
};

__global__ void __launch_bounds__(32 * kSepmWarps) k_sepm_frames(const float *__restrict__ x16, const float *__restrict__ y16,
                                                               int64_t T16, const Utt *__restrict__ utt, CritTable ct,
                                                               unsigned which, int nf_max, double *__restrict__ seg,
                                                               double *__restrict__ llr, double *__restrict__ wss) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ float2 s_tw[kSepmM], s_tws[kSepmM / 2 + 1];
    __shared__ double s_win[kSepmWin];
    __shared__ CritTable s_ct;
    make_twiddles(s_tw, s_tws, kSepmM);
    for (int i = threadIdx.x; i < kSepmWin; i += blockDim.x) s_win[i] = sepm_win(i);
    if (which & DFB_METRIC_WSS) {
        const int *src = reinterpret_cast<const int *>(&ct);
        int *dst = reinterpret_cast<int *>(&s_ct);
        for (int i = threadIdx.x; i < (int)(sizeof(CritTable) / sizeof(int)); i += blockDim.x) dst[i] = src[i];
    }
    __syncthreads();
    const int b = blockIdx.y, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int i = blockIdx.x * kSepmWarps + warp;
    if (i >= utt[b].nf) return;
    SepmWarpSmem &w = reinterpret_cast<SepmWarpSmem *>(smem_raw)[warp];
    const float *xr = x16 + (int64_t)b * T16 + (int64_t)i * kSepmHop, *yr = y16 + (int64_t)b * T16 + (int64_t)i * kSepmHop;
    for (int n = lane; n < kSepmWin; n += 32) {
        w.wx[n] = s_win[n] * (double)__ldg(xr + n);
        w.wy[n] = s_win[n] * (double)__ldg(yr + n);
    }
    __syncwarp();
    const int64_t o = (int64_t)b * nf_max + i;
    if (which & DFB_METRIC_SSNR) {
        double sig = 0.0, noise = 0.0;
        for (int n = lane; n < kSepmWin; n += 32) {
            const double d = w.wx[n] - w.wy[n];
            sig = fma(w.wx[n], w.wx[n], sig);
            noise = fma(d, d, noise);
        }
        sig = warp_sum(sig);
        noise = warp_sum(noise);
        const double snr = 10.0 * log10(sig / (noise + kDblEps) + kDblEps);
        if (lane == 0) seg[o] = snr < -10.0 ? -10.0 : snr > 35.0 ? 35.0 : snr;   // NaN stays NaN, as the masked clamp
    }
    if (which & DFB_METRIC_LLR) {
        for (int k = 0; k <= kLpc; k++) {
            double rx = 0.0, ry = 0.0;
            for (int n = lane; n < kSepmWin - k; n += 32) {
                rx = fma(w.wx[n], w.wx[n + k], rx);
                ry = fma(w.wy[n], w.wy[n + k], ry);
            }
            rx = warp_sum(rx);
            ry = warp_sum(ry);
            if (lane == 0) {
                w.R[0][k] = rx;
                w.R[1][k] = ry;
            }
        }
        __syncwarp();
        if (lane < 2) levinson(w.R[lane], w.A[lane], w.work[lane][0], w.work[lane][1]);
        __syncwarp();
        // numerator A_p' T(R_c) A_p and denominator A_c' T(R_c) A_c with the float32 acorr / lpparams of lpcoeff; row
        // `lane` of the Toeplitz products
        double tn = 0.0, td = 0.0;
        if (lane <= kLpc) {
            double rp = 0.0, rc = 0.0;
            for (int j = 0; j <= kLpc; j++) {
                const double r = (double)(float)w.R[0][lane > j ? lane - j : j - lane];
                rp = fma(r, w.A[1][j], rp);
                rc = fma(r, w.A[0][j], rc);
            }
            tn = w.A[1][lane] * rp;
            td = w.A[0][lane] * rc;
        }
        tn = warp_sum(tn);
        td = warp_sum(td);
        if (lane == 0) {
            double frac = tn / (td + kDblEps);
            if (!(frac > 0.0) && frac == frac) frac = 1000.0;   // frac <= 0 -> 1000 (NaN stays NaN)
            llr[o] = log(frac);
        }
    }
    if (which & DFB_METRIC_WSS) {
        for (int s = 0; s < 2; s++) {
            const float *r = s ? yr : xr;
            for (int n = lane; n < kSepmM; n += 32) {
                float2 v = make_float2(0.f, 0.f);
                if (n < kSepmWin / 2) {
                    v.x = (float)(s_win[2 * n] * ((double)__ldg(r + 2 * n) + kDblEps));
                    v.y = (float)(s_win[2 * n + 1] * ((double)__ldg(r + 2 * n + 1) + kDblEps));
                }
                w.fa[n] = v;
            }
            __syncwarp();
            const float *P = warp_power(w.fa, w.fb, s_tw, s_tws, kSepmM, lane, false);
            if (lane < kCrit) {
                double e = 0.0;
                const double *cv = s_ct.v + s_ct.off[lane];
                for (int k = 0; k < s_ct.cnt[lane]; k++) e = fma(cv[k], (double)P[s_ct.lo[lane] + k], e);
                const double le = 10.0 * log10(e);
                w.logE[s][lane] = le < -100.0 ? -100.0 : le;
            }
            __syncwarp();
        }
        double num = 0.0, den = 0.0;
        if (lane < kCrit - 1) {
            double wgt[2], slope[2];
#pragma unroll
            for (int s = 0; s < 2; s++) {
                const double *L = w.logE[s];
                double mx = L[0];
                for (int m = 1; m < kCrit; m++) mx = fmax(mx, L[m]);
                // findLocPeaks (sepm.py:280-295) on the slopes L[m + 1] - L[m]
                auto sl = [&](int m) { return L[m + 1] - L[m]; };
                int n = lane;
                double peak;
                if (sl(lane) > 0) {
                    while (n < kCrit - 1 && sl(n) > 0) n++;
                    peak = L[n - 1];
                } else {
                    while (n >= 0 && sl(n) <= 0) n--;
                    peak = L[n + 1];
                }
                slope[s] = sl(lane);
                wgt[s] = 20.0 / (20.0 + mx - L[lane]) * (1.0 / (1.0 + peak - L[lane]));
            }
            const double W = (wgt[0] + wgt[1]) / 2.0, d = slope[0] - slope[1];
            num = W * (d * d);
            den = W;
        }
        num = warp_sum(num);
        den = warp_sum(den);
        if (lane == 0) wss[o] = num / den;
    }
}

// order-preserving key of a double (NaN after +inf, as np.sort)
__device__ __forceinline__ unsigned long long dkey(double v) {
    unsigned long long u = v == v ? (unsigned long long)__double_as_longlong(v) : 0x7ff8000000000000ull;
    return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}
__device__ __forceinline__ double dkey_inv(unsigned long long k) {
    return __longlong_as_double((long long)((k >> 63) ? (k & 0x7fffffffffffffffull) : ~k));
}

// mean of the k smallest of v[0..n) (sepm.py: sort, keep the first round(0.95 n), mean): the k-th smallest key by an
// 8-pass radix select, then (sum of the values below it + the ties it needs) / k.  Called by the whole block.
__device__ double trimmed_mean(const double *v, int n, int k, unsigned *s_hist, double *s_red, int *s_sel) {
    unsigned long long prefix = 0, mask = 0;
    int kk = k;
    for (int shift = 56; shift >= 0; shift -= 8) {
        for (int d = threadIdx.x; d < 256; d += blockDim.x) s_hist[d] = 0;
        __syncthreads();
        for (int i = threadIdx.x; i < n; i += blockDim.x) {
            const unsigned long long u = dkey(v[i]);
            if ((u & mask) == prefix) atomicAdd(&s_hist[(u >> shift) & 255], 1u);
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            int cum = 0, d = 0;
            for (; d < 255 && cum + (int)s_hist[d] < kk; d++) cum += s_hist[d];
            s_sel[0] = d;
            s_sel[1] = kk - cum;
        }
        __syncthreads();
        prefix |= (unsigned long long)s_sel[0] << shift;
        mask |= 255ull << shift;
        kk = s_sel[1];
        __syncthreads();
    }
    double sum = 0.0, cnt = 0.0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        if (dkey(v[i]) < prefix) {
            sum += v[i];
            cnt += 1.0;
        }
    }
    sum = block_sum(sum, s_red);
    cnt = block_sum(cnt, s_red);
    return (sum + ((double)k - cnt) * dkey_inv(prefix)) / (double)k;
}

// per utterance: mean of the frame SNRs (SNRseg), trimmed means of the LLR / WSS frame values.  grid B, block 256.
__global__ void __launch_bounds__(256) k_sepm_reduce(const Utt *__restrict__ utt, const double *__restrict__ seg,
                                                     const double *__restrict__ llr, const double *__restrict__ wss, int nf_max,
                                                     unsigned which, float *__restrict__ out, int ncol, int c_ssnr, int c_llr,
                                                     int c_wss) {
    __shared__ double s_red[32];
    __shared__ unsigned s_hist[256];
    __shared__ int s_sel[2];
    const int b = blockIdx.x, nf = utt[b].nf;
    float *o = out + (int64_t)b * ncol;
    if (nf == 0) {
        if (threadIdx.x == 0) {
            if (which & DFB_METRIC_SSNR) o[c_ssnr] = NAN;
            if (which & DFB_METRIC_LLR) o[c_llr] = NAN;
            if (which & DFB_METRIC_WSS) o[c_wss] = NAN;
        }
        return;
    }
    const int64_t base = (int64_t)b * nf_max;
    if (which & DFB_METRIC_SSNR) {
        double s = 0.0;
        for (int i = threadIdx.x; i < nf; i += blockDim.x) s += seg[base + i];
        s = block_sum(s, s_red);
        if (threadIdx.x == 0) o[c_ssnr] = (float)(s / nf);
    }
    const int k = (int)rint((double)nf * 0.95);   // int(round(len * alpha)): round half to even, like Python
    if (which & DFB_METRIC_LLR) {
        const double m = k > 0 ? trimmed_mean(llr + base, nf, k, s_hist, s_red, s_sel) : NAN;
        if (threadIdx.x == 0) o[c_llr] = (float)m;
    }
    if (which & DFB_METRIC_WSS) {
        const double m = k > 0 ? trimmed_mean(wss + base, nf, k, s_hist, s_red, s_sel) : NAN;
        if (threadIdx.x == 0) o[c_wss] = (float)m;
    }
}

// -------------------------------------------------------------------------------------------------- host ----
bool supported_rate(int sr) {
    switch (sr) {
        case 8000: case 16000: case 22050: case 24000: case 32000: case 44100: case 48000: return true;
        default: return false;
    }
}

// torchaudio's _get_sinc_resample_kernel for sinc_interp_hann, lowpass_filter_width 16, rolloff 0.99 (df.io.resample
// "sinc_fast"; the same taps as deepfilternet_b200/io.py resample_kernel)
struct ResampleTaps {
    int og = 1, nw = 1, width = 0;
    std::vector<float> k;
};
ResampleTaps resample_taps(int orig, int target) {
    ResampleTaps r;
    int a = orig, b = target;
    while (b) { const int t = a % b; a = b; b = t; }
    r.og = orig / a;
    r.nw = target / a;
    const double lpw = 16.0, base = (r.og < r.nw ? r.og : r.nw) * 0.99;
    r.width = (int)std::ceil(lpw * r.og / base);
    const int K = 2 * r.width + r.og;
    r.k.resize((size_t)r.nw * K);
    const double kPiD = 3.14159265358979323846, scale = base / r.og;
    for (int j = 0; j < r.nw; j++) {
        const float tj = (float)(-j) / (float)r.nw;   // torchaudio divides the integer arange in float32
        for (int i = 0; i < K; i++) {
            double t = (double)tj + (double)(i - r.width) / r.og;
            t *= base;
            t = t < -lpw ? -lpw : t > lpw ? lpw : t;
            const double c = std::cos(t * kPiD / lpw / 2);
            const double window = c * c;
            t *= kPiD;
            const double v = t == 0 ? 1.0 : std::sin(t) / t;
            r.k[(size_t)j * K + i] = (float)(v * (window * scale));
        }
    }
    return r;
}

StoiBands stoi_bands() {   // thirdoct(10000, 512, 15, 150): argmin of the squared distance to each edge
    StoiBands sb;
    const int nb = kStoiM + 1;
    auto nearest = [&](double f) {
        int best = 0;
        double bd = INFINITY;
        for (int i = 0; i < nb; i++) {
            const double fi = (double)i * kStoiFs / (2 * kStoiM), d = (fi - f) * (fi - f);
            if (d < bd) { bd = d; best = i; }
        }
        return best;
    };
    for (int m = 0; m < kStoiBands; m++) {
        sb.lo[m] = nearest(150.0 * std::pow(2.0, (2.0 * m - 1) / 6));
        sb.hi[m] = nearest(150.0 * std::pow(2.0, (2.0 * m + 1) / 6));
    }
    return sb;
}

int crit_table(CritTable &ct) {   // sepm.py:389-405 at fs = 16000, n_fft = 1024
    static const double cent[kCrit] = {50.0, 120.0, 190.0, 260.0, 330.0, 400.0, 470.0, 540.0, 617.372, 703.378, 798.717,
                                       904.128, 1020.38, 1148.30, 1288.72, 1442.54, 1610.70, 1794.16, 1993.93, 2211.08,
                                       2446.71, 2701.97, 2978.04, 3276.17, 3597.63};
    static const double bwd[kCrit] = {70.0, 70.0, 70.0, 70.0, 70.0, 70.0, 70.0, 77.3724, 86.0056, 95.3398, 105.411,
                                      116.256, 127.914, 140.423, 153.823, 168.154, 183.457, 199.776, 217.153, 235.631,
                                      255.255, 276.072, 298.126, 321.465, 346.136};
    const double min_factor = std::exp(-30.0 / (2.0 * 2.303)), maxf = kSepmFs / 2.0;
    int off = 0;
    for (int m = 0; m < kCrit; m++) {
        const double f0 = std::floor(cent[m] / maxf * kSepmM), bw = bwd[m] / maxf * kSepmM;
        const double norm = std::log(bwd[0]) - std::log(bwd[m]);
        ct.lo[m] = -1;
        ct.cnt[m] = 0;
        ct.off[m] = off;
        for (int j = 0; j < kSepmM; j++) {
            const double q = (j - f0) / bw, v = std::exp(-11 * (q * q) + norm);
            if (!(v > min_factor)) continue;
            if (ct.lo[m] < 0) ct.lo[m] = j;
            if (j != ct.lo[m] + ct.cnt[m] || off >= kMaxCf) return fail(DFB_ERR_UNSUPPORTED, "critical-band table layout");
            ct.v[off++] = v;
            ct.cnt[m]++;
        }
    }
    return DFB_OK;
}

// stream-ordered device scratch, released on the stream when the call returns
struct AsyncScratch {
    cudaStream_t s;
    std::vector<void *> ptrs;
    explicit AsyncScratch(cudaStream_t st) : s(st) {}
    ~AsyncScratch() { for (void *p : ptrs) cudaFreeAsync(p, s); }
    template <typename T>
    T *alloc(size_t n) {
        void *p = nullptr;
        if (cudaMallocAsync(&p, (n ? n : 1) * sizeof(T), s) != cudaSuccess) return nullptr;
        ptrs.push_back(p);
        return (T *)p;
    }
};

int check_metrics_args(const void *clean, const void *deg, const int64_t *lengths, int64_t B, int64_t T, int sr,
                       unsigned which, const void *out) {
    if (!clean || !deg || !out) return fail(DFB_ERR_INVALID, "null argument");
    if (B <= 0 || T <= 0) return fail(DFB_ERR_INVALID, "empty batch: B = %lld, T = %lld", (long long)B, (long long)T);
    if (B > 65535) return fail(DFB_ERR_INVALID, "more than 65535 utterances per call");
    if (which == 0 || (which & ~31u)) return fail(DFB_ERR_INVALID, "metric mask %u: bits 1 (STOI) .. 16 (WSS) only", which);
    if (!supported_rate(sr))
        return fail(DFB_ERR_INVALID, "unsupported sample rate %d (8000, 16000, 22050, 24000, 32000, 44100, 48000)", sr);
    if (lengths)
        for (int64_t b = 0; b < B; b++)
            if (lengths[b] <= 0 || lengths[b] > T)
                return fail(DFB_ERR_INVALID, "lengths[%lld] = %lld outside [1, T = %lld]", (long long)b,
                            (long long)lengths[b], (long long)T);
    return DFB_OK;
}

}  // namespace
}  // namespace dfb

using namespace dfb;

extern "C" int dfb_metrics(int device, const float *d_clean, const float *d_deg, const int64_t *lengths, int64_t B, int64_t T,
                           int sr, unsigned which, float *d_out, void *stream) {
    int rc = check_metrics_args(d_clean, d_deg, lengths, B, T, sr, which, d_out);
    if (rc) return rc;
    rc = use_device(device);
    if (rc) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    int col[5], ncol = 0;
    for (int m = 0; m < 5; m++) col[m] = (which >> m) & 1 ? ncol++ : -1;
    const bool stoi = which & DFB_METRIC_STOI, sepm = which & (DFB_METRIC_SSNR | DFB_METRIC_LLR | DFB_METRIC_WSS);

    // per-utterance geometry
    ResampleTaps t10 = stoi && sr != kStoiFs ? resample_taps(sr, kStoiFs) : ResampleTaps{};
    ResampleTaps t16 = sepm && sr != kSepmFs ? resample_taps(sr, kSepmFs) : ResampleTaps{};
    auto out_len = [](const ResampleTaps &t, int64_t n) { return (t.nw * n + t.og - 1) / t.og; };
    std::vector<Utt> utt((size_t)B);
    std::vector<int64_t> lens((size_t)B);
    int nw_max = 1, nf_max = 1;
    for (int64_t b = 0; b < B; b++) {
        Utt &u = utt[(size_t)b];
        u.len = lens[(size_t)b] = lengths ? lengths[b] : T;
        u.l10 = out_len(t10, u.len);
        u.l16 = out_len(t16, u.len);
        const int pad = kStoiFrame - (int)(u.l10 % kStoiFrame);
        u.pad_front = pad / 2;
        u.pad_end = pad - pad / 2;
        u.nw = (int)((u.l10 + pad) / kStoiHop - 1);
        u.nf = u.l16 >= 5 * kSepmHop ? (int)(u.l16 / kSepmHop - 4) : 0;
        nw_max = std::max(nw_max, u.nw);
        nf_max = std::max(nf_max, u.nf);
    }
    AsyncScratch ws(s);
    Utt *d_utt = ws.alloc<Utt>((size_t)B);
    int64_t *d_len = ws.alloc<int64_t>((size_t)B);
    if (!d_utt || !d_len) return fail(DFB_ERR_OOM, "cudaMallocAsync failed");
    DFB_CUDA(cudaMemcpyAsync(d_utt, utt.data(), sizeof(Utt) * B, cudaMemcpyHostToDevice, s));
    DFB_CUDA(cudaMemcpyAsync(d_len, lens.data(), sizeof(int64_t) * B, cudaMemcpyHostToDevice, s));

    // resample the ragged rows (rows keep stride T_out of the longest)
    auto resampled = [&](const ResampleTaps &t, const float *d_in, float **d_res, int64_t *T_res) -> int {
        if (t.k.empty()) {
            *d_res = const_cast<float *>(d_in);
            *T_res = T;
            return DFB_OK;
        }
        *T_res = out_len(t, T);
        float *d_k = ws.alloc<float>(t.k.size());
        *d_res = ws.alloc<float>((size_t)(B * *T_res));
        if (!d_k || !*d_res) return fail(DFB_ERR_OOM, "cudaMallocAsync failed");
        DFB_CUDA(cudaMemcpyAsync(d_k, t.k.data(), sizeof(float) * t.k.size(), cudaMemcpyHostToDevice, s));
        return launch_resample(d_in, B, T, d_len, d_k, t.og, t.nw, t.width, *d_res, *T_res, s);
    };

    if (which & DFB_METRIC_SISDR) {
        k_sisdr<<<(unsigned)B, 512, 0, s>>>(d_clean, d_deg, T, d_utt, d_out, ncol, col[1]);
        DFB_LAUNCH_CHECK();
    }
    if (stoi) {
        float *x10, *y10;
        int64_t T10;
        if ((rc = resampled(t10, d_clean, &x10, &T10)) || (rc = resampled(t10, d_deg, &y10, &T10))) return rc;
        float *d_e = ws.alloc<float>((size_t)B * nw_max), *d_xb = ws.alloc<float>((size_t)B * nw_max * 16),
              *d_yb = ws.alloc<float>((size_t)B * nw_max * 16);
        int *d_kidx = ws.alloc<int>((size_t)B * nw_max);
        StoiInfo *d_info = ws.alloc<StoiInfo>((size_t)B);
        if (!d_e || !d_xb || !d_yb || !d_kidx || !d_info) return fail(DFB_ERR_OOM, "cudaMallocAsync failed");
        const dim3 grid((unsigned)((nw_max + kStoiWarps - 1) / kStoiWarps), (unsigned)B);
        {
            k_stoi_energy<<<grid, 32 * kStoiWarps, 0, s>>>(x10, T10, d_utt, d_e, nw_max);
            DFB_LAUNCH_CHECK();
        }
        {
            k_stoi_select<<<(unsigned)B, 256, 0, s>>>(d_e, nw_max, d_utt, d_kidx, d_info);
            DFB_LAUNCH_CHECK();
        }
        {
            const size_t smem = sizeof(float2) * 2 * kStoiM * kStoiWarps;
            k_stoi_bands<<<grid, 32 * kStoiWarps, smem, s>>>(x10, y10, T10, d_utt, d_info, d_kidx, nw_max, stoi_bands(),
                                                              d_xb, d_yb);
            DFB_LAUNCH_CHECK();
        }
        {
            k_stoi_corr<<<(unsigned)B, 256, 0, s>>>(d_info, d_xb, d_yb, nw_max, d_out, ncol, col[0]);
            DFB_LAUNCH_CHECK();
        }
    }
    if (sepm) {
        static CritTable ct;
        static int ct_rc = crit_table(ct);
        if (ct_rc) return ct_rc;
        float *x16, *y16;
        int64_t T16;
        if ((rc = resampled(t16, d_clean, &x16, &T16)) || (rc = resampled(t16, d_deg, &y16, &T16))) return rc;
        double *d_seg = ws.alloc<double>((size_t)B * nf_max), *d_llr = ws.alloc<double>((size_t)B * nf_max),
               *d_wss = ws.alloc<double>((size_t)B * nf_max);
        if (!d_seg || !d_llr || !d_wss) return fail(DFB_ERR_OOM, "cudaMallocAsync failed");
        {
            const size_t smem = sizeof(SepmWarpSmem) * kSepmWarps;
            static PerDeviceOnce attr_once;
            if (auto once_guard = attr_once.first())
                DFB_CUDA(cudaFuncSetAttribute(k_sepm_frames, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            const dim3 grid((unsigned)((nf_max + kSepmWarps - 1) / kSepmWarps), (unsigned)B);
            k_sepm_frames<<<grid, 32 * kSepmWarps, smem, s>>>(x16, y16, T16, d_utt, ct, which, nf_max, d_seg, d_llr, d_wss);
            DFB_LAUNCH_CHECK();
        }
        {
            k_sepm_reduce<<<(unsigned)B, 256, 0, s>>>(d_utt, d_seg, d_llr, d_wss, nf_max, which, d_out, ncol, col[2], col[3],
                                                      col[4]);
            DFB_LAUNCH_CHECK();
        }
    }
    return DFB_OK;
}

extern "C" int dfb_metrics_host(int device, const float *h_clean, const float *h_deg, const int64_t *lengths, int64_t B,
                                int64_t T, int sr, unsigned which, float *h_out) {
    int rc = check_metrics_args(h_clean, h_deg, lengths, B, T, sr, which, h_out);
    if (rc) return rc;
    rc = use_device(device);
    if (rc) return rc;
    const int ncol = __builtin_popcount(which);
    cudaStream_t s = 0;
    float *d_in = nullptr, *d_out = nullptr;
    DFB_CUDA(cudaMalloc(&d_in, sizeof(float) * 2 * B * T));
    if (cudaMalloc(&d_out, sizeof(float) * B * ncol) != cudaSuccess) {
        cudaFree(d_in);
        return fail(DFB_ERR_OOM, "cudaMalloc failed");
    }
    rc = DFB_OK;
    if (cudaMemcpyAsync(d_in, h_clean, sizeof(float) * B * T, cudaMemcpyHostToDevice, s) != cudaSuccess ||
        cudaMemcpyAsync(d_in + B * T, h_deg, sizeof(float) * B * T, cudaMemcpyHostToDevice, s) != cudaSuccess)
        rc = fail(DFB_ERR_CUDA, "host to device copy failed");
    if (!rc) rc = dfb_metrics(device, d_in, d_in + B * T, lengths, B, T, sr, which, d_out, s);
    if (!rc && cudaMemcpy(h_out, d_out, sizeof(float) * B * ncol, cudaMemcpyDeviceToHost) != cudaSuccess)
        rc = fail(DFB_ERR_CUDA, "device to host copy failed: %s", cudaGetErrorString(cudaGetLastError()));
    cudaFree(d_in);
    cudaFree(d_out);
    return rc;
}
