// dfb_dsp.cu -- analysis (windowed real FFT + ERB band energies), feature normalisation scans,
// and the fused apply (ERB gain x spectrum + deep filter) + synthesis (irFFT + window + OLA)
// kernels, plus the C-ABI entry points of the DSP state.
//
// Reference semantics (paths relative to /root/reference):
//   frame_analysis        libDF/src/lib.rs:356-394     (pyDF/src/lib.rs:41-72 batches it)
//   compute_band_corr     libDF/src/lib.rs:280-295, dB at :207-210
//   band_mean_norm_erb    libDF/src/lib.rs:244-251
//   band_unit_norm        libDF/src/lib.rs:253-259
//   apply_interp_band_gain libDF/src/lib.rs:314-326 == Mask.forward DeepFilterNet/df/modules.py:266-269
//   MF.DF                 DeepFilterNet/df/multiframe.py:72-74,126-136,169-180
//   frame_synthesis       libDF/src/lib.rs:396-427     (pyDF/src/lib.rs:74-107)
//
// HBM layout: audio f32[B,T]; spec c64[B,Tf,F] (frame-major, F = fft/2 + 1: 481 bins / 3848 B rows at
// 960 / 480); features f32[B,Tf,E] and c64[B,Tf,nb_df]; every kernel reads/writes whole rows with
// consecutive lanes on consecutive addresses.
// Geometry: fft 960 / hop 480 (every shipped model) runs the specialised kernels k_analysis and, for the shipped models'
// apply shape, k_apply_synthesis; every other supported geometry, and 960 / 480's plain ISTFT and other apply shapes, run
// k_analysis_any / k_apply_synthesis_any (runtime mixed-radix FFT).
#include <cmath>
#include <cstdlib>
#include <cstring>

#include "dfb_common.cuh"
#include "dfb_fft.cuh"

namespace dfb {

thread_local std::string g_err;
std::atomic<int64_t> g_launches{0};

// ---- per-kernel event profiler -------------------------------------------------------------
namespace {
struct ProfRec { std::string name; cudaEvent_t a, b; };
std::vector<ProfRec> g_prof;
std::vector<std::pair<cudaEvent_t, cudaEvent_t>> g_prof_pool;
bool g_prof_on = false;
std::string g_prof_only;
}  // namespace

ProfScope::ProfScope(const char *name, cudaStream_t stream) : s(stream) {
    if (!g_prof_on) return;
    if (!g_prof_only.empty() && g_prof_only != name) return;
    ProfRec r;
    r.name = name;
    if (!g_prof_pool.empty()) {
        r.a = g_prof_pool.back().first; r.b = g_prof_pool.back().second;
        g_prof_pool.pop_back();
    } else if (cudaEventCreate(&r.a) != cudaSuccess || cudaEventCreate(&r.b) != cudaSuccess) {
        return;
    }
    cudaEventRecord(r.a, s);
    g_prof.push_back(r);
    slot = (int)g_prof.size() - 1;
}
ProfScope::~ProfScope() {
    if (slot >= 0) cudaEventRecord(g_prof[slot].b, s);
}

int use_device(int device) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
        return fail(DFB_ERR_CUDA, "no CUDA device available (%s); libdfb200 has no CPU fallback",
                    e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    if (device < 0 || device >= n) return fail(DFB_ERR_INVALID, "device %d out of range [0,%d)", device, n);
    DFB_CUDA(cudaSetDevice(device));
    cudaDeviceProp p;
    DFB_CUDA(cudaGetDeviceProperties(&p, device));
    if (p.major != 10)
        return fail(DFB_ERR_CUDA, "device %d is sm_%d%d; libdfb200 is built for sm_100a only", device, p.major,
                    p.minor);
    return DFB_OK;
}

int Arena::reserve(size_t bytes) {
    if (bytes <= cap) return DFB_OK;
    if (base) {
        DFB_CUDA(cudaDeviceSynchronize());
        DFB_CUDA(cudaFree(base));
        base = nullptr;
        cap = 0;
    }
    size_t want = (bytes + (size_t(1) << 20)) & ~((size_t(1) << 20) - 1);
    cudaError_t e = cudaMalloc(&base, want);
    if (e != cudaSuccess) {
        base = nullptr;
        return fail(DFB_ERR_OOM, "cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e));
    }
    cap = want;
    return DFB_OK;
}
void Arena::release() {
    if (base) cudaFree(base);
    base = nullptr;
    cap = off = 0;
}

// ============================================================================ kernels =====

constexpr int kFft = 960, kHop = 480, kF = 481;
constexpr int kAnaWarps = 8;           // frames per CTA in the analysis kernel (one per warp)
constexpr int kSynWarps = 4;           // warps per CTA in the synthesis kernel
constexpr int kSynChunk = 16;          // consecutive frames per warp in the synthesis kernel
constexpr int kAnaSmem = sizeof(float) * ((kAnaWarps + 1) * 480 + 960) + sizeof(float2) * (242 + kN2 * kN1 + kAnaWarps * kTileFloat2);

// One warp: 480-point complex FFT of the values gathered by `load(n)` (n = 24 n1 + lane), result
// in natural order in buf[0..480).  `buf` is a per-warp shared buffer of kTileFloat2 float2 that
// serves as the pass-A/B transpose tile and then as the natural-order output; `load` may read it.
// tw_lane -> the 20 pass-A twiddles of this lane (shared memory).
template <bool INV, typename LoadF>
__device__ __forceinline__ void warp_fft480(LoadF load, const float2 *tw_lane, float2 *buf, int lane) {
    float2 a[kN1];
    if (lane < kN2) {
#pragma unroll
        for (int n1 = 0; n1 < kN1; n1++) a[n1] = load(kN2 * n1 + lane);
    }
    __syncwarp();
    if (lane < kN2) fft480_pass_a<INV>(a, tw_lane, buf, lane);
    __syncwarp();
    float2 b[kN2];
    if (lane < kN1) fft480_pass_b<INV>(b, buf, lane);
    __syncwarp();
    if (lane < kN1) fft480_store_natural(b, buf, lane);
    __syncwarp();
}

// ERB band energies of one frame from its power spectrum P, in dB, to out[0..E): sequential sum inside each band, factor
// 1/width inside the sum (lib.rs:288-292)
__device__ __forceinline__ void erb_band_db(const float *P, const DspTables &tb, float *out, int lane) {
    for (int band = lane; band < tb.E; band += 32) {
        int o = tb.erb_off[band], n = tb.erb_off[band + 1] - o;
        float kinv = tb.erb_kinv[band];
        float acc = 0.f;
        for (int j = 0; j < n; j++) acc = __fadd_rn(acc, __fmul_rn(P[o + j], kinv));
        out[band] = __fmul_rn(log10f(__fadd_rn(acc, 1e-10f)), 10.f);
    }
}

// ---------------------------------------------------------------------------- analysis ----
// grid (ceil(Tf / kAnaWarps), B), block 32 * kAnaWarps.  Warp w transforms frame t0 + w.
// Algorithmic HBM bytes per frame: 1920 R (audio hop) + 3848 W (spec) + 128 W (erb dB).
// Frame window: the grid covers frames [t_begin, t_begin + nf) of every stream (time-chunked execution); their rows
// go to out_t0 ... of spec / erb_db buffers that hold Tbuf frames per stream.  The whole-signal call is
// (t_begin, nf, out_t0, Tbuf) = (0, Tf, 0, Tf).
__global__ void __launch_bounds__(32 * kAnaWarps, 4)
k_analysis(const float *__restrict__ audio, int64_t T, int Tf, float2 *__restrict__ spec,
           float *__restrict__ erb_db, DspTables tb, const float *__restrict__ init_mem, int t_begin, int nf, int out_t0,
           int Tbuf) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float *s_stage = reinterpret_cast<float *>(smem_raw);                    // (W + 1) * hop
    float *s_win = s_stage + (kAnaWarps + 1) * kHop;                         // fft
    float2 *s_tw960 = reinterpret_cast<float2 *>(s_win + kFft);              // 241 (+1 pad)
    float2 *s_twa = s_tw960 + 242;                                           // pass-A twiddles [24][20]
    float2 *s_buf = s_twa + kN2 * kN1;                                       // W * kTileFloat2
    const int b = blockIdx.y, tl0 = blockIdx.x * kAnaWarps, t0 = t_begin + tl0;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const float *x = audio + (int64_t)b * T;
    const int64_t s_end = (int64_t)Tf * kHop;
    // stage samples [(t0-1)*hop, (t0+W)*hop); zeros before the stream start (analysis_mem = 0).  All 17 loads of a thread
    // are issued into registers before the first store: as a load / store loop with the bounds checks inside, the compiler
    // kept them in program order -- 17 dependent round trips to L2 / HBM per CTA, 85 % of the kernel's stall samples
    // (ncu source page, profiles/README.md) -- 0.565 -> 0.344 ms for 128 x 10 s.
    // (Also tried: a CTA looping over 4 / 8 groups of frames with the next group's samples prefetched into registers during
    // the transforms: 128 registers, 2 CTAs per SM, 0.51 / 0.49 ms.)
    {
        constexpr int kPre = ((kAnaWarps + 1) * kHop + 32 * kAnaWarps - 1) / (32 * kAnaWarps);
        float pre[kPre];
        const int64_t s0 = (int64_t)(t0 - 1) * kHop;
#pragma unroll
        for (int q = 0; q < kPre; q++) {
            const int i = tid + q * 32 * kAnaWarps;
            const int64_t sidx = s0 + i;
            float v = 0.f;
            if (i < (kAnaWarps + 1) * kHop) {
                if (sidx >= 0 && sidx < s_end) v = __ldg(x + sidx);
                else if (sidx < 0 && init_mem) v = init_mem[(int64_t)b * kHop + (kHop + sidx)];  // carried analysis_mem (reset = False)
            }
            pre[q] = v;
        }
        for (int i = tid; i < kFft; i += blockDim.x) s_win[i] = tb.window[i];
        for (int i = tid; i < 241; i += blockDim.x) s_tw960[i] = tb.tw_split[i];
        for (int i = tid; i < kN2 * kN1; i += blockDim.x) s_twa[i] = tb.tw_a_fwd[i];
#pragma unroll
        for (int q = 0; q < kPre; q++) {
            const int i = tid + q * 32 * kAnaWarps;
            if (i < (kAnaWarps + 1) * kHop) s_stage[i] = pre[q];
        }
    }
    __syncthreads();
    const int t = t0 + warp;
    if (tl0 + warp >= nf || t >= Tf) return;
    const int64_t orow = (int64_t)b * Tbuf + out_t0 + tl0 + warp;   // row of this frame in the output buffers
    const float *fr = s_stage + warp * kHop;  // frame t = samples [(t-1) hop, (t+1) hop)
    float2 *nat = s_buf + warp * kTileFloat2;
    warp_fft480<false>(
        [&](int n) {
            float2 v = *reinterpret_cast<const float2 *>(fr + 2 * n);
            float2 w = *reinterpret_cast<const float2 *>(s_win + 2 * n);
            return make_float2(v.x * w.x, v.y * w.y);
        },
        s_twa + (lane < kN2 ? lane : 0) * kN1, nat, lane);
    // split step + wnorm, write spec row, keep |X|^2 for the band energies
    float2 *row = spec + orow * kF;
    float pk[8], pnk[8];
#pragma unroll
    for (int j = 0; j < 8; j++) {
        int k = lane + 32 * j;
        pk[j] = pnk[j] = 0.f;
        if (k <= 240) {
            float2 zk = nat[k], znk = nat[(kC - k) % kC];
            float2 xk, xnk;
            rfft_split(zk, znk, s_tw960[k], xk, xnk);
            xk.x *= tb.wnorm; xk.y *= tb.wnorm;
            xnk.x *= tb.wnorm; xnk.y *= tb.wnorm;
            row[k] = xk;
            if (k != 240) row[kC - k] = xnk;
            pk[j] = __fadd_rn(__fmul_rn(xk.x, xk.x), __fmul_rn(xk.y, xk.y));
            pnk[j] = __fadd_rn(__fmul_rn(xnk.x, xnk.x), __fmul_rn(xnk.y, xnk.y));
        }
    }
    if (erb_db == nullptr) return;
    __syncwarp();
    float *P = reinterpret_cast<float *>(nat);  // 481 floats, reuses the natural-order buffer
#pragma unroll
    for (int j = 0; j < 8; j++) {
        int k = lane + 32 * j;
        if (k <= 240) {
            P[k] = pk[j];
            if (k != 240) P[kC - k] = pnk[j];
        }
    }
    __syncwarp();
    erb_band_db(P, tb, erb_db + orow * tb.E, lane);
}

// ----------------------------------------------------------- generic ERB (libdf.erb) ----
// one warp per frame, arbitrary F / E (API parity path, not the hot path)
__global__ void k_erb(const float2 *__restrict__ spec, int64_t n_frames, int F, const int *__restrict__ off,
                      int E, int db, float *__restrict__ out) {
    int64_t fr = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    int lane = threadIdx.x & 31;
    if (fr >= n_frames) return;
    const float2 *x = spec + fr * F;
    for (int band = lane; band < E; band += 32) {
        int o = off[band], n = off[band + 1] - o;
        float kinv = __fdiv_rn(1.f, (float)n);
        float acc = 0.f;
        for (int j = 0; j < n; j++) {
            float2 v = x[o + j];
            acc = __fadd_rn(acc, __fmul_rn(__fadd_rn(__fmul_rn(v.x, v.x), __fmul_rn(v.y, v.y)), kinv));
        }
        out[fr * E + band] = db ? __fmul_rn(log10f(__fadd_rn(acc, 1e-10f)), 10.f) : acc;
    }
}

__global__ void k_erb_inv(const float *__restrict__ gains, int64_t n_frames, int F, int E,
                          const unsigned char *__restrict__ band_of_bin, float *__restrict__ out) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_frames * F) return;
    int64_t fr = i / F;
    int k = (int)(i - fr * F);
    out[i] = gains[fr * E + band_of_bin[k]];
}

// ------------------------------------------------------------- polyphase resampler ----
// torchaudio.functional.resample as used by df/io.py:107-129 (the reference resamples files to / from the model rate,
// enhance.py:56,85): out[c][i * nw + j] = sum_k kern[j][k] * xpad[c][i * og + k], xpad = x zero padded by `width` in
// front (torchaudio _apply_sinc_resample_kernel: conv1d with stride og).  kern [nw][K = 2 width + og] is built on the
// host exactly like torchaudio's _get_sinc_resample_kernel (io.py resample_kernel).
__global__ void __launch_bounds__(256) k_resample(const float *__restrict__ x, int64_t T, const int64_t *__restrict__ lens,
                                                  const float *__restrict__ kern, int og, int nw, int width, int K,
                                                  float *__restrict__ out, int64_t Tout) {
    extern __shared__ float s_k[];   // the nw x K taps when they fit (else read through L1)
    const bool in_smem = (size_t)nw * K * sizeof(float) <= 96 * 1024;
    if (in_smem) {
        for (int i = threadIdx.x; i < nw * K; i += blockDim.x) s_k[i] = kern[i];
        __syncthreads();
    }
    const float *kk = in_smem ? s_k : kern;
    const int c = blockIdx.y;
    const float *xc = x + (int64_t)c * T;
    // ragged rows (lens != null): row c holds lens[c] samples (the rest of its T is ignored) and yields
    // ceil(nw lens[c] / og) outputs, exactly as that row resampled alone
    const int64_t Tc = lens ? lens[c] : T, Toc = lens ? (nw * Tc + og - 1) / og : Tout;
    for (int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; n < Toc; n += (int64_t)gridDim.x * blockDim.x) {
        const int64_t i = n / nw;
        const int j = (int)(n - i * nw);
        const int64_t p0 = i * og - width;
        const float *kr = kk + (size_t)j * K;
        float acc = 0.f;
        for (int k = 0; k < K; k++) {
            const int64_t p = p0 + k;
            if (p >= 0 && p < Tc) acc = fmaf(kr[k], xc[p], acc);
        }
        out[(int64_t)c * Tout + n] = acc;
    }
}

// ------------------------------------------------------------- feature norm scans ----
// Exponential mean norm of the ERB dB features and exponential unit norm of the first Fd bins,
// sequential in t per (stream, band | bin) exactly like the reference loops.
// grid B, block E + Fd threads (thread j < E: band j; else bin j - E).  Loads are batched kPf
// frames ahead so the dependent chain is arithmetic only.
// kPf = frames of loads in flight per thread: 24 for the enhancement path's shape (E + Fd = 128 threads per stream; with 8
// the kernel was latency bound at 0.10 of HBM), 4 for the generic libdf.erb_norm / unit_norm shapes (up to 1024 threads)
// Ts = frames per stream in the four buffers (the pointers are pre-offset to the first frame to process, Tf = number of
// frames processed); *_state_out (may alias the inputs) receive the EMA states after the last frame.
template <int kPf>
__global__ void __launch_bounds__(kPf > 8 ? 128 : 1024) k_feat_norm(const float *erb_in, int E, int64_t erb_stride_t,
                            const float2 *__restrict__ spec_in, int Fd, int64_t spec_stride_t, int Tf,
                            float alpha, const float *erb_state, const float *unit_state,
                            float *feat_erb, float2 *__restrict__ feat_spec, int Ts, float *erb_state_out,
                            float *unit_state_out) {
    const int b = blockIdx.x, j = threadIdx.x;
    const float one_m_alpha = __fsub_rn(1.f, alpha);
    if (j < E) {
        const float *src = erb_in + (int64_t)b * Ts * erb_stride_t + j;
        float *dst = feat_erb + (int64_t)b * Ts * E + j;
        float s;
        if (erb_state) s = erb_state[(int64_t)b * E + j];
        else s = (E == 1) ? -60.f : __fadd_rn(-60.f, __fmul_rn((float)j, __fdiv_rn(-30.f, (float)(E - 1))));
        // software pipelined: the loads of batch n + 1 are in flight while batch n runs its (sequential) EMA
        float vn[kPf];
#pragma unroll
        for (int u = 0; u < kPf; u++) vn[u] = (u < Tf) ? src[(int64_t)u * erb_stride_t] : 0.f;
        for (int t = 0; t < Tf; t += kPf) {
            float v[kPf];
#pragma unroll
            for (int u = 0; u < kPf; u++) {
                v[u] = vn[u];
                vn[u] = (t + kPf + u < Tf) ? src[(int64_t)(t + kPf + u) * erb_stride_t] : 0.f;
            }
#pragma unroll
            for (int u = 0; u < kPf; u++) {
                if (t + u < Tf) {
                    s = __fadd_rn(__fmul_rn(v[u], one_m_alpha), __fmul_rn(s, alpha));
                    dst[(int64_t)(t + u) * E] = __fdiv_rn(__fsub_rn(v[u], s), 40.f);
                }
            }
        }
        if (erb_state_out) erb_state_out[(int64_t)b * E + j] = s;
    } else if (j < E + Fd) {
        const int k = j - E;
        const float2 *src = spec_in + (int64_t)b * Ts * spec_stride_t + k;
        float2 *dst = feat_spec + (int64_t)b * Ts * Fd + k;
        float s;
        if (unit_state) s = unit_state[(int64_t)b * Fd + k];
        else s = (Fd == 1) ? 0.001f : __fadd_rn(0.001f, __fmul_rn((float)k, __fdiv_rn(__fsub_rn(0.0001f, 0.001f), (float)(Fd - 1))));
        float2 vn[kPf];
#pragma unroll
        for (int u = 0; u < kPf; u++) vn[u] = (u < Tf) ? src[(int64_t)u * spec_stride_t] : make_float2(0.f, 0.f);
        for (int t = 0; t < Tf; t += kPf) {
            float2 v[kPf];
            float nrm[kPf], sv[kPf];
#pragma unroll
            for (int u = 0; u < kPf; u++) {
                v[u] = vn[u];
                vn[u] = (t + kPf + u < Tf) ? src[(int64_t)(t + kPf + u) * spec_stride_t] : make_float2(0.f, 0.f);
            }
            // the magnitudes and the normalisation are independent across frames; only the two-op EMA chain is serial
#pragma unroll
            for (int u = 0; u < kPf; u++) nrm[u] = hypotf(v[u].x, v[u].y);
#pragma unroll
            for (int u = 0; u < kPf; u++) {
                if (t + u < Tf) s = __fadd_rn(__fmul_rn(nrm[u], one_m_alpha), __fmul_rn(s, alpha));
                sv[u] = s;
            }
#pragma unroll
            for (int u = 0; u < kPf; u++) {
                if (t + u < Tf) {
                    float d = __fsqrt_rn(sv[u]);
                    dst[(int64_t)(t + u) * Fd] = make_float2(__fdiv_rn(v[u].x, d), __fdiv_rn(v[u].y, d));
                }
            }
        }
        if (unit_state_out) unit_state_out[(int64_t)b * Fd + k] = s;
    }
}

// Time-segmented version for the enhancement path's shape (E + Fd <= 128 values per stream, long windows): the EMA is a
// linear recurrence, so a stream's frames are cut into kSeg segments scanned concurrently by kSeg x 128 threads --
//   pass 1: every (segment, value) thread runs the recurrence over its segment from state 0 (no stores) -> local end state
//   fold:   state at the start of segment g = alpha^(frames before) * s_in + sum of the earlier local end states, each
//           decayed by alpha^(frames after it) (evaluated in double: at most kSeg terms per thread)
//   pass 2: the same loop as k_feat_norm from the segment's true start state, with the reference's operation order, storing
//           the features (the inputs are re-read from L2)
// The serial chain per thread drops from Tf to 2 Tf / kSeg steps (128 x 10 s: 0.35 -> 0.1 ms); the results differ from
// the one-thread scan only through the rounding of the folded start states (~1e-7 relative).
constexpr int kNormSeg = 8, kNormPf = 8;
template <bool WRITE>
__device__ __forceinline__ float norm_scan_erb(const float *src, int64_t stride, float *dst, int E, int ta, int tb, float s, float alpha,
                                               float one_m_alpha) {
    float vn[kNormPf];
#pragma unroll
    for (int u = 0; u < kNormPf; u++) vn[u] = (ta + u < tb) ? src[(int64_t)(ta + u) * stride] : 0.f;
    for (int t = ta; t < tb; t += kNormPf) {
        float v[kNormPf];
#pragma unroll
        for (int u = 0; u < kNormPf; u++) {
            v[u] = vn[u];
            vn[u] = (t + kNormPf + u < tb) ? src[(int64_t)(t + kNormPf + u) * stride] : 0.f;
        }
#pragma unroll
        for (int u = 0; u < kNormPf; u++) {
            if (t + u < tb) {
                s = __fadd_rn(__fmul_rn(v[u], one_m_alpha), __fmul_rn(s, alpha));
                if (WRITE) dst[(int64_t)(t + u) * E] = __fdiv_rn(__fsub_rn(v[u], s), 40.f);
            }
        }
    }
    return s;
}
template <bool WRITE>
__device__ __forceinline__ float norm_scan_unit(const float2 *src, int64_t stride, float2 *dst, int Fd, int ta, int tb, float s, float alpha,
                                                float one_m_alpha) {
    float2 vn[kNormPf];
#pragma unroll
    for (int u = 0; u < kNormPf; u++) vn[u] = (ta + u < tb) ? src[(int64_t)(ta + u) * stride] : make_float2(0.f, 0.f);
    for (int t = ta; t < tb; t += kNormPf) {
        float2 v[kNormPf];
        float nrm[kNormPf], sv[kNormPf];
#pragma unroll
        for (int u = 0; u < kNormPf; u++) {
            v[u] = vn[u];
            vn[u] = (t + kNormPf + u < tb) ? src[(int64_t)(t + kNormPf + u) * stride] : make_float2(0.f, 0.f);
        }
#pragma unroll
        for (int u = 0; u < kNormPf; u++) nrm[u] = hypotf(v[u].x, v[u].y);
#pragma unroll
        for (int u = 0; u < kNormPf; u++) {
            if (t + u < tb) s = __fadd_rn(__fmul_rn(nrm[u], one_m_alpha), __fmul_rn(s, alpha));
            sv[u] = s;
        }
        if (WRITE) {
#pragma unroll
            for (int u = 0; u < kNormPf; u++) {
                if (t + u < tb) {
                    const float d = __fsqrt_rn(sv[u]);
                    dst[(int64_t)(t + u) * Fd] = make_float2(__fdiv_rn(v[u].x, d), __fdiv_rn(v[u].y, d));
                }
            }
        }
    }
    return s;
}
__global__ void __launch_bounds__(128 * kNormSeg) k_feat_norm_seg(const float *erb_in, int E, int64_t erb_stride_t,
                            const float2 *__restrict__ spec_in, int Fd, int64_t spec_stride_t, int Tf,
                            float alpha, const float *erb_state, const float *unit_state,
                            float *feat_erb, float2 *__restrict__ feat_spec, int Ts, float *erb_state_out,
                            float *unit_state_out) {
    __shared__ float s_loc[kNormSeg][128];
    const int b = blockIdx.x, j = threadIdx.x & 127, seg = threadIdx.x >> 7;
    const float one_m_alpha = __fsub_rn(1.f, alpha);
    const int L = (Tf + kNormSeg - 1) / kNormSeg;
    const int ta = min(seg * L, Tf), tb = min(ta + L, Tf);
    const bool is_erb = j < E, is_unit = !is_erb && j < E + Fd;
    const float *esrc = erb_in + (int64_t)b * Ts * erb_stride_t + j;
    float *edst = feat_erb + (int64_t)b * Ts * E + j;
    const int k = j - E;
    const float2 *usrc = spec_in + (int64_t)b * Ts * spec_stride_t + k;
    float2 *udst = feat_spec + (int64_t)b * Ts * Fd + k;
    float loc = 0.f;
    if (seg + 1 < kNormSeg) {   // the last segment's local end state is never folded
        if (is_erb) loc = norm_scan_erb<false>(esrc, erb_stride_t, nullptr, E, ta, tb, 0.f, alpha, one_m_alpha);
        else if (is_unit) loc = norm_scan_unit<false>(usrc, spec_stride_t, nullptr, Fd, ta, tb, 0.f, alpha, one_m_alpha);
    }
    s_loc[seg][j] = loc;
    __syncthreads();
    if (!is_erb && !is_unit) return;
    float s0;
    if (is_erb) {
        if (erb_state) s0 = erb_state[(int64_t)b * E + j];
        else s0 = (E == 1) ? -60.f : __fadd_rn(-60.f, __fmul_rn((float)j, __fdiv_rn(-30.f, (float)(E - 1))));
    } else {
        if (unit_state) s0 = unit_state[(int64_t)b * Fd + k];
        else s0 = (Fd == 1) ? 0.001f : __fadd_rn(0.001f, __fmul_rn((float)k, __fdiv_rn(__fsub_rn(0.0001f, 0.001f), (float)(Fd - 1))));
    }
    if (seg > 0) {
        double sd = (double)s0;
        const double pL = pow((double)alpha, (double)L);
        for (int g = 0; g < seg; g++) {   // segment g covers min(L, Tf - g L) frames
            const int lg = min(L, max(Tf - g * L, 0));
            sd = sd * (lg == L ? pL : pow((double)alpha, (double)lg)) + (double)s_loc[g][j];
        }
        s0 = (float)sd;
    }
    float s;
    if (is_erb) s = norm_scan_erb<true>(esrc, erb_stride_t, edst, E, ta, tb, s0, alpha, one_m_alpha);
    else s = norm_scan_unit<true>(usrc, spec_stride_t, udst, Fd, ta, tb, s0, alpha, one_m_alpha);
    if (seg == kNormSeg - 1 || tb == Tf) {   // the thread whose segment ends the window owns the carried state
        if (ta < tb || seg == 0) {
            if (is_erb && erb_state_out) erb_state_out[(int64_t)b * E + j] = s;
            if (is_unit && unit_state_out) unit_state_out[(int64_t)b * Fd + k] = s;
        }
    }
}

// ------------------------------------------------------ fused apply + synthesis ----
// mode 0: plain ISTFT of `spec` (pyDF DF.synthesis)
// mode 1: DeepFilterNet3: bins < nb_df <- deep filter of the NOISY spectrum, bins >= nb_df <- spec * gain
// mode 2: DeepFilterNet2: spectrum masked first (all bins), deep filter applied to the masked spectrum
// Optional attenuation limit: X <- noisy * lim + X * (1 - lim)   (enhance.py:238-240)
// One warp owns kSynChunk consecutive frames of one stream and keeps the overlap tail in registers;
// it re-synthesises frame t0-1 to obtain the tail of its first frame.
// Algorithmic HBM bytes per frame (mode 1/2): 3848 R spec + 128 R m + 3840 R coefs + 1920 W audio.

// Valin's post filter on an ERB gain (Mask.pf, modules.py:234-245).  __sinf on [0, pi/2] is within 2^-21 absolute; the
// accurate sinf / hypotf (argument-reduction slow paths, 16 inlined copies in the unrolled bin loop) bloated the apply kernel
// past the instruction cache and cost 30 % even with the filter off.
__device__ __forceinline__ float pf_gain_mask(float m, float beta) {
    const float ms = fmaxf(m * __sinf(3.14159265358979f * m / 2.f), 1e-12f);
    const float q = m / ms;
    return (1.f + beta) * m / (1.f + beta * q * q);
}
// ... and on an enhanced bin y of the noisy bin x (deepfilternet3.py:448-454): returns the factor for y
__device__ __forceinline__ float pf_gain_spec(float2 y, float2 x, float beta) {
    const float eps = 1e-12f;
    const float mask = fminf(fmaxf(sqrtf(y.x * y.x + y.y * y.y) / (sqrtf(x.x * x.x + x.y * x.y) + eps), eps), 1.f);
    const float ms = mask * fmaxf(__sinf(3.14159265358979f * mask / 2.f), eps);
    const float q = mask / ms;
    return (1.f + beta) / (1.f + beta * q * q);
}

// F: spectrum row stride (bins); gains_only: this frame takes the ERB gains on every bin (LSNR stage 2)
__device__ __forceinline__ float2 apply_bin(const ApplyParams &p, const DspTables &tb, const float2 *srow0,
                                            const float *mrow0, const float *crow, int t, int k, int F,
                                            bool gains_only = false) {
    // srow0 / mrow0: row pointers of frame 0 of this stream
    float2 x = srow0[(int64_t)t * F + k];
    float2 y;
    if (p.mode == 0) return x;
    const int band = tb.band_of_bin[k];
    const bool pf2 = p.pf && p.mode == 2;
    if (k >= p.nb_df || p.mask_only || gains_only) {
        float g = mrow0[(int64_t)t * tb.E + band];
        if (pf2) g = pf_gain_mask(g, 0.02f);
        y = make_float2(x.x * g, x.y * g);
    } else {
        // Y[t,k] = sum_o S[t + o - (O-1-L), k] * W[o,t,k]   (multiframe.py:72-74,126-136)
        const float *c = crow + (int64_t)k * (2 * p.order);
        float yr = 0.f, yi = 0.f;
        for (int o = 0; o < p.order; o++) {
            int tt = t + o - (p.order - 1 - p.lookahead);
            if (tt < 0 || tt >= (p.Tv ? p.Tv : p.Tf)) continue;
            float2 s = srow0[(int64_t)tt * F + k];
            if (p.mode == 2 && tt < (p.mc_T ? p.mc_T : p.Tf)) {
                float g = mrow0[(int64_t)tt * tb.E + band];
                if (pf2) g = pf_gain_mask(g, 0.02f);
                s.x *= g; s.y *= g;
            }
            float wr = c[2 * o], wi = c[2 * o + 1];
            yr += s.x * wr - s.y * wi;
            yi += s.x * wi + s.y * wr;
        }
        y = make_float2(yr, yi);
        if (p.alpha && p.mode == 2) {
            const float a = p.alpha[(mrow0 - p.m) / tb.E + t];   // same [b][mc_T] indexing as the mask rows
            float g = mrow0[(int64_t)t * tb.E + band];
            if (pf2) g = pf_gain_mask(g, 0.02f);
            y.x = y.x * a + x.x * g * (1.f - a);
            y.y = y.y * a + x.y * g * (1.f - a);
        }
    }
    if (p.pf && p.mode == 1) { const float g = pf_gain_spec(y, x, p.pf_beta); y.x *= g; y.y *= g; }
    if (p.atten_lim > 0.f) {
        y.x = x.x * p.atten_lim + y.x * (1.f - p.atten_lim);
        y.y = x.y * p.atten_lim + y.y * (1.f - p.atten_lim);
    }
    return y;
}

// LSNR stage of frame row i (tract.rs apply_stages): 0 zero gains, 1 unprocessed, 2 gains only, 3 gains + deep filter
__device__ __forceinline__ int lsnr_stage(const ApplyParams &p, int64_t i) {
    int stage = 3;
    if (p.lsnr) {
        const float l = p.lsnr[i];
        stage = l < p.th_min ? 0 : (l > p.th_erb ? 1 : (l > p.th_df ? 2 : 3));
    }
    return stage;
}

// apply shape of the shipped models: df_order 5, nb_df 96 = 3 DF bins per lane, 32 ERB bands
constexpr int kOrder = 5, kNdfj = 3, kBands = 32;

// Specialised version for the shipped models' apply shape at 960 / 480: a lane owns the bins
// k = lane + 32 j (and 480 - k) for every frame of its chunk, so the deep-filter input history of its DF
// bins lives in registers as a 5-deep shift register (one new look-ahead value per bin and frame instead of
// five reloads), the band gains come from one register per lane via warp shuffles, and all global loads of
// a frame are issued up front, coalesced (256-byte rows), before any use.
// 2 CTAs / SM (no spills) measured fastest.
__global__ void __launch_bounds__(32 * kSynWarps, 2) k_apply_synthesis(ApplyParams p, DspTables tb) {
    __shared__ __align__(16) float s_win[kFft];
    __shared__ __align__(16) float2 s_tw960[241];
    __shared__ __align__(16) float2 s_buf[kSynWarps][kTileFloat2];
    __shared__ __align__(16) float2 s_twa[kN2 * kN1];  // pass-A twiddles, reloaded into registers per frame
    const int b = blockIdx.y;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int i = tid; i < kFft; i += blockDim.x) s_win[i] = tb.window[i];
    for (int i = tid; i < 241; i += blockDim.x) s_tw960[i] = tb.tw_split[i];
    for (int i = tid; i < kN2 * kN1; i += blockDim.x) s_twa[i] = tb.tw_a_inv[i];
    __syncthreads();
    const int syn_chunk = p.frames_per_warp ? p.frames_per_warp : kSynChunk;
    const int t0 = (blockIdx.x * kSynWarps + warp) * syn_chunk;
    if (t0 >= p.Tf) return;
    const int t1 = min(t0 + syn_chunk, p.Tf);
    const int Tf = p.Tf, L = p.lookahead, back = kOrder - 1 - L;
    const int Tv = p.Tv ? p.Tv : Tf;                       // spectrum rows >= Tv do not exist (end of the stream)
    const float2 *srow0 = p.spec + (int64_t)b * (p.spec_T ? p.spec_T : Tf) * kF;
    const int mcT = p.mc_T ? p.mc_T : Tf;                  // m / coefs rows per stream
    const float *mrow0 = p.m + (int64_t)b * mcT * kBands;
    const bool masked_df = p.mode == 2 && !p.mask_only;
    const bool pf1 = p.pf && p.mode == 1, pf2 = p.pf && p.mode == 2;
    const bool blend = p.alpha != nullptr && masked_df;   // DeepFilterNet v1: alpha blend with the masked bin
    const bool need_xk = p.atten_lim > 0.f || pf1 || p.mask_only || p.lsnr || blend;   // noisy DF bins are only loaded when something reads them
    // bands of this lane's bins: bk[j] for k = lane + 32 j, bn[j] for 480 - k
    unsigned long long bkp = 0, bnp = 0;  // 8 band indices each, one byte per j
#pragma unroll
    for (int j = 0; j < 8; j++) {
        const int k = lane + 32 * j;
        bkp |= (unsigned long long)(k <= 240 ? tb.band_of_bin[k] : 0) << (8 * j);
        bnp |= (unsigned long long)(k <= 240 ? tb.band_of_bin[kC - k] : 0) << (8 * j);
    }
#define BK(j) ((int)((bkp >> (8 * (j))) & 0xff))
#define BN(j) ((int)((bnp >> (8 * (j))) & 0xff))
    float2 *nat = s_buf[warp];
    float *yb = reinterpret_cast<float *>(nat);
    float tail[15];
#pragma unroll
    for (int j = 0; j < 15; j++) tail[j] = 0.f;
    // S'[tt][k] for the DF bins; tt = t + o - back.  Rows outside [0, Tf) are zero (multiframe.py:72-74).
    auto load_df_row = [&](int tt, float2 (&dst)[kNdfj]) {
        float g = 1.f;
        const bool ok = tt >= 0 && tt < Tv;
        // (DFN2) the mask of a look-ahead frame beyond the window's DNN frames does not exist yet: such rows are only
        // read for frames that are re-synthesised in the next window
        float mrow = (ok && masked_df && tt < mcT) ? mrow0[(int64_t)tt * kBands + lane] : 1.f;
        if (pf2 && ok && masked_df && tt < mcT) mrow = pf_gain_mask(mrow, 0.02f);
#pragma unroll
        for (int j = 0; j < kNdfj; j++) {
            float2 v = ok ? srow0[(int64_t)tt * kF + lane + 32 * j] : make_float2(0.f, 0.f);
            if (masked_df) { g = __shfl_sync(0xffffffffu, mrow, BK(j)); v.x *= g; v.y *= g; }
            dst[j] = v;
        }
    };
    const int tstart = t0 > 0 ? t0 - 1 : 0;
    float2 hist[kOrder][kNdfj];
#pragma unroll
    for (int o = 1; o < kOrder; o++) load_df_row(tstart + o - 1 - back, hist[o]);  // becomes taps 0..O-2 after the first shift
    for (int t = tstart; t < t1; t++) {
        // ---- loads of this frame, all issued before use
        float mcur = mrow0[(int64_t)t * kBands + lane];
        if (pf2) mcur = pf_gain_mask(mcur, 0.02f);
        const float al = blend ? p.alpha[(int64_t)b * mcT + t] : 1.f;
        const int stage = lsnr_stage(p, (int64_t)b * mcT + t);
#pragma unroll
        for (int o = 0; o < kOrder - 1; o++)
#pragma unroll
            for (int j = 0; j < kNdfj; j++) hist[o][j] = hist[o + 1][j];
        load_df_row(t + L, hist[kOrder - 1]);
        float2 cf[kNdfj][kOrder];
        const float2 *crow = reinterpret_cast<const float2 *>(p.coefs + ((int64_t)b * mcT + t) * (kNdfj * 32) * (2 * kOrder));
#pragma unroll
        for (int j = 0; j < kNdfj; j++)
#pragma unroll
            for (int o = 0; o < kOrder; o++) cf[j][o] = crow[(lane + 32 * j) * kOrder + o];
        float2 xk[8], xn[8];
        const float2 *srow = srow0 + (int64_t)t * kF;
#pragma unroll
        for (int j = 0; j < 8; j++) {
            const int k = lane + 32 * j;
            xk[j] = (k <= 240 && (j >= kNdfj || need_xk)) ? srow[k] : make_float2(0.f, 0.f);
            xn[j] = k <= 240 ? srow[kC - k] : make_float2(0.f, 0.f);
        }
        // ---- deep filter (bins < 96), gain (others), optional attenuation limit
#pragma unroll
        for (int j = 0; j < 8; j++) {
            const int k = lane + 32 * j;
            float2 y;
            if (j < kNdfj && !p.mask_only && stage == 3) {
                float yr = 0.f, yi = 0.f;
#pragma unroll
                for (int o = 0; o < kOrder; o++) {
                    const float2 s = hist[o][j], w = cf[j][o];
                    yr += s.x * w.x - s.y * w.y;
                    yi += s.x * w.y + s.y * w.x;
                }
                y = make_float2(yr, yi);
                if (blend) {
                    const float g = __shfl_sync(0xffffffffu, mcur, BK(j)) * (1.f - al);
                    y.x = y.x * al + xk[j].x * g; y.y = y.y * al + xk[j].y * g;
                }
            } else {
                const float g = __shfl_sync(0xffffffffu, mcur, BK(j));
                y = make_float2(xk[j].x * g, xk[j].y * g);
            }
            const float gn = __shfl_sync(0xffffffffu, mcur, BN(j));
            float2 yn = make_float2(xn[j].x * gn, xn[j].y * gn);
            if (stage == 0) { y = make_float2(0.f, 0.f); yn = y; }
            else if (stage == 1) { y = xk[j]; yn = xn[j]; }
            if (pf1 && stage >= 2) {
                const float g1 = pf_gain_spec(y, xk[j], p.pf_beta), g2 = pf_gain_spec(yn, xn[j], p.pf_beta);
                y.x *= g1; y.y *= g1; yn.x *= g2; yn.y *= g2;
            }
            if (p.atten_lim > 0.f) {
                const float a = p.atten_lim, c = 1.f - a;
                y.x = xk[j].x * a + y.x * c; y.y = xk[j].y * a + y.y * c;
                yn.x = xn[j].x * a + yn.x * c; yn.y = xn[j].y * a + yn.y * c;
            }
            if (k <= 240) {
                if (p.spec_out && t >= t0) {
                    float2 *orow = p.spec_out + ((int64_t)b * Tf + t) * kF;
                    orow[k] = y;
                    orow[kC - k] = yn;
                }
                if (k == 0) { y.y = 0.f; yn.y = 0.f; }  // imag of DC / Nyquist ignored (lib.rs:402)
                const float2 w = s_tw960[k];
                float2 zk, znk;
                irfft_merge(y, yn, make_float2(w.x, -w.y), zk, znk);
                nat[k] = zk;
                if (k > 0 && k < 240) nat[kC - k] = znk;
            }
        }
        __syncwarp();
        if (p.audio) {
            warp_fft480<true>([&](int n) { return nat[n]; }, s_twa + (lane < kN2 ? lane : 0) * kN1, nat, lane);
#pragma unroll
            for (int j = 0; j < 15; j++) {
                int n = lane + 32 * j;
                float2 v = nat[n];
                float2 w = *reinterpret_cast<const float2 *>(s_win + 2 * n);
                nat[n] = make_float2(v.x * w.x, v.y * w.y);
            }
            __syncwarp();
            float *orow = p.audio + (int64_t)b * p.out_stride;
#pragma unroll
            for (int j = 0; j < 15; j++) {
                int i = lane + 32 * j;
                float o = yb[i] + tail[j];      // lib.rs:407-411
                tail[j] = yb[kHop + i];         // lib.rs:423-426 (hop == fft/2)
                int64_t g = (int64_t)t * kHop + i - p.out_offset;
                if (t >= t0 && t >= p.t_first && g >= 0 && g < p.out_len) orow[g] = o;
            }
        }
        __syncwarp();
    }
}

// ================================================== runtime mixed-radix kernels (any geometry) ====
// fft = N = 2 M (M <= 2048 with no prime factor above 7), any hop H <= N / 2.  One warp per frame runs the runtime
// mixed-radix transform of dfb_fft.cuh in shared memory (dynamic): per CTA the window [N], tw_m [M] and tw_split
// [M/2 + 1]; per warp two M-point ping-pong buffers and, in the synthesis kernel, the overlap-add memory [N - H].
constexpr int kAnyAnaWarps = 4, kAnySynWarps = 4;
// profiler names (dfb_profile_report); constants rather than literals at the launch sites because bench.py's roofline table
// lists the kernels of the 960 / 480 workloads it runs, and these kernels never run there
constexpr const char *kAnaAnyName = "k_analysis_any", *kSynAnyName = "k_apply_synthesis_any";
constexpr int kAnySmemCap = 200 * 1024;   // the synthesis launcher halves its warps per CTA until the CTA fits

__host__ __device__ inline size_t any_align16(size_t b) { return (b + 15) & ~size_t(15); }
__host__ __device__ inline size_t any_cta_bytes(int N) {
    const int M = N / 2;
    return any_align16(sizeof(float) * N) + any_align16(sizeof(float2) * (M + M / 2 + 1));
}
__host__ __device__ inline size_t any_warp_bytes(int N, int H, bool syn) {
    return any_align16(sizeof(float2) * N) + (syn ? any_align16(sizeof(float) * (N - H)) : 0);
}
__host__ inline size_t any_smem_bytes(int N, int H, int warps, bool syn) {
    return any_cta_bytes(N) + (size_t)warps * any_warp_bytes(N, H, syn);
}

// per-CTA tables into shared memory; returns the first per-warp byte
__device__ __forceinline__ unsigned char *any_load_tables(unsigned char *smem, const DspTables &tb, float *&s_win, float2 *&s_twm,
                                                          float2 *&s_tws) {
    const int N = tb.fft, M = N / 2;
    s_win = reinterpret_cast<float *>(smem);
    s_twm = reinterpret_cast<float2 *>(smem + any_align16(sizeof(float) * N));
    s_tws = s_twm + M;
    for (int i = threadIdx.x; i < N; i += blockDim.x) s_win[i] = tb.window[i];
    for (int i = threadIdx.x; i < M; i += blockDim.x) s_twm[i] = tb.tw_m[i];
    for (int i = threadIdx.x; i <= M / 2; i += blockDim.x) s_tws[i] = tb.tw_split[i];
    return smem + any_cta_bytes(N);
}

// Analysis of any geometry: same arguments and frame window as k_analysis (t_begin, nf, out_t0, Tbuf, row_stride,
// init_mem).  Frame t covers samples [t H - (N - H), t H + H) (libDF analysis_mem of N - H samples, lib.rs:360-384);
// init_mem [B][N - H] holds the samples before the stream start (null: zeros).
// grid (ceil(nf / kAnyAnaWarps), B), block 32 * kAnyAnaWarps.
// Algorithmic HBM bytes per frame: 4 H R (audio hop) + 8 F W (spec) + 4 E W (erb dB).
__global__ void __launch_bounds__(32 * kAnyAnaWarps)
k_analysis_any(const float *__restrict__ audio, int64_t T, int Tf, float2 *__restrict__ spec, float *__restrict__ erb_db,
               DspTables tb, const float *__restrict__ init_mem, int t_begin, int nf, int out_t0, int Tbuf) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float *s_win;
    float2 *s_twm, *s_tws;
    unsigned char *wbase = any_load_tables(smem_raw, tb, s_win, s_twm, s_tws);
    __syncthreads();
    const int N = tb.fft, M = N / 2, H = tb.hop, F = tb.F, mem_n = N - H;
    const int b = blockIdx.y, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int tl = blockIdx.x * kAnyAnaWarps + warp, t = t_begin + tl;
    if (tl >= nf || t >= Tf) return;
    float2 *A = reinterpret_cast<float2 *>(wbase + (size_t)warp * any_warp_bytes(N, H, false)), *Bf = A + M;
    const float *x = audio + (int64_t)b * T;
    const int64_t s0 = (int64_t)t * H - mem_n, s_end = (int64_t)Tf * H;
    auto sample = [&](int n) -> float {
        const int64_t i = s0 + n;
        if (i >= 0) return i < s_end ? __ldg(x + i) : 0.f;
        return init_mem ? init_mem[(int64_t)b * mem_n + (mem_n + i)] : 0.f;   // carried analysis_mem (reset = False)
    };
    for (int n = lane; n < M; n += 32)
        A[n] = make_float2(sample(2 * n) * s_win[2 * n], sample(2 * n + 1) * s_win[2 * n + 1]);
    __syncwarp();
    const float2 *Z = warp_fft_any<false>(A, Bf, s_twm, M, lane);
    float2 *P2 = Z == A ? Bf : A;   // the free buffer: |X|^2 for the band energies (F <= 2 M floats)
    float *P = reinterpret_cast<float *>(P2);
    const int64_t orow = (int64_t)b * Tbuf + out_t0 + tl;
    float2 *row = spec + orow * F;
    for (int k = lane; k <= M / 2; k += 32) {
        float2 xk, xnk;
        rfft_split(Z[k], Z[(M - k) % M], s_tws[k], xk, xnk);
        xk.x *= tb.wnorm; xk.y *= tb.wnorm;
        xnk.x *= tb.wnorm; xnk.y *= tb.wnorm;
        row[k] = xk;
        P[k] = __fadd_rn(__fmul_rn(xk.x, xk.x), __fmul_rn(xk.y, xk.y));
        if (2 * k != M) {
            row[M - k] = xnk;
            P[M - k] = __fadd_rn(__fmul_rn(xnk.x, xnk.x), __fmul_rn(xnk.y, xnk.y));
        }
    }
    if (erb_db == nullptr) return;
    __syncwarp();
    erb_band_db(P, tb, erb_db + orow * tb.E, lane);
}

// Fused apply + synthesis of any geometry, for every apply shape and every ApplyParams field, including the LSNR stage
// gating (mode 1); at 960 / 480 it serves the plain ISTFT and the shapes k_apply_synthesis is not specialised for.
// Overlap-add as libDF frame_synthesis (lib.rs:407-426, S = N - 2 H >= 0):
//   out[t H + i] = y_t[i] + mem[i] (i < H);  mem <- (mem[H + j] (j < S) or 0) + y_t[H + j]  (j < N - H)
// One warp owns frames_per_warp consecutive frames and keeps mem in shared memory; it re-synthesises the
// R = ceil((N - H) / H) frames before its first one to rebuild mem.  With carry (mode 0) the channels form one signal:
// the re-synthesised frames may lie in the channels before (rows -1, -2, ... of the contiguous [C,Tf,F] spectrum) and
// the first frame of channel 0 starts from init_tail.
// Algorithmic HBM bytes per frame (mode 1/2): 8 F R spec + 4 E R m + 8 O nb_df R coefs + 4 H W audio.
__global__ void __launch_bounds__(32 * kAnySynWarps) k_apply_synthesis_any(ApplyParams p, DspTables tb) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float *s_win;
    float2 *s_twm, *s_tws;
    unsigned char *wbase = any_load_tables(smem_raw, tb, s_win, s_twm, s_tws);
    __syncthreads();
    const int N = tb.fft, M = N / 2, H = tb.hop, F = tb.F, mem_n = N - H, S = N - 2 * H, R = (N - 1) / H;
    const int warps = blockDim.x >> 5;
    const int b = blockIdx.y, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int t0 = (blockIdx.x * warps + warp) * p.frames_per_warp;
    if (t0 >= p.Tf) return;
    const int t1 = min(t0 + p.frames_per_warp, p.Tf);
    float2 *A = reinterpret_cast<float2 *>(wbase + (size_t)warp * any_warp_bytes(N, H, true)), *Bf = A + M;
    float *mem = reinterpret_cast<float *>(Bf + M);
    const float2 *srow0 = p.spec + (int64_t)b * (p.spec_T ? p.spec_T : p.Tf) * F;
    const int mcT = p.mc_T ? p.mc_T : p.Tf;
    const float *mrow0 = p.m ? p.m + (int64_t)b * mcT * tb.E : nullptr;
    const int tmin = p.carry ? -b * p.Tf : 0;   // first frame of the (carried) signal relative to this channel
    const int tstart = max(t0 - R, tmin);
    const bool from_init = p.carry && p.init_tail && tstart == tmin;
    for (int j = lane; j < mem_n; j += 32) mem[j] = from_init ? p.init_tail[j] : 0.f;
    float *orow = p.audio ? p.audio + (int64_t)b * p.out_stride : nullptr;
    for (int t = tstart; t < t1; t++) {
        const float *crow = p.coefs ? p.coefs + ((int64_t)b * mcT + t) * p.nb_df * (2 * p.order) : nullptr;
        const int stage = lsnr_stage(p, (int64_t)b * mcT + t);
        auto bin = [&](int k) -> float2 {
            if (stage >= 2) return apply_bin(p, tb, srow0, mrow0, crow, t, k, F, stage == 2);
            const float2 x = srow0[(int64_t)t * F + k];
            if (stage == 1) return x;
            return make_float2(x.x * p.atten_lim, x.y * p.atten_lim);   // zero gains, then the attenuation limit
        };
        for (int k = lane; k <= M / 2; k += 32) {
            float2 xk = bin(k), xnk = bin(M - k);
            if (p.spec_out && t >= t0) {
                float2 *so = p.spec_out + ((int64_t)b * p.Tf + t) * F;
                so[k] = xk;
                so[M - k] = xnk;
            }
            if (k == 0) { xk.y = 0.f; xnk.y = 0.f; }  // imag of DC / Nyquist ignored (lib.rs:402)
            const float2 w = s_tws[k];
            float2 zk, znk;
            irfft_merge(xk, xnk, make_float2(w.x, -w.y), zk, znk);
            A[k] = zk;
            if (k > 0 && 2 * k != M) A[M - k] = znk;
        }
        __syncwarp();
        if (orow) {
            float *y = reinterpret_cast<float *>(warp_fft_any<true>(A, Bf, s_twm, M, lane));   // y[n], n < N
            const bool emit = t >= t0 && t >= p.t_first;
            for (int i = lane; i < H; i += 32) {
                const float o = y[i] * s_win[i] + mem[i];     // lib.rs:407-411
                const int64_t g = (int64_t)t * H + i - p.out_offset;
                if (emit && g >= 0 && g < p.out_len) orow[g] = o;
            }
            for (int j = lane; j < mem_n; j += 32)            // lib.rs:416-426 (rotate_left by H, add, override)
                y[H + j] = y[H + j] * s_win[H + j] + (j < S ? mem[H + j] : 0.f);
            __syncwarp();
            for (int j = lane; j < mem_n; j += 32) mem[j] = y[H + j];
        }
        __syncwarp();
    }
    if (p.final_tail && b == (int)gridDim.y - 1 && t1 == p.Tf)
        for (int j = lane; j < mem_n; j += 32) p.final_tail[j] = mem[j];
}

}  // namespace dfb

// ====================================================================== host side / C ABI ==
using namespace dfb;

extern "C" const char *dfb_last_error(void) { return g_err.c_str(); }
extern "C" const char *dfb_version(void) { return "dfb200 0.1.0 sm_100a"; }
extern "C" int64_t dfb_kernel_launches(void) { return g_launches.load(); }

extern "C" int dfb_profile_enable(int on, const char *only_kernel) {
    g_prof_on = on != 0;
    g_prof_only = only_kernel ? only_kernel : "";
    return DFB_OK;
}

// Writes "name count total_ms\n" lines for everything recorded since the last report and clears.
extern "C" int64_t dfb_profile_report(char *buf, int64_t buflen) {
    if (!buf || buflen <= 0) return fail(DFB_ERR_INVALID, "bad buffer");
    cudaDeviceSynchronize();
    std::vector<std::string> names;
    std::vector<double> ms;
    std::vector<int64_t> cnt;
    // DFB_PROF_TIMELINE=1: start / end of every launch relative to the first one, to stderr (critical-path analysis)
    static const bool timeline = getenv("DFB_PROF_TIMELINE") && atoi(getenv("DFB_PROF_TIMELINE"));
    for (auto &r : g_prof) {
        float t = 0.f;
        if (cudaEventElapsedTime(&t, r.a, r.b) != cudaSuccess) t = 0.f;
        if (timeline) {
            float t0 = 0.f;
            cudaEventElapsedTime(&t0, g_prof.front().a, r.a);
            fprintf(stderr, "[timeline] %-34s %9.3f %9.3f\n", r.name.c_str(), t0, t0 + t);
        }
        size_t i = 0;
        for (; i < names.size(); i++) if (names[i] == r.name) break;
        if (i == names.size()) { names.push_back(r.name); ms.push_back(0); cnt.push_back(0); }
        ms[i] += t; cnt[i] += 1;
        g_prof_pool.push_back({r.a, r.b});
    }
    g_prof.clear();
    std::string out;
    char line[256];
    for (size_t i = 0; i < names.size(); i++) {
        snprintf(line, sizeof line, "%s %lld %.6f\n", names[i].c_str(), (long long)cnt[i], ms[i]);
        out += line;
    }
    if ((int64_t)out.size() + 1 > buflen) return fail(DFB_ERR_INVALID, "profile buffer too small");
    memcpy(buf, out.c_str(), out.size() + 1);
    return (int64_t)out.size();
}

// libDF/src/lib.rs:42-47,68-100 (f32 arithmetic, integer result)
extern "C" int dfb_erb_widths(int sr, int fft_size, int nb_erb, int min_nb_freqs, int64_t *out) {
    if (!out || nb_erb <= 0 || nb_erb > kMaxErb || fft_size <= 0) return fail(DFB_ERR_INVALID, "bad erb parameters");
    auto freq2erb = [](float f) { return 9.265f * log1pf(f / (24.7f * 9.265f)); };
    auto erb2freq = [](float e) { return 24.7f * 9.265f * (expf(e / 9.265f) - 1.f); };
    int nyq = sr / 2;
    float freq_width = (float)sr / (float)fft_size;
    float erb_low = freq2erb(0.f), erb_high = freq2erb((float)nyq);
    float step = (erb_high - erb_low) / (float)nb_erb;
    int prev_freq = 0, freq_over = 0;
    for (int i = 1; i <= nb_erb; i++) {
        float f = erb2freq(erb_low + (float)i * step);
        int fb = (int)roundf(f / freq_width);
        int nb = fb - prev_freq - freq_over;
        if (nb < min_nb_freqs) {
            freq_over = min_nb_freqs - nb;
            nb = min_nb_freqs;
        } else {
            freq_over = 0;
        }
        out[i - 1] = nb;
        prev_freq = fb;
    }
    out[nb_erb - 1] += 1;
    int64_t sum = 0;
    for (int i = 0; i < nb_erb; i++) sum += out[i];
    int64_t too_large = sum - (fft_size / 2 + 1);
    if (too_large > 0) out[nb_erb - 1] -= too_large;
    return DFB_OK;
}

extern "C" int dfb_state_create(dfb_state **out, int device, int sr, int fft_size, int hop_size, int nb_erb,
                                int min_nb_erb_freqs) {
    if (!out) return fail(DFB_ERR_INVALID, "null out");
    *out = nullptr;
    if (hop_size * 2 > fft_size) return fail(DFB_ERR_INVALID, "assertion failed: hop_size * 2 <= fft_size");
    if (hop_size <= 0) return fail(DFB_ERR_INVALID, "hop_size must be positive (got %d)", hop_size);
    // 960 / 480 has specialised kernels; every other geometry needs a size the runtime mixed-radix FFT supports
    const bool spec960 = fft_size == kFft && hop_size == kHop;
    if (!spec960 && (fft_size % 2 || fft_size < 32 || fft_size > 2 * kAnyMaxM || !fft_any_supported(fft_size / 2)))
        return fail(DFB_ERR_UNSUPPORTED,
                    "fft_size %d is not supported: fft_size must be even, 32 <= fft_size <= 4096, and fft_size / 2 must have "
                    "no prime factor above 7",
                    fft_size);
    if (nb_erb <= 0 || nb_erb > kMaxErb) return fail(DFB_ERR_INVALID, "nb_erb out of range");
    int rc = use_device(device);
    if (rc) return rc;
    dfb_state *st = new dfb_state();
    st->device = device; st->sr = sr; st->fft = fft_size; st->hop = hop_size; st->nb_erb = nb_erb;
    st->min_nb_erb_freqs = min_nb_erb_freqs;
    st->analysis_mem.assign(fft_size - hop_size, 0.f);
    st->synthesis_mem.assign(fft_size - hop_size, 0.f);
    st->erb.resize(nb_erb);
    dfb_erb_widths(sr, fft_size, nb_erb, min_nb_erb_freqs, st->erb.data());
    const int F = fft_size / 2 + 1, M = fft_size / 2;
    // vorbis window, f64 -> f32 (lib.rs:126-132)
    st->window.resize(fft_size);
    const double pi = 3.14159265358979323846;
    for (int i = 0; i < fft_size; i++) {
        double s = sin(0.5 * pi * ((double)i + 0.5) / (double)(fft_size / 2));
        st->window[i] = (float)sin(0.5 * pi * s * s);
    }
    // one slab: window | tw_a_fwd | tw_a_inv (960 / 480 only: the specialised kernels) | tw_split | tw_m | erb_off | erb_kinv |
    // band_of_bin
    const int n_twa = spec960 ? kN2 * kN1 : 0;
    std::vector<float2> twf(n_twa), twi(n_twa), tw_split(M / 2 + 1), tw_m(M);
    for (int l = 0; l < kN2 && spec960; l++)
        for (int k1 = 0; k1 < kN1; k1++) {
            double a = 2.0 * pi * (double)((l * k1) % kC) / (double)kC;
            twf[l * kN1 + k1] = make_float2((float)cos(a), (float)-sin(a));
            twi[l * kN1 + k1] = make_float2((float)cos(a), (float)sin(a));
        }
    for (int k = 0; k <= M / 2; k++) {
        double a = 2.0 * pi * (double)k / (double)fft_size;
        tw_split[k] = make_float2((float)cos(a), (float)-sin(a));
    }
    for (int k = 0; k < M; k++) {
        double a = 2.0 * pi * (double)k / (double)M;
        tw_m[k] = make_float2((float)cos(a), (float)-sin(a));
    }
    std::vector<int> off(nb_erb + 1, 0);
    std::vector<float> kinv(nb_erb);
    std::vector<unsigned char> bob(F);
    for (int b = 0; b < nb_erb; b++) {
        off[b + 1] = off[b] + (int)st->erb[b];
        kinv[b] = 1.f / (float)st->erb[b];
        for (int k = off[b]; k < off[b + 1] && k < F; k++) bob[k] = (unsigned char)b;
    }
    if (off[nb_erb] != F) {
        delete st;
        return fail(DFB_ERR_INVALID, "erb widths sum to %d, expected %d", off[nb_erb], F);
    }
    auto a256 = [](size_t b) { return (b + 255) & ~size_t(255); };
    size_t o_win = 0, o_twf = o_win + a256(sizeof(float) * fft_size), o_twi = o_twf + a256(sizeof(float2) * twf.size()),
           o_split = o_twi + a256(sizeof(float2) * twi.size()), o_twm = o_split + a256(sizeof(float2) * tw_split.size()),
           o_off = o_twm + a256(sizeof(float2) * tw_m.size()), o_kinv = o_off + sizeof(int) * (kMaxErb + 1 + 3),
           o_bob = o_kinv + sizeof(float) * kMaxErb, total = o_bob + a256(F);
    std::vector<char> slab(total, 0);
    memcpy(slab.data() + o_win, st->window.data(), sizeof(float) * fft_size);
    memcpy(slab.data() + o_twf, twf.data(), sizeof(float2) * twf.size());
    memcpy(slab.data() + o_twi, twi.data(), sizeof(float2) * twi.size());
    memcpy(slab.data() + o_split, tw_split.data(), sizeof(float2) * tw_split.size());
    memcpy(slab.data() + o_twm, tw_m.data(), sizeof(float2) * tw_m.size());
    memcpy(slab.data() + o_off, off.data(), sizeof(int) * off.size());
    memcpy(slab.data() + o_kinv, kinv.data(), sizeof(float) * kinv.size());
    memcpy(slab.data() + o_bob, bob.data(), bob.size());
    char *d = nullptr;
    if (cudaMalloc(&d, total) != cudaSuccess || cudaMemcpy(d, slab.data(), total, cudaMemcpyHostToDevice) != cudaSuccess) {
        delete st;
        return fail(DFB_ERR_CUDA, "table upload failed: %s", cudaGetErrorString(cudaGetLastError()));
    }
    st->d_tables = d;
    st->tb.window = (const float *)(d + o_win);
    st->tb.tw_a_fwd = spec960 ? (const float2 *)(d + o_twf) : nullptr;
    st->tb.tw_a_inv = spec960 ? (const float2 *)(d + o_twi) : nullptr;
    st->tb.tw_split = (const float2 *)(d + o_split);
    st->tb.tw_m = (const float2 *)(d + o_twm);
    st->tb.erb_off = (const int *)(d + o_off);
    st->tb.erb_kinv = (const float *)(d + o_kinv);
    st->tb.band_of_bin = (const unsigned char *)(d + o_bob);
    st->tb.wnorm = 1.f / ((float)((int64_t)fft_size * fft_size) / (float)(2 * hop_size));  // lib.rs:133
    st->tb.fft = fft_size; st->tb.hop = hop_size; st->tb.F = F; st->tb.E = nb_erb;
    cudaFuncSetAttribute(k_analysis_any, cudaFuncAttributeMaxDynamicSharedMemorySize, kAnySmemCap);
    cudaFuncSetAttribute(k_apply_synthesis_any, cudaFuncAttributeMaxDynamicSharedMemorySize, kAnySmemCap);
    cudaFuncSetAttribute(k_analysis, cudaFuncAttributeMaxDynamicSharedMemorySize, kAnaSmem);
    if (cudaStreamCreateWithFlags(&st->stream, cudaStreamNonBlocking) != cudaSuccess) {
        cudaFree(d);
        delete st;
        return fail(DFB_ERR_CUDA, "stream creation failed");
    }
    *out = st;
    return DFB_OK;
}

extern "C" void dfb_state_free(dfb_state *st) {
    if (!st) return;
    cudaSetDevice(st->device);
    st->arena.release();
    if (st->d_tables) cudaFree(st->d_tables);
    if (st->stream) cudaStreamDestroy(st->stream);
    delete st;
}

extern "C" int dfb_state_erb_widths(const dfb_state *st, int64_t *w) {
    if (!st || !w) return fail(DFB_ERR_INVALID, "null argument");
    memcpy(w, st->erb.data(), sizeof(int64_t) * st->nb_erb);
    return DFB_OK;
}
extern "C" int dfb_state_fft_window(const dfb_state *st, float *w) {
    if (!st || !w) return fail(DFB_ERR_INVALID, "null argument");
    memcpy(w, st->window.data(), sizeof(float) * st->fft);
    return DFB_OK;
}
extern "C" int dfb_state_params(const dfb_state *st, int *sr, int *fft, int *hop, int *nb_erb) {
    if (!st) return fail(DFB_ERR_INVALID, "null state");
    if (sr) *sr = st->sr;
    if (fft) *fft = st->fft;
    if (hop) *hop = st->hop;
    if (nb_erb) *nb_erb = st->nb_erb;
    return DFB_OK;
}

namespace dfb {

int launch_analysis(dfb_state *st, const float *d_audio, int64_t C, int64_t T, float *d_spec, float *d_erb_db,
                    cudaStream_t s, const float *d_init_mem, const AnaWindow *w) {
    int64_t Tf = T / st->hop;
    if (C <= 0 || Tf <= 0) return DFB_OK;
    if (C > 65535) return fail(DFB_ERR_INVALID, "more than 65535 channels per call");
    const int t_begin = w ? w->t_begin : 0, nf = w ? w->nf : (int)Tf, out_t0 = w ? w->out_t0 : 0, Tbuf = w ? w->Tbuf : (int)Tf;
    if (nf <= 0) return DFB_OK;
    const int64_t row_stride = w && w->row_stride ? w->row_stride : T;
    if (st->fft == kFft && st->hop == kHop) {
        dim3 grid((unsigned)((nf + kAnaWarps - 1) / kAnaWarps), (unsigned)C);
        DFB_PROF("k_analysis", s);
        k_analysis<<<grid, 32 * kAnaWarps, kAnaSmem, s>>>(d_audio, row_stride, (int)Tf, (float2 *)d_spec, d_erb_db, st->tb,
                                                         d_init_mem, t_begin, nf, out_t0, Tbuf);
    } else {
        dim3 grid((unsigned)((nf + kAnyAnaWarps - 1) / kAnyAnaWarps), (unsigned)C);
        DFB_PROF(kAnaAnyName, s);
        k_analysis_any<<<grid, 32 * kAnyAnaWarps, any_smem_bytes(st->fft, st->hop, kAnyAnaWarps, false), s>>>(
            d_audio, row_stride, (int)Tf, (float2 *)d_spec, d_erb_db, st->tb, d_init_mem, t_begin, nf, out_t0, Tbuf);
    }
    DFB_LAUNCH_CHECK();
    return DFB_OK;
}

int launch_feat_norm(const float *d_erb, int E, int64_t erb_stride, const float *d_spec, int Fd, int64_t spec_stride,
                     int64_t C, int64_t Tf, float alpha, const float *d_erb_state, const float *d_unit_state,
                     float *d_feat_erb, float *d_feat_spec, cudaStream_t s, int64_t Ts, float *d_erb_state_out,
                     float *d_unit_state_out) {
    if (C <= 0 || Tf <= 0 || E + Fd == 0) return DFB_OK;
    if (E + Fd > 1024) return fail(DFB_ERR_INVALID, "E + F > 1024 in norm scan");
    int threads = ((E + Fd + 31) / 32) * 32;
    DFB_PROF("k_feat_norm", s);
    if (threads <= 128 && Tf >= 16 * kNormSeg)
        k_feat_norm_seg<<<(unsigned)C, 128 * kNormSeg, 0, s>>>(d_erb, E, erb_stride, (const float2 *)d_spec, Fd, spec_stride, (int)Tf,
                                                            alpha, d_erb_state, d_unit_state, d_feat_erb, (float2 *)d_feat_spec,
                                                            (int)(Ts > 0 ? Ts : Tf), d_erb_state_out, d_unit_state_out);
    else if (threads <= 128)
        k_feat_norm<24><<<(unsigned)C, threads, 0, s>>>(d_erb, E, erb_stride, (const float2 *)d_spec, Fd, spec_stride, (int)Tf,
                                                       alpha, d_erb_state, d_unit_state, d_feat_erb, (float2 *)d_feat_spec,
                                                       (int)(Ts > 0 ? Ts : Tf), d_erb_state_out, d_unit_state_out);
    else
        k_feat_norm<4><<<(unsigned)C, threads, 0, s>>>(d_erb, E, erb_stride, (const float2 *)d_spec, Fd, spec_stride, (int)Tf,
                                                      alpha, d_erb_state, d_unit_state, d_feat_erb, (float2 *)d_feat_spec,
                                                      (int)(Ts > 0 ? Ts : Tf), d_erb_state_out, d_unit_state_out);
    DFB_LAUNCH_CHECK();
    return DFB_OK;
}

int launch_apply_synthesis(dfb_state *st, const ApplyParams &p, int64_t B, cudaStream_t s) {
    if (B <= 0 || p.Tf <= 0) return DFB_OK;
    if (B > 65535) return fail(DFB_ERR_INVALID, "more than 65535 channels per call");
    if (p.mode != 0 && (p.nb_df > st->tb.F || p.order > 8))
        return fail(DFB_ERR_UNSUPPORTED, "nb_df > %d bins or df_order > 8", st->tb.F);
    if (p.lsnr && !(p.mode == 1 && p.m && p.coefs))
        return fail(DFB_ERR_UNSUPPORTED, "LSNR stage gating is built for DeepFilterNet3 (apply mode 1) only");
    // frames per warp: 16 amortises the re-synthesis of the frame before a warp's first one; short windows (time chunks)
    // take 8 so that the grid still fills the device with a few waves
    ApplyParams q = p;
    q.frames_per_warp = (B * (int64_t)p.Tf / kSynChunk >= 6000) ? kSynChunk : kSynChunk / 2;
    if (st->fft == kFft && st->hop == kHop && p.mode != 0 && p.order == kOrder && p.nb_df == 32 * kNdfj && st->tb.E == kBands &&
        p.m && p.coefs) {
        const int per_cta = kSynWarps * q.frames_per_warp;
        dim3 grid((unsigned)((p.Tf + per_cta - 1) / per_cta), (unsigned)B);
        DFB_PROF("k_apply_synthesis", s);
        k_apply_synthesis<<<grid, 32 * kSynWarps, 0, s>>>(q, st->tb);
    } else {
        int warps = kAnySynWarps;
        while (warps > 1 && any_smem_bytes(st->fft, st->hop, warps, true) > (size_t)kAnySmemCap) warps /= 2;
        const int per_cta = warps * q.frames_per_warp;
        dim3 grid((unsigned)((p.Tf + per_cta - 1) / per_cta), (unsigned)B);
        DFB_PROF(kSynAnyName, s);
        k_apply_synthesis_any<<<grid, 32 * warps, any_smem_bytes(st->fft, st->hop, warps, true), s>>>(q, st->tb);
    }
    DFB_LAUNCH_CHECK();
    return DFB_OK;
}

}  // namespace dfb

extern "C" int dfb_analysis(dfb_state *st, const float *d_audio, int64_t C, int64_t T, float *d_spec, void *stream) {
    if (!st || !d_audio || !d_spec) return fail(DFB_ERR_INVALID, "null argument");
    DFB_CUDA(cudaSetDevice(st->device));
    return launch_analysis(st, d_audio, C, T, d_spec, nullptr, (cudaStream_t)stream);
}

extern "C" int dfb_state_reset(dfb_state *st);

// pyDF DF.analysis(input, reset): reset != 0 starts every channel from zero memory (pyDF/src/lib.rs:56-58);
// reset == 0 carries the STFT memory from the previous call into channel 0 and from channel c into c + 1
// (one DFState is shared by all channels).  Either way the memory left behind is the last hop of the last channel.
// analysis_mem after the frames of one channel: the last fft - hop samples of [mem, x[0, L)) (lib.rs:375-384)
static void next_analysis_mem(const float *mem, const float *x, int64_t L, int64_t mn, float *out) {
    for (int64_t j = 0; j < mn; j++) out[j] = L + j < mn ? mem[L + j] : x[L + j - mn];
}

extern "C" int dfb_analysis_host_ex(dfb_state *st, const float *h_audio, int64_t C, int64_t T, int reset, float *h_spec) {
    if (!st || !h_audio || !h_spec) return fail(DFB_ERR_INVALID, "null argument");
    if (C <= 0 || T <= 0) return fail(DFB_ERR_INVALID, "[df] Input array empty or not contiguous.");
    DFB_CUDA(cudaSetDevice(st->device));
    const int64_t Tf = T / st->hop, hop = st->hop, mn = st->fft - st->hop;
    if (reset) dfb_state_reset(st);  // DFState::reset clears BOTH memories (libDF/src/lib.rs:156-159)
    size_t nb_in = sizeof(float) * C * T, nb_out = sizeof(float) * 2 * C * Tf * st->tb.F;
    int rc = st->arena.reserve(nb_in + nb_out + sizeof(float) * C * mn + 2048);
    if (rc) return rc;
    st->arena.reset();
    float *d_in = st->arena.take<float>(C * T), *d_out = st->arena.take<float>(2 * C * Tf * st->tb.F + 2);
    float *d_mem = nullptr;
    DFB_CUDA(cudaMemcpyAsync(d_in, h_audio, nb_in, cudaMemcpyHostToDevice, st->stream));
    // memory each channel starts from: channel 0 the carried one, channel c the one channel c - 1 leaves
    std::vector<float> mem;
    if (!reset && Tf > 0) {
        mem.resize((size_t)C * mn);
        memcpy(mem.data(), st->analysis_mem.data(), sizeof(float) * mn);
        for (int64_t c = 1; c < C; c++) next_analysis_mem(mem.data() + (c - 1) * mn, h_audio + (c - 1) * T, Tf * hop, mn, mem.data() + c * mn);
        d_mem = st->arena.take<float>(C * mn);
        DFB_CUDA(cudaMemcpyAsync(d_mem, mem.data(), sizeof(float) * C * mn, cudaMemcpyHostToDevice, st->stream));
    }
    rc = launch_analysis(st, d_in, C, T, d_out, nullptr, st->stream, d_mem);
    if (rc) return rc;
    if (nb_out) DFB_CUDA(cudaMemcpyAsync(h_spec, d_out, nb_out, cudaMemcpyDeviceToHost, st->stream));
    DFB_CUDA(cudaStreamSynchronize(st->stream));
    if (Tf > 0) {
        const std::vector<float> start = mem.empty() ? st->analysis_mem : std::vector<float>(mem.end() - mn, mem.end());
        next_analysis_mem(start.data(), h_audio + (C - 1) * T, Tf * hop, mn, st->analysis_mem.data());
    }
    return DFB_OK;
}
extern "C" int dfb_analysis_host(dfb_state *st, const float *h_audio, int64_t C, int64_t T, float *h_spec) {
    return dfb_analysis_host_ex(st, h_audio, C, T, 1, h_spec);
}
extern "C" int dfb_state_reset(dfb_state *st) {
    if (!st) return fail(DFB_ERR_INVALID, "null state");
    std::fill(st->analysis_mem.begin(), st->analysis_mem.end(), 0.f);
    std::fill(st->synthesis_mem.begin(), st->synthesis_mem.end(), 0.f);
    return DFB_OK;
}

extern "C" int dfb_synthesis(dfb_state *st, const float *d_spec, int64_t C, int64_t Tf, float *d_audio, void *stream) {
    if (!st || !d_spec || !d_audio) return fail(DFB_ERR_INVALID, "null argument");
    DFB_CUDA(cudaSetDevice(st->device));
    ApplyParams p{};
    p.spec = (const float2 *)d_spec; p.audio = d_audio; p.out_stride = Tf * st->hop; p.out_offset = 0;
    p.out_len = Tf * st->hop; p.Tf = (int)Tf; p.mode = 0;
    return launch_apply_synthesis(st, p, C, (cudaStream_t)stream);
}

// pyDF DF.synthesis(input, reset): see dfb_analysis_host_ex for the reset semantics (pyDF/src/lib.rs:91-93).
extern "C" int dfb_synthesis_host_ex(dfb_state *st, const float *h_spec, int64_t C, int64_t Tf, int reset, float *h_audio) {
    if (!st || !h_spec || !h_audio) return fail(DFB_ERR_INVALID, "null argument");
    if (C <= 0 || Tf <= 0) return fail(DFB_ERR_INVALID, "[df] Input array empty or not contiguous.");
    DFB_CUDA(cudaSetDevice(st->device));
    const int64_t hop = st->hop, mn = st->fft - st->hop;   // synthesis_mem holds fft - hop samples
    if (reset) dfb_state_reset(st);  // clears the analysis memory as well (libDF/src/lib.rs:156-159)
    size_t nb_in = sizeof(float) * 2 * C * Tf * st->tb.F, nb_out = sizeof(float) * C * Tf * hop;
    int rc = st->arena.reserve(nb_in + nb_out + sizeof(float) * 2 * mn + 2048);
    if (rc) return rc;
    st->arena.reset();
    float *d_in = st->arena.take<float>(2 * C * Tf * st->tb.F), *d_out = st->arena.take<float>(C * Tf * hop);
    float *d_init = st->arena.take<float>(mn), *d_final = st->arena.take<float>(mn);
    DFB_CUDA(cudaMemcpyAsync(d_in, h_spec, nb_in, cudaMemcpyHostToDevice, st->stream));
    DFB_CUDA(cudaMemcpyAsync(d_init, st->synthesis_mem.data(), sizeof(float) * mn, cudaMemcpyHostToDevice, st->stream));
    ApplyParams p{};
    p.spec = (const float2 *)d_in; p.audio = d_out; p.out_stride = Tf * hop; p.out_offset = 0;
    p.out_len = Tf * hop; p.Tf = (int)Tf; p.mode = 0;
    p.carry = reset ? 0 : 1; p.init_tail = d_init; p.final_tail = d_final;
    rc = launch_apply_synthesis(st, p, C, st->stream);
    if (rc) return rc;
    DFB_CUDA(cudaMemcpyAsync(h_audio, d_out, nb_out, cudaMemcpyDeviceToHost, st->stream));
    DFB_CUDA(cudaMemcpyAsync(st->synthesis_mem.data(), d_final, sizeof(float) * mn, cudaMemcpyDeviceToHost, st->stream));
    DFB_CUDA(cudaStreamSynchronize(st->stream));
    return DFB_OK;
}
extern "C" int dfb_synthesis_host(dfb_state *st, const float *h_spec, int64_t C, int64_t Tf, float *h_audio) {
    return dfb_synthesis_host_ex(st, h_spec, C, Tf, 1, h_audio);
}

namespace {
// tiny RAII scratch for the stateless *_host helpers
struct Scratch {
    std::vector<void *> ptrs;
    ~Scratch() { for (void *p : ptrs) cudaFree(p); }
    template <typename T>
    T *alloc(size_t n) {
        void *p = nullptr;
        if (cudaMalloc(&p, (n ? n : 1) * sizeof(T)) != cudaSuccess) return nullptr;
        ptrs.push_back(p);
        return (T *)p;
    }
};
}  // namespace

extern "C" int dfb_erb_host(int device, const float *h_spec, int64_t n_frames, int64_t F, const int64_t *widths, int E,
                            int db, float *h_out) {
    if (!h_spec || !widths || !h_out || n_frames <= 0 || F <= 0 || E <= 0) return fail(DFB_ERR_INVALID, "bad argument");
    std::vector<int> off(E + 1, 0);
    for (int b = 0; b < E; b++) off[b + 1] = off[b] + (int)widths[b];
    if (off[E] != F) return fail(DFB_ERR_INVALID, "DF shape error: erb widths sum to %d but input has %lld bins", off[E], (long long)F);
    int rc = use_device(device);
    if (rc) return rc;
    Scratch s;
    float2 *d_in = s.alloc<float2>(n_frames * F);
    float *d_out = s.alloc<float>(n_frames * E);
    int *d_off = s.alloc<int>(E + 1);
    if (!d_in || !d_out || !d_off) return fail(DFB_ERR_OOM, "cudaMalloc failed");
    DFB_CUDA(cudaMemcpy(d_in, h_spec, sizeof(float2) * n_frames * F, cudaMemcpyHostToDevice));
    DFB_CUDA(cudaMemcpy(d_off, off.data(), sizeof(int) * (E + 1), cudaMemcpyHostToDevice));
    k_erb<<<(unsigned)((n_frames + 7) / 8), 256>>>(d_in, n_frames, (int)F, d_off, E, db, d_out);
    DFB_LAUNCH_CHECK();
    DFB_CUDA(cudaMemcpy(h_out, d_out, sizeof(float) * n_frames * E, cudaMemcpyDeviceToHost));
    return DFB_OK;
}

extern "C" int dfb_erb_inv_host(int device, const float *h_gains, int64_t n_frames, const int64_t *widths, int E,
                                float *h_out) {
    if (!h_gains || !widths || !h_out || n_frames <= 0 || E <= 0 || E > 255) return fail(DFB_ERR_INVALID, "bad argument");
    int64_t F = 0;
    for (int b = 0; b < E; b++) F += widths[b];
    std::vector<unsigned char> bob(F);
    int64_t o = 0;
    for (int b = 0; b < E; b++) { for (int64_t j = 0; j < widths[b]; j++) bob[o + j] = (unsigned char)b; o += widths[b]; }
    int rc = use_device(device);
    if (rc) return rc;
    Scratch s;
    float *d_in = s.alloc<float>(n_frames * E), *d_out = s.alloc<float>(n_frames * F);
    unsigned char *d_bob = s.alloc<unsigned char>(F);
    if (!d_in || !d_out || !d_bob) return fail(DFB_ERR_OOM, "cudaMalloc failed");
    DFB_CUDA(cudaMemcpy(d_in, h_gains, sizeof(float) * n_frames * E, cudaMemcpyHostToDevice));
    DFB_CUDA(cudaMemcpy(d_bob, bob.data(), F, cudaMemcpyHostToDevice));
    int64_t n = n_frames * F;
    k_erb_inv<<<(unsigned)((n + 255) / 256), 256>>>(d_in, n_frames, (int)F, E, d_bob, d_out);
    DFB_LAUNCH_CHECK();
    DFB_CUDA(cudaMemcpy(h_out, d_out, sizeof(float) * n, cudaMemcpyDeviceToHost));
    return DFB_OK;
}

extern "C" int dfb_erb_norm_host(int device, const float *h_erb, int64_t C, int64_t T, int64_t E, float alpha,
                                 const float *h_state, float *h_out) {
    if (!h_erb || !h_out || C <= 0 || T <= 0 || E <= 0) return fail(DFB_ERR_INVALID, "bad argument");
    int rc = use_device(device);
    if (rc) return rc;
    Scratch s;
    float *d_in = s.alloc<float>(C * T * E), *d_out = s.alloc<float>(C * T * E), *d_st = nullptr;
    if (!d_in || !d_out) return fail(DFB_ERR_OOM, "cudaMalloc failed");
    DFB_CUDA(cudaMemcpy(d_in, h_erb, sizeof(float) * C * T * E, cudaMemcpyHostToDevice));
    if (h_state) {
        d_st = s.alloc<float>(C * E);
        DFB_CUDA(cudaMemcpy(d_st, h_state, sizeof(float) * C * E, cudaMemcpyHostToDevice));
    }
    rc = launch_feat_norm(d_in, (int)E, E, nullptr, 0, 0, C, T, alpha, d_st, nullptr, d_out, nullptr, 0);
    if (rc) return rc;
    DFB_CUDA(cudaMemcpy(h_out, d_out, sizeof(float) * C * T * E, cudaMemcpyDeviceToHost));
    return DFB_OK;
}

extern "C" int dfb_unit_norm_host(int device, const float *h_spec, int64_t C, int64_t T, int64_t F, float alpha,
                                  const float *h_state, float *h_out) {
    if (!h_spec || !h_out || C <= 0 || T <= 0 || F <= 0) return fail(DFB_ERR_INVALID, "bad argument");
    int rc = use_device(device);
    if (rc) return rc;
    Scratch s;
    float *d_in = s.alloc<float>(2 * C * T * F), *d_out = s.alloc<float>(2 * C * T * F), *d_st = nullptr;
    if (!d_in || !d_out) return fail(DFB_ERR_OOM, "cudaMalloc failed");
    DFB_CUDA(cudaMemcpy(d_in, h_spec, sizeof(float) * 2 * C * T * F, cudaMemcpyHostToDevice));
    if (h_state) {
        d_st = s.alloc<float>(C * F);
        DFB_CUDA(cudaMemcpy(d_st, h_state, sizeof(float) * C * F, cudaMemcpyHostToDevice));
    }
    rc = launch_feat_norm(nullptr, 0, 0, d_in, (int)F, F, C, T, alpha, nullptr, d_st, nullptr, d_out, 0);
    if (rc) return rc;
    DFB_CUDA(cudaMemcpy(h_out, d_out, sizeof(float) * 2 * C * T * F, cudaMemcpyDeviceToHost));
    return DFB_OK;
}

extern "C" int dfb_unit_norm_init(int64_t n, float *h_out) {
    if (!h_out || n <= 0) return fail(DFB_ERR_INVALID, "bad argument");
    if (n == 1) { h_out[0] = 0.001f; return DFB_OK; }
    float step = (0.0001f - 0.001f) / (float)(n - 1);
    for (int64_t i = 0; i < n; i++) h_out[i] = 0.001f + (float)i * step;
    return DFB_OK;
}

extern "C" int dfb_features(dfb_state *st, const float *d_audio, int64_t C, int64_t T, int nb_df, float alpha,
                            float *d_spec, float *d_feat_erb, float *d_feat_spec, void *stream) {
    if (!st || !d_audio || !d_spec || !d_feat_erb || !d_feat_spec) return fail(DFB_ERR_INVALID, "null argument");
    if (nb_df <= 0 || nb_df > st->tb.F) return fail(DFB_ERR_INVALID, "nb_df out of range");
    DFB_CUDA(cudaSetDevice(st->device));
    cudaStream_t s = (cudaStream_t)stream;
    int64_t Tf = T / st->hop;
    // raw ERB dB goes to feat_erb and is normalised in place by the scan kernel
    int rc = launch_analysis(st, d_audio, C, T, d_spec, d_feat_erb, s);
    if (rc) return rc;
    return launch_feat_norm(d_feat_erb, st->tb.E, st->tb.E, d_spec, nb_df, st->tb.F, C, Tf, alpha, nullptr, nullptr,
                            d_feat_erb, d_feat_spec, s);
}

extern "C" int dfb_features_host(dfb_state *st, const float *h_audio, int64_t C, int64_t T, int nb_df, float alpha,
                                 float *h_spec, float *h_feat_erb, float *h_feat_spec) {
    if (!st || !h_audio || !h_spec || !h_feat_erb || !h_feat_spec) return fail(DFB_ERR_INVALID, "null argument");
    if (C <= 0 || T <= 0) return fail(DFB_ERR_INVALID, "[df] Input array empty or not contiguous.");
    DFB_CUDA(cudaSetDevice(st->device));
    int64_t Tf = T / st->hop, F = st->tb.F, E = st->tb.E;
    size_t n_spec = 2 * C * Tf * F, n_fe = C * Tf * E, n_fs = 2 * C * Tf * nb_df;
    int rc = st->arena.reserve(sizeof(float) * (C * T + n_spec + n_fe + n_fs) + 4096);
    if (rc) return rc;
    st->arena.reset();
    float *d_in = st->arena.take<float>(C * T), *d_spec = st->arena.take<float>(n_spec + 2),
          *d_fe = st->arena.take<float>(n_fe + 1), *d_fs = st->arena.take<float>(n_fs + 2);
    DFB_CUDA(cudaMemcpyAsync(d_in, h_audio, sizeof(float) * C * T, cudaMemcpyHostToDevice, st->stream));
    rc = dfb_features(st, d_in, C, T, nb_df, alpha, d_spec, d_fe, d_fs, st->stream);
    if (rc) return rc;
    if (Tf > 0) {
        DFB_CUDA(cudaMemcpyAsync(h_spec, d_spec, sizeof(float) * n_spec, cudaMemcpyDeviceToHost, st->stream));
        DFB_CUDA(cudaMemcpyAsync(h_feat_erb, d_fe, sizeof(float) * n_fe, cudaMemcpyDeviceToHost, st->stream));
        DFB_CUDA(cudaMemcpyAsync(h_feat_spec, d_fs, sizeof(float) * n_fs, cudaMemcpyDeviceToHost, st->stream));
    }
    DFB_CUDA(cudaStreamSynchronize(st->stream));
    return DFB_OK;
}

namespace dfb {
int launch_resample(const float *d_x, int64_t C, int64_t T, const int64_t *d_lens, const float *d_kern, int og, int nw, int width,
                    float *d_out, int64_t T_out, cudaStream_t s) {
    if (C > 65535) return fail(DFB_ERR_INVALID, "more than 65535 channels per call");
    const int K = 2 * width + og;
    const size_t smem = (size_t)nw * K * sizeof(float) <= 96 * 1024 ? (size_t)nw * K * sizeof(float) : 0;
    static PerDeviceOnce attr_once;
    if (auto once_guard = attr_once.first()) DFB_CUDA(cudaFuncSetAttribute(k_resample, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
    int64_t blocks = (T_out + 255) / 256;
    if (blocks > 4096) blocks = 4096;
    k_resample<<<dim3((unsigned)blocks, (unsigned)C), 256, smem, s>>>(d_x, T, d_lens, d_kern, og, nw, width, K, d_out, T_out);
    DFB_LAUNCH_CHECK();
    return DFB_OK;
}
}  // namespace dfb

// df/io.py resample (torchaudio.functional.resample): h_audio [C][T] -> h_out [C][T_out]; h_kernel [nw][2 width + og]
extern "C" int dfb_resample_host(int device, const float *h_audio, int64_t C, int64_t T, const float *h_kernel, int og, int nw,
                                 int width, float *h_out, int64_t T_out) {
    if (!h_audio || !h_kernel || !h_out || C <= 0 || T <= 0 || T_out <= 0 || og <= 0 || nw <= 0 || width < 0)
        return fail(DFB_ERR_INVALID, "bad resample argument");
    if (C > 65535) return fail(DFB_ERR_INVALID, "more than 65535 channels per call");
    int rc = use_device(device);
    if (rc) return rc;
    const int K = 2 * width + og;
    Scratch s;
    float *d_in = s.alloc<float>(C * T), *d_out = s.alloc<float>(C * T_out), *d_k = s.alloc<float>((size_t)nw * K);
    if (!d_in || !d_out || !d_k) return fail(DFB_ERR_OOM, "cudaMalloc failed");
    DFB_CUDA(cudaMemcpy(d_in, h_audio, sizeof(float) * C * T, cudaMemcpyHostToDevice));
    DFB_CUDA(cudaMemcpy(d_k, h_kernel, sizeof(float) * (size_t)nw * K, cudaMemcpyHostToDevice));
    rc = launch_resample(d_in, C, T, nullptr, d_k, og, nw, width, d_out, T_out, 0);
    if (rc) return rc;
    DFB_CUDA(cudaMemcpy(h_out, d_out, sizeof(float) * C * T_out, cudaMemcpyDeviceToHost));
    return DFB_OK;
}
