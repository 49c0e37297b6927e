// dfb_common.cuh -- shared host-side plumbing of libdfb200.so (error reporting, launch counter,
// grow-only device arena) and the device tables of the DSP state.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/dfb200.h"

namespace dfb {

extern thread_local std::string g_err;
extern std::atomic<int64_t> g_launches;

inline int fail(int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}

#define DFB_CUDA(expr)                                                                          \
    do {                                                                                        \
        cudaError_t e__ = (expr);                                                               \
        if (e__ != cudaSuccess)                                                                 \
            return dfb::fail(DFB_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), \
                             __FILE__, __LINE__);                                               \
    } while (0)

#define DFB_LAUNCH_CHECK()                                                                      \
    do {                                                                                        \
        dfb::g_launches.fetch_add(1, std::memory_order_relaxed);                                \
        cudaError_t e__ = cudaGetLastError();                                                   \
        if (e__ != cudaSuccess)                                                                 \
            return dfb::fail(DFB_ERR_CUDA, "kernel launch failed: %s (%s:%d)",                  \
                             cudaGetErrorString(e__), __FILE__, __LINE__);                      \
    } while (0)

// Optional per-kernel timing with CUDA events on the launching stream (dfb_profile_* in the C ABI).
// Off by default; when on, every launch site brackets its kernel with two events.
struct ProfScope {
    int slot = -1;
    cudaStream_t s;
    ProfScope(const char *name, cudaStream_t stream);
    ~ProfScope();
};
#define DFB_PROF(name, stream) dfb::ProfScope prof_scope__(name, stream)

// Function attributes (dynamic shared memory limit, cluster size) are per device: launch sites set them the first
// time they run on each device of the process.  `first()` hands the caller a guard that holds the mutex while the
// one-time setup runs, so a second host thread cannot launch before the attribute is in place:
//     if (auto g = once.first()) { cudaFuncSetAttribute(...); }
struct PerDeviceOnce {
    std::mutex mu;
    std::atomic<unsigned long long> done{0};
    struct Guard {
        std::unique_lock<std::mutex> lk;
        PerDeviceOnce *o = nullptr;
        unsigned long long bit = 0;
        Guard() = default;
        Guard(Guard &&g) noexcept : lk(std::move(g.lk)), o(g.o), bit(g.bit) {}
        explicit operator bool() const { return lk.owns_lock(); }
        ~Guard() { if (lk.owns_lock()) o->done.fetch_or(bit, std::memory_order_release); }
    };
    Guard first() {
        int d = 0;
        cudaGetDevice(&d);
        const unsigned long long bit = 1ull << (d & 63);
        Guard g;
        if (done.load(std::memory_order_acquire) & bit) return g;
        g.lk = std::unique_lock<std::mutex>(mu);
        if (done.load(std::memory_order_acquire) & bit) { g.lk.unlock(); g.lk.release(); return g; }
        g.o = this; g.bit = bit;
        return g;
    }
};

// Selects `device` and verifies it is a Blackwell part; no CPU fallback exists.
int use_device(int device);

// Grow-only device arena: one cudaMalloc'd slab, bump allocated per call, reset between calls.
struct Arena {
    char *base = nullptr;
    size_t cap = 0, off = 0;
    int reserve(size_t bytes);  // ensure capacity (may reallocate; invalidates old pointers)
    void reset() { off = 0; }
    template <typename T>
    T *take(size_t n) {
        size_t b = (n * sizeof(T) + 255) & ~size_t(255);
        if (off + b > cap) return nullptr;
        T *p = reinterpret_cast<T *>(base + off);
        off += b;
        return p;
    }
    void release();
};

constexpr int kMaxErb = 64;

// Device-resident tables of one DSP state.  M = fft / 2; the specialised 960 / 480 kernels (k_analysis,
// k_apply_synthesis) read tw_a_*, the runtime FFT (dfb_fft.cuh) of every other kernel tw_m.
struct DspTables {
    const float *window;     // [fft]
    const float2 *tw_a_fwd;  // [24][20]  w480^{-lane k1} (960 / 480 only, else null)
    const float2 *tw_a_inv;  // [24][20]  conj
    const float2 *tw_split;  // [M/2 + 1] e^{-2 pi i k / fft}  (real split / merge steps)
    const float2 *tw_m;      // [M]       e^{-2 pi i k / M}    (runtime FFT passes)
    const int *erb_off;      // [E + 1]
    const float *erb_kinv;   // [E]  1 / width
    const unsigned char *band_of_bin;  // [F]
    float wnorm;
    int fft, hop, F, E;
};

// Parameters of the fused apply + synthesis kernel (dfb_dsp.cu).
// mode 0: plain ISTFT; 1: DeepFilterNet3 (DF on the noisy spectrum); 2: DeepFilterNet2 (DF on the
// masked spectrum).
struct ApplyParams {
    const float2 *spec;   // [B,Tf,F]
    const float *m;       // [B,Tf,E] or null
    const float *coefs;   // [B,Tf,nb_df,2*order] or null
    float *audio;         // [B, out_stride] or null
    float2 *spec_out;     // optional [B,Tf,F]: enhanced spectrum (dfb_apply) or null
    int64_t out_stride;
    int64_t out_offset;   // first synthesised sample that is written (n_fft - hop when pad)
    int64_t out_len;
    int Tf, mode, nb_df, order, lookahead;
    // time-chunked execution (0 = whole signal): the spectrum buffer holds spec_T frames per stream of which Tv exist
    // (rows >= Tv are the end of the stream: zero for the deep filter taps), m / coefs hold Tf; audio of frames < t_first
    // is not written (they belong to the previous window and are only re-synthesised for the overlap-add tail)
    int spec_T, Tv, t_first;
    int mc_T;             // frames per stream in m / coefs (0 = Tf)
    int frames_per_warp;  // consecutive frames one warp synthesises (set by the launcher)
    // optional stages: post filter (DFN3: on the enhanced spectrum, deepfilternet3.py:448-454; DFN2: on the ERB gains,
    // modules.py:234-245 with beta = 0.02) and mask_only (run_df = False: no deep filter, every bin takes the ERB gain)
    int pf, mask_only;
    float pf_beta;
    // LSNR stage gating of the streaming runtime (libDF/src/tract.rs:658-672), mode 1 only: lsnr [B][mc_T] or null;
    // lsnr < th_min -> zero gains, no DF; > th_erb -> frame passes unprocessed; > th_df -> gains only; else gains + DF
    const float *lsnr;
    float th_min, th_erb, th_df;
    // DeepFilterNet v1 (mode 2): alpha [B][mc_T] or null; DF bins <- alpha * deep filter + (1 - alpha) * masked bin
    // (assign_df, modules.py:470-478)
    const float *alpha;
    float atten_lim;      // 0 = off
    // carried ISTFT state (pyDF synthesis(reset=False), mode 0 only): channel 0 starts from init_tail,
    // channel c > 0 from the tail left by channel c - 1; the tail after the last frame goes to final_tail
    const float *init_tail;  // [fft - hop] or null
    float *final_tail;       // [fft - hop] or null
    int carry;
};

}  // namespace dfb

struct dfb_state;
namespace dfb {
// frame window of launch_analysis: frames [t_begin, t_begin + nf) of a signal of T samples per row (row pitch row_stride,
// 0 = T) go to rows out_t0 ... of buffers holding Tbuf frames per stream.  Frame t covers samples
// [t hop - (fft - hop), t hop + hop); samples before 0 come from d_init_mem [C][fft - hop] (null: zeros).
struct AnaWindow { int t_begin, nf, out_t0, Tbuf; int64_t row_stride; };
int launch_analysis(dfb_state *st, const float *d_audio, int64_t C, int64_t T, float *d_spec, float *d_erb_db,
                    cudaStream_t s, const float *d_init_mem = nullptr, const AnaWindow *w = nullptr);
// Ts: frames per stream in the buffers (0 = Tf; pointers pre-offset to the first frame); *_state_out: EMA states after
// the last frame (may be null / alias the inputs)
int launch_feat_norm(const float *d_erb, int E, int64_t erb_stride, const float *d_spec, int Fd, int64_t spec_stride,
                     int64_t C, int64_t Tf, float alpha, const float *d_erb_state, const float *d_unit_state,
                     float *d_feat_erb, float *d_feat_spec, cudaStream_t s, int64_t Ts = 0, float *d_erb_state_out = nullptr,
                     float *d_unit_state_out = nullptr);
int launch_apply_synthesis(dfb_state *st, const ApplyParams &p, int64_t B, cudaStream_t s);
// time window of a recurrence launch: steps 0 .. T-1 are frames t0 .. of buffers holding Ts frames per stream; h0 (null:
// zeros) / hT (null: not stored) are the carried hidden states [B][H]
struct GruWindow { const float *h0; float *hT; int t0, Ts; };
// tensor-core GRU recurrence, H = 256 (dfb_tc.cu)
int launch_gru_tc(cudaStream_t s, const float *xproj, const float *whh, const float *bhh, const float *res, float *hout,
                  unsigned short *hout_hi, unsigned short *hout_lo, int B, int T, long long *dbg = nullptr, int wide = 0,
                  int planes_res = 0, const GruWindow *w = nullptr, int H = 256);
// BF16x3 tcgen05 GEMM on hi/lo planes (dfb_tc.cu)
int launch_gemm_bf16x3(cudaStream_t s, const void *x_hi, const void *x_lo, int64_t ldx, const void *w_hi, const void *w_lo,
                       const float *bias, float *y, int64_t ldy, int64_t M, int N, int K);
// BF16x3 tcgen05 grouped linear on hi/lo planes + host-packed weight image (dfb_gl.cu); DFB_ERR_UNSUPPORTED when the
// shape is outside the kernel (the caller falls back to the FFMA kernel)
int launch_gl_bx(cudaStream_t s, const unsigned short *x_hi, const unsigned short *x_lo, int64_t ldx, const float *w_img,
                 const float *res, int64_t ldr, float *y, int64_t ldy, unsigned short *y_hi, unsigned short *y_lo, int64_t ldp,
                 int64_t M, int G, int Ig, int Hg, int act, float oscale, float ooffset);
bool gl_bx_geometry(int G, int Ig, int Hg, int *gpc_out, int *hgp_out, int *stages_out);
// DF pathway conv (df_convp) on tensor cores (dfb_tc.cu)
int launch_df_convp_tc(cudaStream_t s, const float *c0, const float *w_sw, const float *w2, const float *bias, float *coefs, int B, int T,
                       int Fd);
// fp32 [M][K] -> BF16 hi / lo planes [M][K]
int launch_to_planes(cudaStream_t s, const float *x, int64_t ldx, int64_t M, int K, unsigned short *hi, unsigned short *lo);
}  // namespace dfb

struct dfb_state {
    int device, sr, fft, hop, nb_erb, min_nb_erb_freqs;
    std::vector<int64_t> erb;
    std::vector<float> window;
    void *d_tables = nullptr;  // one slab holding every table
    dfb::DspTables tb{};
    dfb::Arena arena;          // scratch of the *_host entry points
    cudaStream_t stream = nullptr;
    // STFT / ISTFT memories carried between calls (libDF analysis_mem / synthesis_mem, lib.rs:60-62)
    std::vector<float> analysis_mem, synthesis_mem;
};
