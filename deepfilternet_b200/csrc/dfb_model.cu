// dfb_model.cu -- the DNN of the enhancement path (encoder convs, grouped linears, GRUs, ERB and
// DF decoders) as hand-written sm_100a kernels plus the executor behind dfb_model_* / dfb_enhance.
//
// Reference semantics (paths relative to /root/reference/DeepFilterNet/df):
//   Conv2dNormAct / ConvTranspose2dNormAct   modules.py:18-72, 75-126
//   GroupedLinearEinsum                       modules.py:741-780
//   SqueezedGRU_S / SqueezedGRU               modules.py:702-738 / 663-699  (torch.nn.GRU inside)
//   Encoder / ErbDecoder / DfDecoder          deepfilternet3.py:100-331, deepfilternet2.py:98-371
//   DfNet.forward                             deepfilternet3.py:389-456,   deepfilternet2.py:481-505
//
// HBM layout: every activation is channel-last [B, T, F, C=64] (C fastest) so a 1x1 conv is a
// row-major [rows, 64] x [64, 64] product and depthwise taps are +-64-float neighbours;
// embeddings are [B*T, D] row-major.  BatchNorm is folded on the host (weights.py).
// Arithmetic: IEEE fp32 (FFMA) everywhere; accumulation order differs from ATen's, which is
// inside the 1e-4 RMS parity bound (tests/test_gpu_parity.py).
#include <cooperative_groups.h>
#include <cuda_bf16.h>

#include <cmath>
#include <cstring>
#include <functional>
#include <map>
#include <string>

#include "dfb_common.cuh"
#include "dfb_dwpw.cuh"
#include "dfb_ptx.cuh"

namespace cg = cooperative_groups;

namespace dfb {


enum Act { ACT_NONE = 0, ACT_RELU = 1, ACT_TANH = 2, ACT_SIGMOID = 3 };

__device__ __forceinline__ float act_apply(float x, int act) {
    switch (act) {
        case ACT_RELU: return fmaxf(x, 0.f);
        case ACT_TANH: return tanhf(x);
        case ACT_SIGMOID: return 1.f / (1.f + expf(-x));
        default: return x;
    }
}
__device__ __forceinline__ float sigmoidf_(float x) { return 1.f / (1.f + expf(-x)); }

// ------------------------------------------------------- input convs (erb_conv0, df_conv0) ----
// Dense CIN -> 64 conv, kernel (kt,3), causal in time, BN folded, ReLU.
//   erb_conv0 (CIN = 1): modules.py:18-72 with in_ch = 1 (groups = 1, not separable).
//   df_conv0  (CIN = 2): grouped 2 -> 64 (kt,3) conv followed by the 64 x 64 1x1 conv and BN.  The two
//     linear maps are composed on the host (weights.py): W[dt][df][ri][n] = sum_{c in group ri}
//     dw[dt][df][c] * pw[c][n], so the 64-wide intermediate never exists: 18 instead of 73 MACs per output.
// Feature look-ahead: deepfilternet3.py:359,409-410.
// in  x [B,T,F,CIN]; out [B,T,F,64].  One CTA = kInFrames frames; thread = (f slot, channel quad), taps in registers.
constexpr int kInFrames = 8;
template <int CIN>
__global__ void __launch_bounds__(256)
k_conv_in(const float *__restrict__ x, const float *__restrict__ w /*[kt][3][CIN][64]*/, const float *__restrict__ bias,
          float *__restrict__ out, int T, int F, int kt, int lookahead, int Tsx /* frames per stream in x */,
          int Tx /* feature frames that exist; beyond = end of the stream = zero */,
          int tp_min /* 0: the features are shifted by the look-ahead, then padded causally (DeepFilterNet2 / 3, pad_feat);
                        -lookahead: the conv itself pads (kt-1-la, la) around the unshifted features (DeepFilterNet v1) */) {
    extern __shared__ float s_in[];  // [(kInFrames + kt - 1)][(F + 2) * CIN]
    const int b = blockIdx.y, t0 = blockIdx.x * kInFrames;
    const int rows = kInFrames + kt - 1, ld = (F + 2) * CIN;
    for (int i = threadIdx.x; i < rows * ld; i += blockDim.x) {
        int r = i / ld, j = i - r * ld;
        int f = j / CIN - 1, ci = j - (f + 1) * CIN;
        int tp = t0 - (kt - 1) + r;  // time index in the look-ahead shifted feature sequence
        float v = 0.f;
        if (f >= 0 && f < F && tp >= tp_min && tp + lookahead < Tx) v = x[(((int64_t)b * Tsx + tp + lookahead) * F + f) * CIN + ci];
        s_in[i] = v;
    }
    const int cq = threadIdx.x & 15, fl = threadIdx.x >> 4;  // 16 channel quads x 16 f per pass
    // taps of this thread's channel quad as two packed fp32 pairs: the MACs run as FFMA2 (fma.rn.f32x2, one issue slot for two
    // channels; the scalar version of df_conv0 was issue bound: 69 % of the slots, FMA pipe 49 %)
    unsigned long long wr[9 * CIN][2];
#pragma unroll
    for (int i = 0; i < 9 * CIN; i++) {
        const float4 v = (i >= (3 - kt) * 3 * CIN) ? *reinterpret_cast<const float4 *>(w + (i - (3 - kt) * 3 * CIN) * kCh + cq * 4)
                                                   : make_float4(0.f, 0.f, 0.f, 0.f);
        wr[i][0] = f2_pack(v.x, v.y); wr[i][1] = f2_pack(v.z, v.w);
    }
    const float4 bv = *reinterpret_cast<const float4 *>(bias + cq * 4);
    const unsigned long long b01 = f2_pack(bv.x, bv.y), b23 = f2_pack(bv.z, bv.w);
    __syncthreads();
    for (int fr = 0; fr < kInFrames; fr++) {
        int t = t0 + fr;
        if (t >= T) break;
        for (int f = fl; f < F; f += 16) {
            unsigned long long a01 = b01, a23 = b23;
#pragma unroll
            for (int dt = 0; dt < 3; dt++) {
                if (dt < 3 - kt) continue;
                const float *row = s_in + (fr + dt - (3 - kt)) * ld + f * CIN;  // f-1 .. f+1 -> +0 .. +2
#pragma unroll
                for (int j = 0; j < 3 * CIN; j++) {
                    const float xv = row[j];
                    const unsigned long long xx = f2_pack(xv, xv);
                    a01 = f2_fma(xx, wr[dt * 3 * CIN + j][0], a01);
                    a23 = f2_fma(xx, wr[dt * 3 * CIN + j][1], a23);
                }
            }
            float4 acc;
            f2_unpack(a01, acc.x, acc.y); f2_unpack(a23, acc.z, acc.w);
            acc.x = fmaxf(acc.x, 0.f); acc.y = fmaxf(acc.y, 0.f); acc.z = fmaxf(acc.z, 0.f); acc.w = fmaxf(acc.w, 0.f);
            *reinterpret_cast<float4 *>(out + (((int64_t)b * T + t) * F + f) * kCh + cq * 4) = acc;
        }
    }
}

// ------------------------------------------------- depthwise (+pathway) -> 1x1 -> ReLU ----
// One fused kernel for every "separable" block of the reference (modules.py:49-71, 104-125):
//   prologue  A[r][c] = sum_{dt,df} dw[dt][df][c] * X[t-(kt-1)+dt][fi(fo,df)][c]
//             with X = in (+ relu(path * ps + pb) when a pathway tensor is given; that is
//             `convNp(eN) + prev`, deepfilternet3.py:250-253)
//   GEMM      out[r][n] = relu(sum_c A[r][c] * pw[c][n] + b[n])
// Modes: S1 stride 1, S2 stride 2 (fi = 2 fo + df - 1), T2 transposed stride 2
// (out[2j] = w1 x[j]; out[2j+1] = w2 x[j] + w0 x[j+1]; ConvTranspose2d padding 1, output_padding 1),
// DF0 the grouped 2 -> 64 input conv on the complex features (with look-ahead shift).
// Tile: NF frames x Fout rows (R = NF * Fout <= 128, multiple of 4); thread tile 4 rows x 8 cols.
template <int MODE>
__global__ void __launch_bounds__(256) k_dwpw(DwPwParams p) {
    extern __shared__ __align__(16) float smem[];
    float *Ws = smem;                 // [64][64]
    float *As = smem + kCh * kCh;     // [R][kLdA]
    const int b = blockIdx.y, t0 = blockIdx.x * p.NF;
    const int tid = threadIdx.x;
    const int nf = min(p.NF, p.T - t0);
    const int R = nf * p.Fout;        // rows actually present
    const int Rfull = p.NF * p.Fout;
    for (int i = tid; i < kCh * kCh / 4; i += 256)
        reinterpret_cast<float4 *>(Ws)[i] = reinterpret_cast<const float4 *>(p.pw)[i];
    // ---- prologue: thread = (row slot, channel quad)
    {
        const int cq = tid & 15;
        DwTaps taps;
        dw_load_taps(p, cq, taps);
        for (int r = tid >> 4; r < Rfull; r += 16) {
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
            if (r < R) {
                const int fr = r / p.Fout, fo = r - fr * p.Fout;
                acc = dw_prologue<MODE>(p, taps, b, t0 + fr, fo, cq);
            }
            *reinterpret_cast<float4 *>(As + r * kLdA + cq * 4) = acc;
        }
    }
    __syncthreads();
    // ---- GEMM: thread (rg, cg): rows rg + RG * i (i < 4), cols 8 cg .. 8 cg + 7
    const int RG = Rfull >> 2;
    const int cgid = tid & 7, rg = tid >> 3;
    if (rg >= RG) return;
    float acc[4][8];
#pragma unroll
    for (int i = 0; i < 4; i++)
#pragma unroll
        for (int j = 0; j < 8; j++) acc[i][j] = 0.f;
#pragma unroll 4
    for (int k = 0; k < kCh; k += 4) {
        float4 a[4];
#pragma unroll
        for (int i = 0; i < 4; i++) a[i] = *reinterpret_cast<const float4 *>(As + (rg + RG * i) * kLdA + k);
#pragma unroll
        for (int kk = 0; kk < 4; kk++) {
            float4 w0 = *reinterpret_cast<const float4 *>(Ws + (k + kk) * kCh + cgid * 8);
            float4 w1 = *reinterpret_cast<const float4 *>(Ws + (k + kk) * kCh + cgid * 8 + 4);
#pragma unroll
            for (int i = 0; i < 4; i++) {
                float av = kk == 0 ? a[i].x : kk == 1 ? a[i].y : kk == 2 ? a[i].z : a[i].w;
                acc[i][0] += av * w0.x; acc[i][1] += av * w0.y; acc[i][2] += av * w0.z; acc[i][3] += av * w0.w;
                acc[i][4] += av * w1.x; acc[i][5] += av * w1.y; acc[i][6] += av * w1.z; acc[i][7] += av * w1.w;
            }
        }
    }
    const float4 b0 = *reinterpret_cast<const float4 *>(p.bias + cgid * 8);
    const float4 b1 = *reinterpret_cast<const float4 *>(p.bias + cgid * 8 + 4);
#pragma unroll
    for (int i = 0; i < 4; i++) {
        int r = rg + RG * i;
        if (r >= R) continue;
        int fr = r / p.Fout, fo = r - fr * p.Fout;
        float *dst = p.out + ((int64_t)b * p.T + t0 + fr) * p.out_fs + fo * kCh + cgid * 8;
        float4 o0 = make_float4(fmaxf(acc[i][0] + b0.x, 0.f), fmaxf(acc[i][1] + b0.y, 0.f),
                                fmaxf(acc[i][2] + b0.z, 0.f), fmaxf(acc[i][3] + b0.w, 0.f));
        float4 o1 = make_float4(fmaxf(acc[i][4] + b1.x, 0.f), fmaxf(acc[i][5] + b1.y, 0.f),
                                fmaxf(acc[i][6] + b1.z, 0.f), fmaxf(acc[i][7] + b1.w, 0.f));
        *reinterpret_cast<float4 *>(dst) = o0;
        *reinterpret_cast<float4 *>(dst + 4) = o1;
    }
}

// ------------------------------------------------------------------ grouped linear ----
// Y[m, g*Hg + n] = act( sum_i X[m, g*Ig + i] * W[g][i][n] + bias ) * oscale + ooffset + R[m, ...]
// (GroupedLinearEinsum, modules.py:766-776; G = 1 with bias = GRU input projection W_ih x + b_ih
// with W given as [I][H] i.e. already transposed on upload.)
// CTA tile 64 rows x 64 cols (one group, or a 64-wide slice of a wide group); K chunks of 32.
struct GlParams {
    const float *x; int64_t ldx;
    const float *w;          // [G][Ig][Hg]
    const float *bias;       // [G*Hg] or null
    const float *res; int64_t ldr;  // optional residual, added after the activation
    float *y; int64_t ldy;
    int64_t M;
    int G, Ig, Hg, act;
    float oscale, ooffset;
    unsigned short *y_hi, *y_lo;  // optional BF16 hi/lo planes of y (same pitch): operand of a tcgen05 GEMM
};
constexpr int kGlBM = 64, kGlBN = 64, kGlBK = 32, kGlMaxGpc = 4;

// Narrow groups (Hg = 16 or 32) are packed kGpc = 64 / Hg per CTA so that all 256 threads own real
// output columns (the first version ran one group per CTA: 25 % of the threads active for Hg = 16).
__global__ void __launch_bounds__(256) k_grouped_linear(GlParams p) {
    __shared__ __align__(16) float As[kGlMaxGpc][kGlBM][kGlBK + 4];
    __shared__ __align__(16) float Ws[kGlBK][kGlBN];
    const int gpc = (p.Hg < kGlBN && kGlBN % p.Hg == 0) ? min(kGlBN / p.Hg, p.G) : 1;  // groups per CTA
    const int tiles_per_group = (p.Hg + kGlBN - 1) / kGlBN;                         // > 1 only when gpc == 1
    const int gb = blockIdx.y / tiles_per_group, nt = blockIdx.y - gb * tiles_per_group;
    const int g0 = gb * gpc;                       // first group of this CTA
    const int n0 = nt * kGlBN;                     // column offset inside the group (gpc == 1)
    const int wcols = gpc > 1 ? p.Hg : min(kGlBN, p.Hg - n0);  // valid columns per group in this tile
    const int ngrp = min(gpc, p.G - g0);
    const int64_t m0 = (int64_t)blockIdx.x * kGlBM;
    const int tid = threadIdx.x;
    const int tc = tid & 15, tr = tid >> 4;  // thread tile: rows tr + 16 i, cols 4 tc .. 4 tc + 3
    const int gsub = gpc > 1 ? (tc * 4) / p.Hg : 0;  // which of the CTA's groups this thread's columns belong to
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; i++)
#pragma unroll
        for (int j = 0; j < 4; j++) acc[i][j] = 0.f;
    // loader roles are fixed per thread (no per-element division): A tile -- row ar + 32 i of group ags, k quad akq;
    // W tile -- column quad wn (group wgs, in-group offset wnn), rows wk + 16 i
    const int akq = (tid & 7) * 4, ar = tid >> 3;
    const int wn = (tid & 15) * 4, wk = tid >> 4;
    int wgs = 0, wnn = n0 + wn;
    if (gpc > 1) { wgs = wn / p.Hg; wnn = wn - wgs * p.Hg; }
    const bool wvec = (p.Hg & 3) == 0;                       // a column quad never straddles a group and is 16-byte aligned
    const bool wok = gpc > 1 ? wgs < ngrp : wn < wcols;
    const float *xrow[2];
#pragma unroll
    for (int i = 0; i < 2; i++) {
        const int64_t m = m0 + ar + 32 * i;
        xrow[i] = m < p.M ? p.x + m * p.ldx + (int64_t)g0 * p.Ig + akq : nullptr;
    }
    const float *wbase = p.w + ((int64_t)(g0 + wgs) * p.Ig) * p.Hg + wnn;
    for (int k0 = 0; k0 < p.Ig; k0 += kGlBK) {
        const int kc = min(kGlBK, p.Ig - k0);
        // A tiles: per group 64 rows x 32 k  (8 threads x float4 per row)
        for (int gs = 0; gs < ngrp; gs++) {
#pragma unroll
            for (int i = 0; i < 2; i++) {
                float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                if (xrow[i] && akq < kc) v = *reinterpret_cast<const float4 *>(xrow[i] + gs * p.Ig + k0);
                *reinterpret_cast<float4 *>(&As[gs][ar + 32 * i][akq]) = v;
            }
        }
        // W tile: 32 k x 64 columns (column n -> group n / Hg when several groups share the CTA)
#pragma unroll
        for (int i = 0; i < 2; i++) {
            const int k = wk + 16 * i;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (k < kc && wok) {
                const float *src = wbase + (int64_t)(k0 + k) * p.Hg;
                if (wvec) {
                    if (gpc > 1 || wn + 3 < wcols) v = *reinterpret_cast<const float4 *>(src);
                    else { v.x = src[0]; if (wn + 1 < wcols) v.y = src[1]; if (wn + 2 < wcols) v.z = src[2]; }
                } else {
                    const int lim = gpc > 1 ? p.Hg - wnn : wcols - wn;
                    v.x = src[0]; if (lim > 1) v.y = src[1]; if (lim > 2) v.z = src[2]; if (lim > 3) v.w = src[3];
                }
            }
            *reinterpret_cast<float4 *>(&Ws[k][wn]) = v;
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < kGlBK; k += 4) {
            float4 a[4];
#pragma unroll
            for (int i = 0; i < 4; i++) a[i] = *reinterpret_cast<const float4 *>(&As[gsub][tr + 16 * i][k]);
#pragma unroll
            for (int kk = 0; kk < 4; kk++) {
                float4 w = *reinterpret_cast<const float4 *>(&Ws[k + kk][tc * 4]);
#pragma unroll
                for (int i = 0; i < 4; i++) {
                    float av = kk == 0 ? a[i].x : kk == 1 ? a[i].y : kk == 2 ? a[i].z : a[i].w;
                    acc[i][0] += av * w.x; acc[i][1] += av * w.y; acc[i][2] += av * w.z; acc[i][3] += av * w.w;
                }
            }
        }
        __syncthreads();
    }
    // columns of this thread: group g0 + gsub, inside-group offset nn0 .. nn0 + 3
    const int nn0 = gpc > 1 ? tc * 4 - gsub * p.Hg : n0 + tc * 4;
    if (gsub >= ngrp) return;
    const int colbase = (g0 + gsub) * p.Hg + nn0;
    const int nvalid = min(4, p.Hg - nn0);  // <= 0 when the thread's columns are past the group end
#pragma unroll
    for (int i = 0; i < 4; i++) {
        int64_t m = m0 + tr + 16 * i;
        if (m >= p.M || nvalid <= 0) continue;
        float v[4];
#pragma unroll
        for (int j = 0; j < 4; j++) {
            v[j] = acc[i][j];
            if (j < nvalid) {
                const int col = colbase + j;
                if (p.bias) v[j] += p.bias[col];
                v[j] = act_apply(v[j], p.act) * p.oscale + p.ooffset;
                if (p.res) v[j] += p.res[m * p.ldr + col];
            }
        }
        float *dst = p.y + m * p.ldy + colbase;
        if (nvalid == 4 && (((uintptr_t)dst) & 15) == 0) {
            *reinterpret_cast<float4 *>(dst) = make_float4(v[0], v[1], v[2], v[3]);
        } else {
            for (int j = 0; j < nvalid; j++) dst[j] = v[j];
        }
        if (p.y_hi) {
            unsigned short hi[4], lo[4];
#pragma unroll
            for (int j = 0; j < 4; j++) {
                __nv_bfloat16 hb = __float2bfloat16_rn(v[j]);
                hi[j] = __bfloat16_as_ushort(hb);
                lo[j] = __bfloat16_as_ushort(__float2bfloat16_rn(v[j] - __bfloat162float(hb)));
            }
            unsigned short *dh = p.y_hi + m * p.ldy + colbase, *dl = p.y_lo + m * p.ldy + colbase;
            if (nvalid == 4 && (((uintptr_t)dh) & 7) == 0) {
                *reinterpret_cast<uint2 *>(dh) = make_uint2(hi[0] | (uint32_t)hi[1] << 16, hi[2] | (uint32_t)hi[3] << 16);
                *reinterpret_cast<uint2 *>(dl) = make_uint2(lo[0] | (uint32_t)lo[1] << 16, lo[2] | (uint32_t)lo[3] << 16);
            } else {
                for (int j = 0; j < nvalid; j++) { dh[j] = hi[j]; dl[j] = lo[j]; }
            }
        }
    }
}

// ------------------------------------------------------------------- GRU recurrence ----
// torch.nn.GRU cell (gate order r, z, n; modules.py:684,723):
//   r = s(xr + Whr h + bhr), z = s(xz + Whz h + bhz), n = tanh(xn + r (Whn h + bhn)), h' = (1-z) n + z h
// xproj = W_ih x + b_ih comes from k_grouped_linear.  One thread-block CLUSTER owns a group of Bc
// streams for the whole sequence: CTA `rank` keeps the W_hh rows of its U = H / C hidden units
// (3U rows x H) in REGISTERS: 384 threads, each an 8-row x 16-k tile (128 weights), so a thread
// reads only 16 h values per stream and step from shared memory; the H/16 lanes that share a row
// group combine their partial sums with a shuffle reduce-scatter.  The hidden state of the group
// lives in shared memory of every CTA (double buffered); the new slice is broadcast with st.async
// DSMEM stores that complete bytes on the receiver's mbarrier, so a step needs neither a cluster
// barrier nor a memory fence (ncu on the first version: membar was the top stall, the release
// fence of cluster.sync() waited for the global h stores).  H = 256: C = 4, U = 64;  H = 512: C = 16, U = 32.
constexpr int kGruThreads = 384, kGruRT = 8, kGruKT = 16, kGruSB = 4, kGruMaxBc = 16;

// packed fp32x2 FMA (Blackwell FFMA2): d = a * b + c on both halves; a scalar b is broadcast by the
// compiler through the .F32 operand form, so a pair of W rows costs one issue slot per (k, stream)
__device__ __forceinline__ unsigned long long gru_pack2(float lo, float hi) {
    unsigned long long r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void gru_unpack2(unsigned long long v, float &lo, float &hi) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ unsigned long long gru_ffma2(unsigned long long a, unsigned long long b, unsigned long long c) {
    unsigned long long d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}
__device__ __forceinline__ uint32_t gru_smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint32_t gru_mapa(uint32_t saddr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(rank));
    return r;
}
// remote (DSMEM) store that completes `4` bytes on the destination CTA's mbarrier: no fence or
// cluster barrier is needed on the consumer side, it just waits for the expected byte count
__device__ __forceinline__ void gru_st_async(uint32_t dst, float v, uint32_t mbar) {
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.b32 [%0], %1, [%2];" ::"r"(dst),
                 "r"(__float_as_uint(v)), "r"(mbar)
                 : "memory");
}
__device__ __forceinline__ void gru_mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(gru_smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void gru_mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(gru_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void gru_mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t"
        "}\n" ::"r"(gru_smem_u32(bar)),
        "r"(parity)
        : "memory");
}

struct GruParams {
    const float *xproj;  // [B,T,3H]
    const float *whh;    // [3H][H]
    const float *bhh;    // [3H]
    const float *res;    // optional [B,T,H] added to the OUTPUT only (identity skip, modules.py:696)
    float *hout;         // [B,T,H]
    int B, T, Bc;
    long long *dbg;      // optional [T][8] clock64 phase stamps of CTA 0 (dfb_debug_gru_timing)
    // time-chunked execution (see GruWindow): frames t0 + t of buffers with Ts frames per stream, carried state h0 -> hT
    const float *h0;
    float *hT;
    int t0, Ts;
};

template <int H, int C>
__global__ void __launch_bounds__(kGruThreads, 1) k_gru(GruParams p) {
    constexpr int U = H / C;                       // hidden units per CTA
    constexpr int LPR = H / kGruKT;                // lanes sharing one row group (16 or 32)
    constexpr int NRG = 3 * U / kGruRT;            // row groups per CTA
    static_assert(NRG * LPR == kGruThreads, "layout");
    constexpr int V = kGruRT * kGruSB;             // partial sums per thread and stream chunk (32)
    constexpr int VF = V / LPR;                    // fully reduced values a lane ends up with
    constexpr int HP = H + 4;                      // padded h row
    cg::cluster_group cluster = cg::this_cluster();
    const int rank = (int)cluster.block_rank();
    const int group = blockIdx.x / C;
    const int b0 = group * p.Bc;
    const int nb = min(p.Bc, p.B - b0);
    extern __shared__ __align__(16) float gru_smem[];
    float (*s_h)[kGruMaxBc][HP] = reinterpret_cast<float (*)[kGruMaxBc][HP]>(gru_smem);            // [2][Bc][HP]
    float (*s_pre)[kGruMaxBc + 1] = reinterpret_cast<float (*)[kGruMaxBc + 1]>(gru_smem + 2 * kGruMaxBc * HP);  // [3U]
    __shared__ __align__(8) uint64_t s_bar[2];     // s_bar[b]: all of h for buffer b has arrived
    const int tid = threadIdx.x;
    const int rg = tid / LPR, kl = tid % LPR;      // row group, k slice [16 kl, 16 kl + 16)
    // weights -> registers as row pairs: w2[rp][k] = (Whh[row(2 rp)][16 kl + k], Whh[row(2 rp + 1)][16 kl + k])
    unsigned long long w2[kGruRT / 2][kGruKT];
#pragma unroll
    for (int rp = 0; rp < kGruRT / 2; rp++) {
        const int row0 = rg * kGruRT + 2 * rp, row1 = row0 + 1;  // row in [0, 3U): gate = row / U, unit = row % U
        const float *s0 = p.whh + ((int64_t)(row0 / U) * H + rank * U + (row0 % U)) * H + kl * kGruKT;
        const float *s1 = p.whh + ((int64_t)(row1 / U) * H + rank * U + (row1 % U)) * H + kl * kGruKT;
#pragma unroll
        for (int k = 0; k < kGruKT; k += 4) {
            float4 a = *reinterpret_cast<const float4 *>(s0 + k), c = *reinterpret_cast<const float4 *>(s1 + k);
            w2[rp][k] = gru_pack2(a.x, c.x); w2[rp][k + 1] = gru_pack2(a.y, c.y);
            w2[rp][k + 2] = gru_pack2(a.z, c.z); w2[rp][k + 3] = gru_pack2(a.w, c.w);
        }
    }
    // index of the first fully reduced value this lane owns after the reduce-scatter
    int vbase = 0;
#pragma unroll
    for (int bit = LPR / 2, n = V / 2; bit >= 1 && n >= 1; bit >>= 1, n >>= 1)
        if (kl & bit) vbase += n;
    for (int i = tid; i < 2 * kGruMaxBc * HP; i += kGruThreads) gru_smem[i] = 0.f;  // h0 = 0
    if (p.h0) {  // carried state (every CTA of the cluster keeps the whole h of its streams)
        __syncthreads();
        for (int i = tid; i < nb * H; i += kGruThreads) {
            const int s = i / H, gu = i - s * H;
            s_h[0][s][(((gu % kGruKT) / 4) * LPR + gu / kGruKT) * 4 + (gu & 3)] = p.h0[(int64_t)(b0 + s) * H + gu];
        }
    }
    // gate-phase items (s, u): this thread's slots
    constexpr int kItems = (kGruMaxBc * U + kGruThreads - 1) / kGruThreads;
    float bh[kItems][3];
#pragma unroll
    for (int it = 0; it < kItems; it++) {
        int item = tid + it * kGruThreads;
        int u = item % U;
        bh[it][0] = p.bhh[rank * U + u]; bh[it][1] = p.bhh[H + rank * U + u]; bh[it][2] = p.bhh[2 * H + rank * U + u];
    }
    if (tid == 0) {
        gru_mbar_init(&s_bar[0], 1);
        gru_mbar_init(&s_bar[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    cluster.sync();  // barriers initialised and h0 = 0 visible before any remote store can arrive
    const uint32_t bar_local[2] = {gru_smem_u32(&s_bar[0]), gru_smem_u32(&s_bar[1])};
    const uint32_t step_bytes = (uint32_t)(H * nb * 4);
    int cur = 0;
    for (int t = 0; t < p.T; t++) {
        // arm the barrier of the other buffer for the h_{t+1} bytes, then wait for h_t
        if (tid == 0 && t + 1 < p.T) gru_mbar_expect_tx(&s_bar[cur ^ 1], step_bytes);
        const bool dbg_on = p.dbg && blockIdx.x == 0 && tid == 0;
        if (dbg_on) p.dbg[t * 8 + 0] = clock64();
        if (t > 0) gru_mbar_wait(&s_bar[cur], (uint32_t)(((t - 1) >> 1) & 1));
        if (dbg_on) p.dbg[t * 8 + 1] = clock64();
        // prefetch the input projections of this step for the gate phase (independent of h)
        float xr[kItems][3];
#pragma unroll
        for (int it = 0; it < kItems; it++) {
            int item = tid + it * kGruThreads;
            if (item < nb * U) {
                int s = item / U, u = item - s * U;
                const float *xp = p.xproj + ((int64_t)(b0 + s) * p.Ts + p.t0 + t) * (3 * H) + rank * U + u;
                xr[it][0] = xp[0]; xr[it][1] = xp[H]; xr[it][2] = xp[2 * H];
            }
        }
        // matvec: pre[row][s] = sum_k W[row][k] h[s][k]
        for (int sc = 0; sc < nb; sc += kGruSB) {
            unsigned long long acc2[kGruRT / 2][kGruSB];
#pragma unroll
            for (int rp = 0; rp < kGruRT / 2; rp++)
#pragma unroll
                for (int s = 0; s < kGruSB; s++) acc2[rp][s] = 0ull;
#pragma unroll
            for (int s = 0; s < kGruSB; s++) {
                // h is stored permuted (hpos) so that the LPR lanes read consecutive float4s
                const float *hb = &s_h[cur][sc + s][kl * 4];
#pragma unroll
                for (int k = 0; k < kGruKT; k += 4) {
                    float4 hv = *reinterpret_cast<const float4 *>(hb + (k / 4) * LPR * 4);
                    const unsigned long long h0 = gru_pack2(hv.x, hv.x), h1 = gru_pack2(hv.y, hv.y),
                                             h2 = gru_pack2(hv.z, hv.z), h3 = gru_pack2(hv.w, hv.w);
#pragma unroll
                    for (int rp = 0; rp < kGruRT / 2; rp++) {
                        unsigned long long a = acc2[rp][s];
                        a = gru_ffma2(w2[rp][k], h0, a); a = gru_ffma2(w2[rp][k + 1], h1, a);
                        a = gru_ffma2(w2[rp][k + 2], h2, a); a = gru_ffma2(w2[rp][k + 3], h3, a);
                        acc2[rp][s] = a;
                    }
                }
            }
            float acc[V];
#pragma unroll
            for (int rp = 0; rp < kGruRT / 2; rp++)
#pragma unroll
                for (int s = 0; s < kGruSB; s++)
                    gru_unpack2(acc2[rp][s], acc[(2 * rp) * kGruSB + s], acc[(2 * rp + 1) * kGruSB + s]);
            if (dbg_on && sc == 0) p.dbg[t * 8 + 2] = clock64();
            // reduce-scatter over the LPR lanes of this row group
#pragma unroll
            for (int bit = LPR / 2, n = V / 2; bit >= 1 && n >= 1; bit >>= 1, n >>= 1) {
                const bool up = (kl & bit) != 0;
#pragma unroll
                for (int i = 0; i < V / 2; i++) {
                    if (i < n) {
                        float send = up ? acc[i] : acc[i + n];
                        float keep = up ? acc[i + n] : acc[i];
                        acc[i] = keep + __shfl_xor_sync(0xffffffffu, send, bit);
                    }
                }
            }
#pragma unroll
            for (int i = 0; i < VF; i++) {
                int v = vbase + i;                      // v = r * kGruSB + s
                int r = v / kGruSB, s = v % kGruSB;
                if (sc + s < nb) s_pre[rg * kGruRT + r][sc + s] = acc[i];
            }
        }
        if (dbg_on) p.dbg[t * 8 + 3] = clock64();
        __syncthreads();
        if (dbg_on) p.dbg[t * 8 + 4] = clock64();
        // gates
#pragma unroll
        for (int it = 0; it < kItems; it++) {
            int item = tid + it * kGruThreads;
            if (item < nb * U) {
                int s = item / U, u = item - s * U;
                int gu = rank * U + u;
                float r = sigmoidf_(xr[it][0] + s_pre[u][s] + bh[it][0]);
                float z = sigmoidf_(xr[it][1] + s_pre[U + u][s] + bh[it][1]);
                float n = tanhf(xr[it][2] + r * (s_pre[2 * U + u][s] + bh[it][2]));
                const int hp = (((gu % kGruKT) / 4) * LPR + gu / kGruKT) * 4 + (gu & 3);  // hpos(gu)
                float hprev = s_h[cur][s][hp];
                float hn = (1.f - z) * n + z * hprev;
                int64_t o = ((int64_t)(b0 + s) * p.Ts + p.t0 + t) * H + gu;
                p.hout[o] = p.res ? hn + p.res[o] : hn;
                if (p.hT && t + 1 == p.T) p.hT[(int64_t)(b0 + s) * H + gu] = hn;
                if (t + 1 < p.T) {
                    // broadcast the new value to every CTA of the cluster (st.async DSMEM store)
                    const uint32_t dst_local = gru_smem_u32(&s_h[cur ^ 1][s][hp]);
#pragma unroll
                    for (int c = 0; c < C; c++) gru_st_async(gru_mapa(dst_local, c), hn, gru_mapa(bar_local[cur ^ 1], c));
                }
            }
        }
        if (dbg_on) p.dbg[t * 8 + 5] = clock64();
        // no CTA barrier here: s_pre is rewritten by the next step's matvec only after the mbarrier
        // wait at the top of the loop, which needs every gate thread's sends (issued after its reads)
        cur ^= 1;
    }
    cluster.sync();  // no CTA exits while peers may still address its shared memory
}

// --------------------------------------------------------------- ERB mask output conv ----
// m[b,t,f] = sigmoid( sum_{dt,df,c} w[dt][df][c] * X[t-(kt-1)+dt][f+df-1][c] + bias ),
// X = relu(e0 * ps + pb) + d1   (conv0_out(conv0p(e0) + e1), deepfilternet3.py:253).
// One warp walks kMaskChunk consecutive frames of one stream; X rows of the current and the
// previous frame are staged in shared memory ([E+2][65] floats, zero rows at f = -1, E).
constexpr int kMaskWarps = 4, kMaskChunk = 8, kMaskLd = kCh + 1;
__global__ void __launch_bounds__(32 * kMaskWarps)
k_mask_out(const float *__restrict__ e0, const float *__restrict__ d1, const float *__restrict__ ps,
           const float *__restrict__ pb, const float *__restrict__ w /*[kt][3][64]*/,
           const float *__restrict__ bias_p, float *__restrict__ m, int T, int E, int kt) {
    extern __shared__ float smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int b = blockIdx.y;
    const int t0 = (blockIdx.x * kMaskWarps + warp) * kMaskChunk;
    float *buf = smem + warp * 2 * (E + 2) * kMaskLd;  // two frames
    float *ws = smem + kMaskWarps * 2 * (E + 2) * kMaskLd;  // [kt*3*64] shared by all warps
    for (int i = threadIdx.x; i < kt * 3 * kCh; i += blockDim.x) ws[i] = w[i];
    for (int i = lane; i < 2 * (E + 2) * kMaskLd; i += 32) buf[i] = 0.f;
    __syncthreads();
    if (t0 >= T) return;
    const int t1 = min(t0 + kMaskChunk, T);
    const float2 ps2 = *reinterpret_cast<const float2 *>(ps + lane * 2);
    const float2 pb2 = *reinterpret_cast<const float2 *>(pb + lane * 2);
    const float bias = bias_p[0];
    for (int t = (kt > 1 && t0 > 0) ? t0 - 1 : t0; t < t1; t++) {
        float *cur = buf + (t & 1) * (E + 2) * kMaskLd;
        const float *prv = buf + ((t & 1) ^ 1) * (E + 2) * kMaskLd;
        const int64_t base = ((int64_t)b * T + t) * E * kCh;
        for (int f = 0; f < E; f++) {
            float2 e = *reinterpret_cast<const float2 *>(e0 + base + f * kCh + lane * 2);
            float2 d = *reinterpret_cast<const float2 *>(d1 + base + f * kCh + lane * 2);
            cur[(f + 1) * kMaskLd + lane * 2] = fmaxf(e.x * ps2.x + pb2.x, 0.f) + d.x;
            cur[(f + 1) * kMaskLd + lane * 2 + 1] = fmaxf(e.y * ps2.y + pb2.y, 0.f) + d.y;
        }
        __syncwarp();
        if (t >= t0) {
            for (int f = lane; f < E; f += 32) {
                float acc = bias;
                for (int dt = 0; dt < kt; dt++) {
                    // dt = kt-1 is the current frame; dt = kt-2 the previous one (kt <= 2)
                    const float *src = (dt == kt - 1) ? cur : prv;
                    if (dt != kt - 1 && t == 0) continue;
                    for (int df = 0; df < 3; df++) {
                        const float *xr = src + (f + df) * kMaskLd;
                        const float *wr = ws + (dt * 3 + df) * kCh;
#pragma unroll 16
                        for (int c = 0; c < kCh; c++) acc += xr[c] * wr[c];
                    }
                }
                m[((int64_t)b * T + t) * E + f] = sigmoidf_(acc);
            }
        }
        __syncwarp();
    }
}

// ------------------------------------------------- DeepFilterNet v1: gather-sum, pathway 1x1 ----
// out[m][k] = act( sum_i src_i[m][idx_i[k]] ), optionally also as BF16 hi / lo planes.  DeepFilterNet v1 flattens channel-major
// into its grouped layers and interleaves ("shuffles") their outputs (deepfilternet.py:135-139,183-185; modules.py:651-654,
// 807-812) while the device tensors are channel-last: every such re-ordering, and the sum over the GRU layers' outputs
// (add_outputs, modules.py:655-656), is one pass of this kernel with host-built index tables (weights.py: v1.idx_*).
struct GatherParams {
    const float *src[3]; long long ld[3]; const int *idx[3]; int n;
    float *out; long long ldo;
    unsigned short *hi, *lo; long long ldp;
    int K, relu;
};
__global__ void __launch_bounds__(256) k_gather_sum(GatherParams p) {
    const long long m = blockIdx.x;
    for (int k = threadIdx.x; k < p.K; k += 256) {
        float v = 0.f;
#pragma unroll
        for (int i = 0; i < 3; i++)
            if (i < p.n) v += p.src[i][m * p.ld[i] + p.idx[i][k]];
        if (p.relu) v = fmaxf(v, 0.f);
        if (p.out) p.out[m * p.ldo + k] = v;
        if (p.hi) {
            unsigned short h, l;
            bf16_split(v, h, l);
            p.hi[m * p.ldp + k] = h; p.lo[m * p.ldp + k] = l;
        }
    }
}

// coefs[r][k] = tanh(coefs[r][k]) + relu(sum_c c0[r][c] w[c][k] + b[k]),  r = (b, t, f), k < 2 O: the dense 1x1 pathway conv
// df_convp (deepfilternet.py:210-212) on top of the df_fc_out pre-activations already in `coefs` (deepfilternet.py:224-228)
template <int O2>
__global__ void __launch_bounds__(128) k_convp_v1(const float *__restrict__ c0, const float *__restrict__ w /*[64][O2]*/,
                                                   const float *__restrict__ bias, float *__restrict__ coefs, long long rows) {
    __shared__ float ws[kCh * O2];
    __shared__ float bs[O2];
    for (int i = threadIdx.x; i < kCh * O2; i += 128) ws[i] = w[i];
    if (threadIdx.x < O2) bs[threadIdx.x] = bias[threadIdx.x];
    __syncthreads();
    const long long r = (long long)blockIdx.x * 128 + threadIdx.x;
    if (r >= rows) return;
    float acc[O2];
#pragma unroll
    for (int k = 0; k < O2; k++) acc[k] = bs[k];
    const float4 *x = reinterpret_cast<const float4 *>(c0 + r * kCh);
#pragma unroll 4
    for (int q = 0; q < kCh / 4; q++) {
        const float4 v = x[q];
#pragma unroll
        for (int k = 0; k < O2; k++)
            acc[k] += v.x * ws[(4 * q) * O2 + k] + v.y * ws[(4 * q + 1) * O2 + k] + v.z * ws[(4 * q + 2) * O2 + k] + v.w * ws[(4 * q + 3) * O2 + k];
    }
    float *o = coefs + r * O2;
#pragma unroll
    for (int k = 0; k < O2; k++) o[k] = tanhf(o[k]) + fmaxf(acc[k], 0.f);
}

// ------------------------------------------------- DF pathway conv ----
// coefs[b,t,f,:] = relu( pw( conv_t(c0) ) + b ); the df_out projection later adds tanh(df_out(c)) on top
// (deepfilternet3.py:293-295, 328-330).  df_convp = grouped (2) temporal conv C -> 2*O with kernel (ktp,1),
// 1x1 conv, BN, ReLU.
// A warp owns two adjacent frequency bins and marches along t: the 512 contiguous bytes of c0 it needs per frame arrive
// by one TMA bulk copy into a per-warp ring of kCpSlots slots (armed kCpSlots frames ahead: ~10 KB in flight per warp,
// 120 KB per SM -- the first version prefetched five frames through registers, ~30 KB per SM, and sat at 0.30 of the HBM
// roofline with 12 % occupancy), lane q reads channel quad q of its bin from the slot, keeps its 4 channels' taps for
// all (dt, o) in registers for the whole kernel, and accumulates the ktp in-flight output frames in rotating registers.
// A finished frame is reduced over the 8 lanes of its channel group with shuffles, the two groups are exchanged, and
// lanes 0..2*O-1 apply the 1x1 conv + bias + ReLU and store 40 contiguous bytes.
constexpr int kMaxO2 = 16, kCpWarps = 4, kCpChunk = 128, kCpSlots = 20;
template <int ORDER, int KTP, int MINB>
__global__ void __launch_bounds__(32 * kCpWarps, MINB)
k_df_convp(const float *__restrict__ c0 /*[B,T,Fd,64]*/, const float *__restrict__ w1 /*[ktp][O2][32]*/,
           const float *__restrict__ w2 /*[O2][O2]*/, const float *__restrict__ bias, float *__restrict__ coefs,
           int T, int Fd) {
    static_assert(kCpSlots % KTP == 0, "a group of KTP frames must not wrap around the ring");
    constexpr int O2 = 2 * ORDER, CG = kCh / 2;
    extern __shared__ __align__(128) unsigned char cp_smem[];   // [warp][slot][512 B] | [warp][slot] mbarriers
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int q = lane & 15, g = q >> 3, cq = q & 7;
    const int f0 = (blockIdx.x * kCpWarps + warp) * 2;        // the warp's first bin (Fd is even: both bins exist or none)
    const bool f_ok = f0 + 1 < Fd;
    const int f = f0 + (lane >> 4);
    const int b = blockIdx.z;
    const int t_begin = blockIdx.y * kCpChunk, t_end = min(T, t_begin + kCpChunk);
    float4 wv[KTP][ORDER];
#pragma unroll
    for (int dt = 0; dt < KTP; dt++)
#pragma unroll
        for (int o = 0; o < ORDER; o++)
            wv[dt][o] = __ldg(reinterpret_cast<const float4 *>(w1 + (dt * O2 + g * ORDER + o) * CG + 4 * cq));
    __shared__ float s_w2[O2 * O2 + O2];  // 1x1 conv | bias; lane q < O2 applies column q
    for (int i = threadIdx.x; i < O2 * O2; i += blockDim.x) s_w2[i] = w2[i];
    if (threadIdx.x < O2) s_w2[O2 * O2 + threadIdx.x] = bias[threadIdx.x];
    const uint32_t ring = smem_u32(cp_smem) + (uint32_t)warp * kCpSlots * 512u;
    const uint32_t bars = smem_u32(cp_smem) + (uint32_t)kCpWarps * kCpSlots * 512u + (uint32_t)warp * kCpSlots * 8u;
    if (lane == 0) {
        for (int i = 0; i < kCpSlots; i++) mbar_init_a(bars + 8 * i, 1);
        fence_barrier_init();
    }
    __syncthreads();
    if (!f_ok) return;
    const float *s2c = s_w2 + (q < O2 ? q : 0);
    float acc[KTP][ORDER];
#pragma unroll
    for (int u = 0; u < KTP; u++)
#pragma unroll
        for (int o = 0; o < ORDER; o++) acc[u][o] = 0.f;
    const float *src0 = c0 + ((int64_t)b * T * Fd + f0) * kCh;   // frame 0 of the warp's two bins (512 contiguous bytes per frame)
    const int64_t fs = (int64_t)Fd * kCh;
    const int tstart = t_begin - (KTP - 1);
    // frame tp lives in slot (tp - tstart) % kCpSlots; frames before the stream start are zeros and never loaded
    auto arm = [&](int tp) {
        const uint32_t slot = (uint32_t)((tp - tstart) % kCpSlots);
        if (tp >= 0 && tp < t_end) {
            mbar_expect_tx_a(bars + 8 * slot, 512);
            bulk_load(ring + slot * 512u, src0 + (int64_t)tp * fs, 512, bars + 8 * slot);
        } else if (tp < 0) {
            mbar_arrive_a(bars + 8 * slot);   // nothing to load: still complete the phase so that the slot's parity stays in step
        }
    };
    if (lane == 0)
        for (int i = 0; i < kCpSlots; i++) arm(tstart + i);
    __syncwarp();
    for (int tb = tstart; tb < t_end; tb += KTP) {
        const uint32_t slot0 = (uint32_t)((tb - tstart) % kCpSlots), parity = (uint32_t)(((tb - tstart) / kCpSlots) & 1);
        float4 x[KTP];
#pragma unroll
        for (int u = 0; u < KTP; u++) {
            const int tp = tb + u;
            if (tp >= 0 && tp < t_end) {
                mbar_wait_a(bars + 8 * (slot0 + u), parity);
                x[u] = lds128(ring + (slot0 + u) * 512u + lane * 16u);
            } else {
                x[u] = make_float4(0.f, 0.f, 0.f, 0.f);
            }
        }
        __syncwarp();                       // every lane has its values: the slots may be refilled
        if (lane == 0)
#pragma unroll
            for (int u = 0; u < KTP; u++) arm(tb + u + kCpSlots);
#pragma unroll
        for (int u = 0; u < KTP; u++) {
            const int tp = tb + u;
            // input frame tp feeds output frame tp + (KTP-1) - dt through tap dt; slot = output frame mod KTP
#pragma unroll
            for (int dt = 0; dt < KTP; dt++) {
                const int slot = (u + KTP - 1 - dt) % KTP;
#pragma unroll
                for (int o = 0; o < ORDER; o++) {
                    const float4 ww = wv[dt][o];
                    float a = dt == 0 ? 0.f : acc[slot][o];
                    a = fmaf(x[u].x, ww.x, a); a = fmaf(x[u].y, ww.y, a);
                    a = fmaf(x[u].z, ww.z, a); a = fmaf(x[u].w, ww.w, a);
                    acc[slot][o] = a;
                }
            }
            if (tp >= t_begin && tp < t_end) {  // output frame tp (slot u) is complete; warp-uniform condition
                float v[ORDER], w[ORDER];
#pragma unroll
                for (int o = 0; o < ORDER; o++) {
                    float r = acc[u][o];
                    r += __shfl_xor_sync(0xffffffffu, r, 1);
                    r += __shfl_xor_sync(0xffffffffu, r, 2);
                    r += __shfl_xor_sync(0xffffffffu, r, 4);
                    v[o] = r;
                    w[o] = __shfl_xor_sync(0xffffffffu, r, 8);  // the other channel group's sums
                }
                float out = s2c[O2 * O2];
#pragma unroll
                for (int k = 0; k < ORDER; k++) out = fmaf(g ? w[k] : v[k], s2c[k * O2], out);
#pragma unroll
                for (int k = 0; k < ORDER; k++) out = fmaf(g ? v[k] : w[k], s2c[(ORDER + k) * O2], out);
                if (q < O2) coefs[(((int64_t)b * T + tp) * Fd + f) * O2 + q] = fmaxf(out, 0.f);
            }
        }
    }
}

}  // namespace dfb

// =========================================================================== executor =====
using namespace dfb;


struct GruLayerW { const float *w_ih_t, *w_hh, *b_ih, *b_hh; int in_dim; };
// carried hidden states of one GRU stack between time chunks: h = [layers][B][H]; t0 = first frame the recurrences run
struct GruChunk { float *h; bool have_state; int t0; };

struct dfb_model {
    int device;
    dfb_model_config cfg;
    std::map<std::string, std::pair<float *, int64_t>> t;  // device tensors
    std::map<std::string, std::pair<const float *, int64_t>> dbg;  // activations of the last forward
    std::vector<GruLayerW> enc_gru, erb_gru, df_gru;
    float *slab = nullptr;
    int conv_tc = 0; // 1: 1x1 convs of the separable blocks on the BF16x3 tcgen05 path
    int proj_tc = 0; // 1: GRU input projections on the BF16x3 tcgen05 GEMM (needs gru_tc)
    int gru_tc = 0;  // 1: tensor-core recurrence (BF16 hi/lo split operands) for H = 256
    long long *gru_dbg = nullptr;  // device buffer for dfb_debug_gru_timing
    Arena arena;
    int dev_chunks = 0, host_chunks = 4, n_lanes = 2;   // chunk pipeline (dfb_model_set_chunking); dev_chunks 0 = auto
    int post_filter = 0, mask_only = 0;       // optional stages (dfb_model_set_options)
    float pf_beta = 0.02f;
    size_t max_workspace = size_t(64) << 30;  // dfb_enhance chunks / groups the batch so that the arena stays below this
    std::vector<int64_t> erb_widths;          // band table the model was built for (checked against the dfb_state)
    Arena aux_arena;                          // carried stream state + padded input of dfb_enhance
    cudaStream_t stream = nullptr;
    cudaStream_t h2d = nullptr, d2h = nullptr;  // copy streams of dfb_enhance_host (both copy engines next to the compute)
    // One forward pass hops from the caller's stream onto the lane's internal streams: `hi` (ERB branch) and `aux` (DF
    // branch) for the encoder phase, `dhi` / `daux` at the greatest priority for the decoder phase (the recurrences are
    // the critical chain), `low` (least priority) for work off the critical path that only fills idle SMs.  Two lanes:
    // consecutive time chunks alternate between them, so that the encoder phase of chunk c + 1 overlaps the decoder
    // phase of chunk c (lane 1 has its own arena; everything outside the chunk loop uses lane 0).
    struct Lane {
        cudaStream_t main = nullptr, hi = nullptr, aux = nullptr, dhi = nullptr, daux = nullptr, low = nullptr;
        cudaEvent_t ev_fork = nullptr, ev_join = nullptr, ev_fork_enc = nullptr, ev_join_enc = nullptr, ev_in = nullptr,
                    ev_out = nullptr, ev_c0 = nullptr, ev_convp = nullptr, ev_skip = nullptr, ev_done = nullptr;
    } lanes[2];
    Arena arena1;                           // lane 1's activations (lane 0 uses `arena`)
    const float *get(const std::string &n) const {
        auto it = t.find(n);
        return it == t.end() ? nullptr : it->second.first;
    }
};

static int need(const dfb_model *m, const char *name, int64_t numel, const float **out) {
    auto it = m->t.find(name);
    if (it == m->t.end()) return fail(DFB_ERR_INVALID, "missing weight tensor '%s'", name);
    if (numel >= 0 && it->second.second != numel)
        return fail(DFB_ERR_INVALID, "weight tensor '%s' has %lld elements, expected %lld", name,
                    (long long)it->second.second, (long long)numel);
    *out = it->second.first;
    return DFB_OK;
}

extern "C" int dfb_model_create(dfb_model **out, int device, const dfb_model_config *cfg, const dfb_tensor *tensors,
                                int n_tensors, const int64_t *erb_widths) {
    if (!out || !cfg || !tensors) return fail(DFB_ERR_INVALID, "null argument");
    *out = nullptr;
    if (cfg->conv_ch != kCh) return fail(DFB_ERR_UNSUPPORTED, "conv_ch = %d (built kernels: 64)", cfg->conv_ch);
    if (cfg->model_kind < 1 || cfg->model_kind > 3) return fail(DFB_ERR_UNSUPPORTED, "model_kind %d", cfg->model_kind);
    if (cfg->model_kind == 1 && (cfg->emb_hidden != cfg->df_hidden || cfg->emb_hidden != cfg->nb_erb / 4 * kCh || cfg->conv_kt != 2 ||
                                 cfg->inp_kt != 2 || cfg->df_order != 5))
        return fail(DFB_ERR_UNSUPPORTED, "DeepFilterNet v1: only the shipped topology is built (hidden = conv_ch * nb_erb / 4, kt 2, order 5)");
    if (cfg->conv_kt < 1 || cfg->conv_kt > 2 || cfg->inp_kt < 1 || cfg->inp_kt > 3)
        return fail(DFB_ERR_UNSUPPORTED, "conv kernel time taps (%d, %d) unsupported", cfg->conv_kt, cfg->inp_kt);
    if ((cfg->emb_hidden != 256 && cfg->emb_hidden != 512) || (cfg->df_hidden != 256 && cfg->df_hidden != 512))
        return fail(DFB_ERR_UNSUPPORTED, "GRU hidden sizes (%d, %d): built kernels cover 256 and 512", cfg->emb_hidden,
                    cfg->df_hidden);
    if (cfg->nb_erb % 8 || cfg->nb_erb > 64 || cfg->nb_df % 8 || cfg->nb_df > 128 || 2 * cfg->df_order > kMaxO2)
        return fail(DFB_ERR_UNSUPPORTED, "nb_erb / nb_df / df_order outside the built kernels");
    int rc = use_device(device);
    if (rc) return rc;
    dfb_model *m = new dfb_model();
    m->device = device;
    m->cfg = *cfg;
    if (erb_widths) m->erb_widths.assign(erb_widths, erb_widths + cfg->nb_erb);
    if (const char *e = getenv("DFB_DEVICE_CHUNKS")) m->dev_chunks = atoi(e) > 0 ? atoi(e) : 0;
    if (const char *e = getenv("DFB_HOST_CHUNKS")) m->host_chunks = atoi(e) > 0 ? atoi(e) : 1;
    if (const char *e = getenv("DFB_LANES")) m->n_lanes = atoi(e) == 1 ? 1 : 2;
    if (const char *e = getenv("DFB_MAX_WORKSPACE_MB")) {
        const long long mb = atoll(e);
        if (mb > 0) m->max_workspace = (size_t)mb << 20;
    }
    // upload: one slab; GRU w_ih is stored transposed ([I][3H]) for the projection GEMM
    size_t total = 0;
    for (int i = 0; i < n_tensors; i++) total += ((size_t)tensors[i].numel * 4 + 255) & ~size_t(255);
    if (cudaMalloc(&m->slab, total + 256) != cudaSuccess) {
        delete m;
        return fail(DFB_ERR_OOM, "cudaMalloc(%zu) for weights failed", total);
    }
    size_t off = 0;
    std::vector<float> tmp;
    for (int i = 0; i < n_tensors; i++) {
        const dfb_tensor &tt = tensors[i];
        if (!tt.name || !tt.data || tt.numel <= 0) { dfb_model_free(m); return fail(DFB_ERR_INVALID, "bad tensor %d", i); }
        float *dst = (float *)((char *)m->slab + off);
        if (cudaMemcpy(dst, tt.data, (size_t)tt.numel * 4, cudaMemcpyHostToDevice) != cudaSuccess) {
            dfb_model_free(m);
            return fail(DFB_ERR_CUDA, "weight upload failed");
        }
        m->t[tt.name] = {dst, tt.numel};
        off += ((size_t)tt.numel * 4 + 255) & ~size_t(255);
    }
    int prio_least = 0, prio_greatest = 0;
    cudaDeviceGetStreamPriorityRange(&prio_least, &prio_greatest);
    // numerically greater = lower priority; the encoder phase sits one level below the decoder phase
    int prio_enc = prio_greatest + 1;
    if (prio_enc > prio_least) prio_enc = prio_least;
    bool ok = cudaStreamCreateWithFlags(&m->stream, cudaStreamNonBlocking) == cudaSuccess &&
              cudaStreamCreateWithFlags(&m->h2d, cudaStreamNonBlocking) == cudaSuccess &&
              cudaStreamCreateWithFlags(&m->d2h, cudaStreamNonBlocking) == cudaSuccess;
    for (auto &L : m->lanes) {
        ok = ok && cudaStreamCreateWithPriority(&L.main, cudaStreamNonBlocking, prio_enc) == cudaSuccess &&
             cudaStreamCreateWithPriority(&L.hi, cudaStreamNonBlocking, prio_enc) == cudaSuccess &&
             cudaStreamCreateWithPriority(&L.aux, cudaStreamNonBlocking, prio_enc) == cudaSuccess &&
             cudaStreamCreateWithPriority(&L.dhi, cudaStreamNonBlocking, prio_greatest) == cudaSuccess &&
             cudaStreamCreateWithPriority(&L.daux, cudaStreamNonBlocking, prio_greatest) == cudaSuccess &&
             cudaStreamCreateWithPriority(&L.low, cudaStreamNonBlocking, prio_least) == cudaSuccess;
        for (cudaEvent_t *e : {&L.ev_fork, &L.ev_join, &L.ev_fork_enc, &L.ev_join_enc, &L.ev_in, &L.ev_out, &L.ev_c0, &L.ev_convp,
                               &L.ev_skip, &L.ev_done})
            ok = ok && cudaEventCreateWithFlags(e, cudaEventDisableTiming) == cudaSuccess;
    }
    if (!ok) {
        dfb_model_free(m);
        return fail(DFB_ERR_CUDA, "stream creation failed");
    }
    *out = m;
    return DFB_OK;
}

extern "C" void dfb_model_free(dfb_model *m) {
    if (!m) return;
    cudaSetDevice(m->device);
    m->arena.release();
    m->arena1.release();
    m->aux_arena.release();
    if (m->h2d) cudaStreamDestroy(m->h2d);
    if (m->d2h) cudaStreamDestroy(m->d2h);
    if (m->slab) cudaFree(m->slab);
    if (m->stream) cudaStreamDestroy(m->stream);
    for (auto &L : m->lanes) {
        for (cudaStream_t st : {L.main, L.hi, L.aux, L.dhi, L.daux, L.low})
            if (st) cudaStreamDestroy(st);
        for (cudaEvent_t e : {L.ev_fork, L.ev_join, L.ev_fork_enc, L.ev_join_enc, L.ev_in, L.ev_out, L.ev_c0, L.ev_convp, L.ev_skip, L.ev_done})
            if (e) cudaEventDestroy(e);
    }
    delete m;
}

// Debug: when `steps` > 0, every following GRU launch stamps clock64() phases of CTA 0 into a device
// buffer [steps][8] (0 step start, 1 h arrived, 2 matvec done, 3 reduce + s_pre stored, 4 CTA barrier
// passed, 5 gates + sends issued); returns them for the LAST launch when called with h_out != NULL.
extern "C" int dfb_debug_gru_timing(dfb_model *m, int steps, long long *h_out) {
    if (!m) return fail(DFB_ERR_INVALID, "null model");
    cudaSetDevice(m->device);
    if (h_out && m->gru_dbg) {
        DFB_CUDA(cudaDeviceSynchronize());
        DFB_CUDA(cudaMemcpy(h_out, m->gru_dbg, sizeof(long long) * 8 * steps, cudaMemcpyDeviceToHost));
    }
    if (m->gru_dbg) { cudaFree(m->gru_dbg); m->gru_dbg = nullptr; }
    if (steps > 0 && !h_out) {
        DFB_CUDA(cudaMalloc(&m->gru_dbg, sizeof(long long) * 8 * steps));
        DFB_CUDA(cudaMemset(m->gru_dbg, 0, sizeof(long long) * 8 * steps));
    }
    return DFB_OK;
}

extern "C" int dfb_model_set_precision(dfb_model *m, int mode) {
    if (!m || mode < 0 || mode > 15 || (mode & 1)) return fail(DFB_ERR_INVALID, "precision mode out of range (bit 0 is reserved)");
    m->gru_tc = (mode >> 1) & 1;  // bit 1: tensor-core GRU recurrence (BF16x3 split, ~fp32 accurate)
    m->proj_tc = (mode >> 2) & 1; // bit 2: GRU input projections on the BF16x3 tcgen05 GEMM
    m->conv_tc = (mode >> 3) & 1; // bit 3: 1x1 convs of the separable blocks and the grouped linears on the BF16x3 tcgen05 kernels
    return DFB_OK;
}

extern "C" int64_t dfb_model_debug_fetch(dfb_model *m, const char *name, float *h_out, int64_t max_numel) {
    if (!m || !name || !h_out) return fail(DFB_ERR_INVALID, "null argument");
    auto it = m->dbg.find(name);
    if (it == m->dbg.end()) return fail(DFB_ERR_INVALID, "no activation named '%s'", name);
    int64_t n = it->second.second < max_numel ? it->second.second : max_numel;
    cudaSetDevice(m->device);
    if (cudaDeviceSynchronize() != cudaSuccess ||
        cudaMemcpy(h_out, it->second.first, (size_t)n * 4, cudaMemcpyDeviceToHost) != cudaSuccess)
        return fail(DFB_ERR_CUDA, "debug fetch failed: %s", cudaGetErrorString(cudaGetLastError()));
    return n;
}

extern "C" int64_t dfb_model_workspace_bytes(const dfb_model *m) { return m ? (int64_t)m->arena.cap : 0; }

namespace {

int run_gl(cudaStream_t s, const float *x, int64_t ldx, const float *w, const float *bias, const float *res,
           int64_t ldr, float *y, int64_t ldy, int64_t M, int G, int I, int Hh, int act, float oscale = 1.f,
           float ooffset = 0.f, unsigned short *y_hi = nullptr, unsigned short *y_lo = nullptr) {
    GlParams p{x, ldx, w, bias, res, ldr, y, ldy, M, G, I / G, Hh / G, act, oscale, ooffset, y_hi, y_lo};
    if ((p.Ig % 4) || (ldx % 4)) return fail(DFB_ERR_UNSUPPORTED, "grouped linear: K not a multiple of 4");
    if (G > 1 && (p.Hg % 4)) return fail(DFB_ERR_UNSUPPORTED, "grouped linear: group width %d not a multiple of 4", p.Hg);
    int tiles = (p.Hg + kGlBN - 1) / kGlBN;
    int gpc = (p.Hg < kGlBN && kGlBN % p.Hg == 0) ? (kGlBN / p.Hg < G ? kGlBN / p.Hg : G) : 1;
    dim3 grid((unsigned)((M + kGlBM - 1) / kGlBM), (unsigned)(((G + gpc - 1) / gpc) * tiles));
    // DFB_PROF_DETAIL=1 splits the grouped linears by shape in the profile (I x H / G)
    static const bool detail = getenv("DFB_PROF_DETAIL") && atoi(getenv("DFB_PROF_DETAIL"));
    char name[64];
    if (detail) snprintf(name, sizeof name, "k_grouped_linear[%dx%d/%d]", I, Hh, G);
    else snprintf(name, sizeof name, "%s", p.G == 1 && p.bias && p.Hg >= 512 ? "k_grouped_linear[gru_proj]" : "k_grouped_linear");
    DFB_PROF(name, s);
    k_grouped_linear<<<grid, 256, 0, s>>>(p);
    DFB_LAUNCH_CHECK();
    return DFB_OK;
}

template <int H, int C>
int launch_gru_t(cudaStream_t s, const GruParams &p, int ngroups) {
    constexpr int smem = (2 * kGruMaxBc * (H + 4) + 3 * (H / C) * (kGruMaxBc + 1)) * 4;
    static PerDeviceOnce attr_once;
    if (auto once_guard = attr_once.first()) {
        if (C > 8) DFB_CUDA(cudaFuncSetAttribute(k_gru<H, C>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
        DFB_CUDA(cudaFuncSetAttribute(k_gru<H, C>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    }
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)(ngroups * C));
    cfg.blockDim = dim3(kGruThreads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = C; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    GruParams pp = p;
    DFB_PROF("k_gru", s);
    DFB_CUDA(cudaLaunchKernelEx(&cfg, k_gru<H, C>, pp));
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return DFB_OK;
}

int pick_bc(int B, int max_clusters) {
    int bc = (B + max_clusters - 1) / max_clusters;
    bc = ((bc + kGruSB - 1) / kGruSB) * kGruSB;
    if (bc < kGruSB) bc = kGruSB;
    if (bc > kGruMaxBc) bc = kGruMaxBc;
    return bc;
}

// x [M, in_dim] -> multi-layer GRU -> y [M, H]  (uses xproj scratch [M,3H] and h ping-pong buffers)
// x_hi/x_lo: BF16 planes of x (written by the producing grouped linear), pl_hi/pl_lo: scratch planes for the
// inter-layer hidden state; used when the projection runs on the BF16x3 tensor-core GEMM.
int run_gru(dfb_model *m, cudaStream_t s, const char *name, int layers, int H, const float *x, int in_dim,
            const float *res_last, float *y, float *xproj, float *tmp_h, int B, int T,
            unsigned short *x_hi = nullptr, unsigned short *x_lo = nullptr, unsigned short *pl_hi = nullptr,
            unsigned short *pl_lo = nullptr, int wide = 0, unsigned short *out_hi = nullptr, unsigned short *out_lo = nullptr,
            bool *out_planes_ok = nullptr, const GruChunk *ck = nullptr) {
    if (out_planes_ok) *out_planes_ok = false;
    // time-chunked execution: the buffers hold T frames per stream, the recurrences run over frames [ck->t0, T) only and
    // continue from / leave behind the carried per-layer states; the projections simply cover every row
    const int t0 = ck ? ck->t0 : 0, Tn = T - t0;
    const int64_t M = (int64_t)B * T;
    const float *cur_in = x;
    int cur_dim = in_dim;
    const bool tc_gru = m->gru_tc && (H == 256 || H == 512);
    const bool tc_proj = m->proj_tc && tc_gru && x_hi && pl_hi && cur_dim % 64 == 0;
    const unsigned short *cur_hi = x_hi, *cur_lo = x_lo;
    for (int l = 0; l < layers; l++) {
        std::string base = std::string(name) + ".l" + std::to_string(l);
        const float *w_ih_t, *w_hh, *b_ih, *b_hh;
        int rc;
        if ((rc = need(m, (base + ".w_ih_t").c_str(), (int64_t)3 * H * cur_dim, &w_ih_t))) return rc;
        if ((rc = need(m, (base + ".w_hh").c_str(), (int64_t)3 * H * H, &w_hh))) return rc;
        if ((rc = need(m, (base + ".b_ih").c_str(), 3 * H, &b_ih))) return rc;
        if ((rc = need(m, (base + ".b_hh").c_str(), 3 * H, &b_hh))) return rc;
        if (tc_proj) {
            const float *w_hi, *w_lo;  // bf16 planes packed two per float
            if ((rc = need(m, (base + ".w_ih_hi").c_str(), (int64_t)3 * H * cur_dim / 2, &w_hi)) ||
                (rc = need(m, (base + ".w_ih_lo").c_str(), (int64_t)3 * H * cur_dim / 2, &w_lo)))
                return rc;
            rc = launch_gemm_bf16x3(s, cur_hi, cur_lo, cur_dim, w_hi, w_lo, b_ih, xproj, 3 * H, M, 3 * H, cur_dim);
        } else {
            rc = run_gl(s, cur_in, cur_dim, w_ih_t, b_ih, nullptr, 0, xproj, 3 * H, M, 1, cur_dim, 3 * H, ACT_NONE);
        }
        if (rc) return rc;
        float *dst = (l == layers - 1) ? y : tmp_h;
        float *hs = ck && ck->h ? ck->h + (int64_t)l * B * H : nullptr;   // carried state of this layer [B][H]
        GruWindow gw{ck && ck->have_state ? hs : nullptr, hs, t0, T};
        GruParams p{xproj, w_hh, b_hh, (l == layers - 1) ? res_last : nullptr, dst, B, Tn, 0, m->gru_dbg, gw.h0, gw.hT, t0, T};
        if (tc_gru) {
            const bool last = l == layers - 1;
            const bool planes = last ? out_hi != nullptr : tc_proj;
            // the last layer's planes feed a grouped linear and include the residual; the others feed the next projection
            rc = launch_gru_tc(s, xproj, w_hh, b_hh, last ? res_last : nullptr, dst, planes ? (last ? out_hi : pl_hi) : nullptr,
                               planes ? (last ? out_lo : pl_lo) : nullptr, B, Tn, m->gru_dbg, wide, last ? 1 : 0, &gw, H);
            if (last && planes && out_planes_ok) *out_planes_ok = true;
            cur_hi = pl_hi; cur_lo = pl_lo;
        } else if (H == 256) {
            p.Bc = pick_bc(B, 148 / 4);
            rc = launch_gru_t<256, 4>(s, p, (B + p.Bc - 1) / p.Bc);
        } else {
            p.Bc = pick_bc(B, 8);
            rc = launch_gru_t<512, 16>(s, p, (B + p.Bc - 1) / p.Bc);
        }
        if (rc) return rc;
        cur_in = dst;
        cur_dim = H;
        // middle layers may write tmp_h in place: the recurrence only reads xproj, which the
        // projection GEMM above has already produced from the previous contents of tmp_h.
    }
    return DFB_OK;
}

}  // namespace
namespace dfb {
template <int MODE>
int launch_dwpw_tc(cudaStream_t s, DwPwParams p, const float *w_sw, int B);
}
namespace {

template <int MODE>
int run_dwpw(cudaStream_t s, DwPwParams p, int B, const float *w_sw = nullptr) {
    if (w_sw) return launch_dwpw_tc<MODE>(s, p, w_sw, B);
    static PerDeviceOnce attr_once;
    const int smem = (kCh * kCh + 128 * kLdA) * 4;
    if (auto once_guard = attr_once.first()) {
        DFB_CUDA(cudaFuncSetAttribute(k_dwpw<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    }
    p.NF = 128 / p.Fout;
    if (p.NF < 1) p.NF = 1;
    if (p.NF * p.Fout > 128 || (p.NF * p.Fout) % 4) return fail(DFB_ERR_UNSUPPORTED, "dwpw tile: Fout = %d", p.Fout);
    dim3 grid((unsigned)((p.T + p.NF - 1) / p.NF), (unsigned)B);
    DFB_PROF(MODE == DW_DF0 ? "k_dwpw[df_conv0]" : "k_dwpw", s);
    k_dwpw<MODE><<<grid, 256, smem, s>>>(p);
    DFB_LAUNCH_CHECK();
    return DFB_OK;
}

}  // namespace

// Buffers of one forward pass (all from the model arena).
struct FwdBufs {
    float *e0, *e1, *e2, *e3, *c0, *c1, *emb_in, *emb, *g_a, *g_b, *g_h, *xproj, *dec_emb, *d3, *d2, *d1, *dfc;
    unsigned short *ga_hi, *ga_lo, *gh_hi, *gh_lo;  // BF16 planes of g_a / inter-layer h (tensor-core projections)
    // second set of GRU scratch: the DF decoder runs concurrently with the ERB decoder on another stream
    float *g_a2, *g_h2, *xproj2, *dfskip;
    unsigned short *ga2_hi, *ga2_lo, *gh2_hi, *gh2_lo;
    // BF16 hi / lo planes of the grouped linears' inputs (tensor-core path): c1, emb_in, GRU outputs, emb
    unsigned short *c1_hi, *c1_lo, *embin_hi, *embin_lo, *gb_hi, *gb_lo, *emb_hi, *emb_lo, *dfc_hi, *dfc_lo;
};

// DeepFilterNet v1 (forward_v1)
struct FwdBufsV1 {
    float *e0, *e1, *e2, *e3, *c0, *c1, *c1g, *cemb, *emb, *xproj, *xproj2, *y[3], *embo, *dec_old, *dec, *p3, *p2, *p1, *p0, *d3, *d2, *d1,
        *z[2], *dfc;
    unsigned short *emb_hi, *emb_lo, *y_hi[3], *y_lo[3], *embo_hi, *embo_lo, *z_hi[2], *z_lo[2], *dfc_hi, *dfc_lo, *scr_hi, *scr_lo;
};
static size_t fwd_plan_v1(const dfb_model_config &c, size_t M, Arena *a, FwdBufsV1 *f) {
    const int E = c.nb_erb, Fd = c.nb_df, H = c.emb_hidden;
    size_t bytes = 0;
    auto take = [&](size_t n) -> float * {
        bytes += (n * 4 + 255) & ~size_t(255);
        return a ? a->take<float>(n) : nullptr;
    };
    auto take16 = [&](size_t n) { return reinterpret_cast<unsigned short *>(take((n + 1) / 2)); };
    FwdBufsV1 t{};
    t.e0 = take(M * E * kCh); t.e1 = take(M * (E / 2) * kCh); t.e2 = take(M * (E / 4) * kCh); t.e3 = take(M * (E / 4) * kCh);
    t.c0 = take(M * Fd * kCh); t.c1 = take(M * (Fd / 2) * kCh); t.c1g = take(M * (Fd / 2) * kCh);
    t.cemb = take(M * H); t.emb = take(M * H); t.xproj = take(M * 3 * H); t.xproj2 = take(M * 3 * H);
    for (int i = 0; i < 3; i++) { t.y[i] = take(M * H); t.y_hi[i] = take16(M * H); t.y_lo[i] = take16(M * H); }
    for (int i = 0; i < 2; i++) { t.z[i] = take(M * H); t.z_hi[i] = take16(M * H); t.z_lo[i] = take16(M * H); }
    t.embo = take(M * H); t.dec_old = take(M * H); t.dec = take(M * H); t.dfc = take(M * H);
    t.p3 = take(M * (E / 4) * kCh); t.p2 = take(M * (E / 4) * kCh); t.p1 = take(M * (E / 2) * kCh); t.p0 = take(M * E * kCh);
    t.d3 = take(M * (E / 4) * kCh); t.d2 = take(M * (E / 2) * kCh); t.d1 = take(M * E * kCh);
    t.emb_hi = take16(M * H); t.emb_lo = take16(M * H); t.embo_hi = take16(M * H); t.embo_lo = take16(M * H);
    t.dfc_hi = take16(M * H); t.dfc_lo = take16(M * H); t.scr_hi = take16(M * H); t.scr_lo = take16(M * H);
    if (f) *f = t;
    return bytes + 4096;
}

// Carves the activations of `M` frames out of `a` (or only counts bytes when a == nullptr).
static size_t fwd_plan(const dfb_model_config &c, size_t M, Arena *a, FwdBufs *f) {
    if (c.model_kind == 1 && !a) return fwd_plan_v1(c, M, nullptr, nullptr);
    const int E = c.nb_erb, Fd = c.nb_df, H = c.emb_hidden, Hd = c.df_hidden;
    const int ED = E / 4 * kCh;
    const int emb_in_dim = c.enc_concat ? 2 * ED : ED;
    const int emb_dim = c.model_kind == 2 ? H : ED;
    const int Hmax = H > Hd ? H : Hd;
    size_t bytes = 0;
    auto take = [&](size_t n) -> float * {
        bytes += (n * 4 + 255) & ~size_t(255);
        return a ? a->take<float>(n) : nullptr;
    };
    FwdBufs t{};
    t.e0 = take(M * E * kCh); t.e1 = take(M * (E / 2) * kCh); t.e2 = take(M * (E / 4) * kCh);
    t.emb_in = take(M * emb_in_dim);
    t.e3 = c.enc_concat ? t.emb_in : take(M * ED);  // DFN2: e3 lives inside the concat buffer
    t.c0 = take(M * Fd * kCh); t.c1 = take(M * (Fd / 2) * kCh);
    t.emb = take(M * emb_dim);
    t.g_a = take(M * Hmax); t.g_b = take(M * Hmax); t.g_h = take(M * Hmax);
    t.xproj = take(M * 3 * Hmax);
    t.dec_emb = take(M * ED); t.d3 = take(M * ED); t.d2 = take(M * (E / 2) * kCh);
    t.d1 = take(M * E * kCh); t.dfc = take(M * Hmax);
    t.ga_hi = reinterpret_cast<unsigned short *>(take(M * Hmax / 2)); t.ga_lo = reinterpret_cast<unsigned short *>(take(M * Hmax / 2));
    t.gh_hi = reinterpret_cast<unsigned short *>(take(M * Hmax / 2)); t.gh_lo = reinterpret_cast<unsigned short *>(take(M * Hmax / 2));
    t.g_a2 = take(M * Hmax); t.g_h2 = take(M * Hmax); t.xproj2 = take(M * 3 * Hmax); t.dfskip = take(M * Hmax);
    t.ga2_hi = reinterpret_cast<unsigned short *>(take(M * Hmax / 2)); t.ga2_lo = reinterpret_cast<unsigned short *>(take(M * Hmax / 2));
    t.gh2_hi = reinterpret_cast<unsigned short *>(take(M * Hmax / 2)); t.gh2_lo = reinterpret_cast<unsigned short *>(take(M * Hmax / 2));
    auto take16 = [&](size_t n) { return reinterpret_cast<unsigned short *>(take((n + 1) / 2)); };
    t.c1_hi = take16(M * (Fd / 2) * kCh); t.c1_lo = take16(M * (Fd / 2) * kCh);
    t.embin_hi = take16(M * emb_in_dim); t.embin_lo = take16(M * emb_in_dim);
    t.gb_hi = take16(M * Hmax); t.gb_lo = take16(M * Hmax);
    t.emb_hi = take16(M * emb_dim); t.emb_lo = take16(M * emb_dim);
    t.dfc_hi = take16(M * Hmax); t.dfc_lo = take16(M * Hmax);
    if (f) *f = t;
    return bytes + 4096;
}

// Time-chunked execution (dfb_enhance's chunk loop, the streaming API): the window holds T frames per stream of which
// the first Rc were already processed by the previous chunk (halo: the feed-forward layers recompute them from the
// carried feature history, the recurrences skip them and continue from the carried hidden states).
struct ChunkCtx {
    int Rc;                        // halo frames at the head of the window
    int Tsx, Tx;                   // feature buffers: frames per stream, frames that exist (beyond = end of stream)
    float *h_enc, *h_erb, *h_df;   // carried GRU states [layers][B][H]
    bool have_state;               // false for the first chunk of a stream (states start at zero)
    float *dec_tail;               // (conv_kt == 2) last kHalo frames of dec_emb [B][kHalo][ED], right aligned
    int dec_tail_n;                // frames of dec_tail that are valid
    int lane;                      // which of the model's two stream / event sets (and arenas) this chunk runs on
    cudaEvent_t wait_dec;          // previous chunk finished (its decoder states / tails are final) or null
};
constexpr int kHalo = 8;           // >= temporal receptive field of every feed-forward chain of the shipped models

static int forward_impl(dfb_model *m, Arena &arena, const float *d_feat_erb, const float *d_feat_spec, int B, int T,
                        float *d_m, float *d_coefs, float *d_lsnr, float *d_alpha, cudaStream_t s, ChunkCtx *cx = nullptr);

extern "C" int dfb_model_forward(dfb_model *m, const float *d_feat_erb, const float *d_feat_spec, int64_t B64,
                                 int64_t T64, float *d_m, float *d_coefs, float *d_lsnr, float *d_alpha,
                                 void *stream) {
    if (!m || !d_feat_erb || !d_feat_spec || !d_m || !d_coefs) return fail(DFB_ERR_INVALID, "null argument");
    if (B64 <= 0 || T64 <= 0) return DFB_OK;
    if (B64 > 65535) return fail(DFB_ERR_INVALID, "more than 65535 streams per call");
    DFB_CUDA(cudaSetDevice(m->device));
    int rc = m->arena.reserve(fwd_plan(m->cfg, (size_t)B64 * T64, nullptr, nullptr));
    if (rc) return rc;
    m->arena.reset();
    rc = forward_impl(m, m->arena, d_feat_erb, d_feat_spec, (int)B64, (int)T64, d_m, d_coefs, d_lsnr, d_alpha,
                      (cudaStream_t)stream);
    m->arena.reset();
    return rc;
}

static int forward_body(dfb_model *m, Arena &arena, const float *d_feat_erb, const float *d_feat_spec, int B, int T,
                        float *d_m, float *d_coefs, float *d_lsnr, float *d_alpha, cudaStream_t s_in, ChunkCtx *cx);

static int forward_v1(dfb_model *m, Arena &arena, const float *d_feat_erb, const float *d_feat_spec, int B, int T,
                      float *d_m, float *d_coefs, float *d_lsnr, float *d_alpha, cudaStream_t s_in, ChunkCtx *cx);

static int forward_impl(dfb_model *m, Arena &arena, const float *d_feat_erb, const float *d_feat_spec, int B, int T,
                        float *d_m, float *d_coefs, float *d_lsnr, float *d_alpha, cudaStream_t s_in, ChunkCtx *cx) {
    const int rc = m->cfg.model_kind == 1
        ? forward_v1(m, arena, d_feat_erb, d_feat_spec, B, T, d_m, d_coefs, d_lsnr, d_alpha, s_in, cx)
        : forward_body(m, arena, d_feat_erb, d_feat_spec, B, T, d_m, d_coefs, d_lsnr, d_alpha, s_in, cx);
    // an early return may leave work on the forked internal streams un-joined while the caller goes on to reuse
    // the arena: drain the device before handing the error back (error path only)
    if (rc) cudaDeviceSynchronize();
    return rc;
}

static int forward_body(dfb_model *m, Arena &arena, const float *d_feat_erb, const float *d_feat_spec, int B, int T,
                        float *d_m, float *d_coefs, float *d_lsnr, float *d_alpha, cudaStream_t s_in, ChunkCtx *cx) {
    const dfb_model_config &c = m->cfg;
    const int Tsx = cx ? cx->Tsx : T, Tx = cx ? cx->Tx : T;
    GruChunk ck_enc{cx ? cx->h_enc : nullptr, cx && cx->have_state, cx ? cx->Rc : 0};
    GruChunk ck_erb{cx ? cx->h_erb : nullptr, cx && cx->have_state, cx ? cx->Rc : 0};
    GruChunk ck_df{cx ? cx->h_df : nullptr, cx && cx->have_state, cx ? cx->Rc : 0};
    // DFB_SERIAL=1: everything on the caller's stream (profiling: per-kernel times without overlap)
    static const bool serial = getenv("DFB_SERIAL") && atoi(getenv("DFB_SERIAL"));
    dfb_model::Lane &L = m->lanes[cx ? cx->lane : 0];
    cudaStream_t s = serial ? s_in : L.hi;
    cudaStream_t sl = serial ? s_in : L.low;
    if (!serial) {
        DFB_CUDA(cudaEventRecord(L.ev_in, s_in));
        DFB_CUDA(cudaStreamWaitEvent(s, L.ev_in, 0));
    }
    auto finish = [&]() -> int {  // join the branches and hand the result back to the caller's stream
        DFB_CUDA(cudaStreamWaitEvent(s, L.ev_join, 0));
        if (!serial) {
            DFB_CUDA(cudaEventRecord(L.ev_out, s));
            DFB_CUDA(cudaStreamWaitEvent(s_in, L.ev_out, 0));
        }
        return DFB_OK;
    };
    const int64_t M = (int64_t)B * T;
    const int E = c.nb_erb, Fd = c.nb_df, H = c.emb_hidden, Hd = c.df_hidden;
    const int ED = E / 4 * kCh;  // embedding width (512)
    const int emb_in_dim = c.enc_concat ? 2 * ED : ED;
    const int emb_dim = c.model_kind == 2 ? H : ED;  // encoder output width
    int rc;
    FwdBufs f{};
    fwd_plan(c, (size_t)M, &arena, &f);
    if (!f.gh2_lo || !f.dfskip || !f.dfc_lo) return fail(DFB_ERR_OOM, "forward workspace exhausted for %lld frames", (long long)M);
    m->dbg.clear();
    m->dbg["e0"] = {f.e0, M * E * kCh}; m->dbg["e1"] = {f.e1, M * (E / 2) * kCh}; m->dbg["e2"] = {f.e2, M * (E / 4) * kCh};
    m->dbg["e3"] = {f.e3, c.enc_concat ? M * emb_in_dim : M * ED}; m->dbg["c0"] = {f.c0, M * Fd * kCh};
    m->dbg["c1"] = {f.c1, M * (Fd / 2) * kCh}; m->dbg["emb_in"] = {f.emb_in, M * emb_in_dim};
    m->dbg["emb"] = {f.emb, M * emb_dim}; m->dbg["dec_emb"] = {f.dec_emb, M * ED}; m->dbg["d3"] = {f.d3, M * ED};
    m->dbg["d2"] = {f.d2, M * (E / 2) * kCh}; m->dbg["d1"] = {f.d1, M * E * kCh}; m->dbg["dfc"] = {f.dfc, M * Hd};
    m->dbg["g_a"] = {f.g_a, M * (H > Hd ? H : Hd)}; m->dbg["g_b"] = {f.g_b, M * (H > Hd ? H : Hd)};
    m->dbg["xproj"] = {f.xproj, M * 3 * (H > Hd ? H : Hd)};
    const int64_t e3_fs = c.enc_concat ? 2 * ED : ED;
    // BF16 hi / lo planes [M][K] (row pitch `ld` elements) of a grouped linear's input; `ok` = already written by the producer
    struct Pl { unsigned short *hi, *lo; int64_t ld; bool ok; };
    Pl pl_c1{f.c1_hi, f.c1_lo, (int64_t)Fd / 2 * kCh, false}, pl_embin{f.embin_hi, f.embin_lo, emb_in_dim, false},
       pl_gb{f.gb_hi, f.gb_lo, H, false}, pl_emb{f.emb_hi, f.emb_lo, emb_dim, false}, pl_dfc{f.dfc_hi, f.dfc_lo, Hd, false},
       pl_ga{f.ga_hi, f.ga_lo, H, false}, pl_ga2{f.ga2_hi, f.ga2_lo, Hd, false};
    const bool gl_tc = m->conv_tc != 0;
    // planes of `x` for a tensor-core consumer: converts on `st` unless the producer already wrote them
    auto ensure_planes = [&](cudaStream_t st, const float *x, int64_t ldx, int K, Pl &pl) -> int {
        if (pl.ok) return DFB_OK;
        if (pl.ld != K) return fail(DFB_ERR_INVALID, "plane pitch mismatch");
        int r = launch_to_planes(st, x, ldx, M, K, pl.hi, pl.lo);
        if (!r) pl.ok = true;
        return r;
    };
    // grouped linear `wname` ([G][I/G][Hh/G]): the BF16x3 tcgen05 kernel when the tensor-core bit is set and the shape is
    // built, else the FFMA kernel.  xin: planes of x (converted on demand); yout (optional): planes of y to produce,
    // ycol: column offset of y inside its plane buffer
    auto gl = [&](cudaStream_t st, const char *wname, const float *x, int64_t ldx, Pl *xin, int G, int I, int Hh, int act,
                  const float *res, int64_t ldr, float *y, int64_t ldy, Pl *yout, int64_t ycol = 0) -> int {
        const float *w;
        int r;
        if ((r = need(m, wname, (int64_t)I * Hh / G, &w))) return r;
        unsigned short *yh = yout ? yout->hi + ycol : nullptr, *yl = yout ? yout->lo + ycol : nullptr;
        const std::string bx = std::string(wname) + "_bx";
        int gpc, hgp, stages;
        if (gl_tc && xin && m->get(bx) && gl_bx_geometry(G, I / G, Hh / G, &gpc, &hgp, &stages)) {
            if ((r = ensure_planes(st, x, ldx, I, *xin))) return r;
            r = launch_gl_bx(st, xin->hi, xin->lo, xin->ld, m->get(bx), res, ldr, y, ldy, yh, yl, yout ? yout->ld : 0, M, G, I / G,
                             Hh / G, act, 1.f, 0.f);
            if (r != DFB_ERR_UNSUPPORTED) {
                if (!r && yout && (ycol == 0 || true)) yout->ok = true;
                return r;
            }
        }
        // NB: the FFMA kernel's plane output shares y's pitch, so it can only serve plane buffers with ld == ldy
        const bool ffma_planes = yout && yout->ld == ldy;
        r = run_gl(st, x, ldx, w, nullptr, res, ldr, y, ldy, M, G, I, Hh, act, 1.f, 0.f, ffma_planes ? yh : nullptr, ffma_planes ? yl : nullptr);
        if (!r && yout) yout->ok = ffma_planes;
        return r;
    };

    // ---- encoder (deepfilternet3.py:166-185)
    {
        const float *w, *bb;
        if ((rc = need(m, "enc.erb_conv0.w", c.inp_kt * 3 * kCh, &w)) || (rc = need(m, "enc.erb_conv0.b", kCh, &bb))) return rc;
        dim3 grid((unsigned)((T + kInFrames - 1) / kInFrames), (unsigned)B);
        int smem = (kInFrames + c.inp_kt - 1) * (E + 2) * 4;
        DFB_PROF("k_conv_in[erb_conv0]", s);
        k_conv_in<1><<<grid, 256, smem, s>>>(d_feat_erb, w, bb, f.e0, T, E, c.inp_kt, c.conv_lookahead, Tsx, Tx, 0);
        DFB_LAUNCH_CHECK();
    }
    const float *pw_sw = nullptr;  // set by blk(): swizzled BF16 hi | lo image of the [C_out][C_in] 1x1 weights (tensor-core path)
    auto blk = [&](const char *name, DwPwParams &p) -> int {
        std::string n(name);
        int r;
        if ((r = need(m, (n + ".dw").c_str(), -1, &p.dw)) || (r = need(m, (n + ".pw").c_str(), kCh * kCh, &p.pw)) ||
            (r = need(m, (n + ".b").c_str(), kCh, &p.bias)))
            return r;
        pw_sw = nullptr;
        if (m->conv_tc && (r = need(m, (n + ".pw_sw").c_str(), kCh * kCh, &pw_sw))) return r;
        return DFB_OK;
    };
    // the DF-branch input convs run concurrently with the ERB-branch convs
    cudaStream_t sa = serial ? s : L.aux;
    DFB_CUDA(cudaEventRecord(L.ev_fork_enc, s));
    DFB_CUDA(cudaStreamWaitEvent(sa, L.ev_fork_enc, 0));
    auto mk = [&](const float *in, int Fin, int64_t in_fs, float *out, int Fout, int64_t out_fs, int kt) {
        DwPwParams p{};
        p.in = in; p.Fin = Fin; p.in_fs = in_fs; p.out = out; p.Fout = Fout; p.out_fs = out_fs; p.kt = kt; p.T = T;
        p.lookahead = 0;
        return p;
    };
    {
        DwPwParams p{};
        {
            const float *w, *bb;
            if ((rc = need(m, "enc.df_conv0.w", c.inp_kt * 3 * 2 * kCh, &w)) || (rc = need(m, "enc.df_conv0.b", kCh, &bb))) return rc;
            dim3 grid((unsigned)((T + kInFrames - 1) / kInFrames), (unsigned)B);
            int smem = (kInFrames + c.inp_kt - 1) * (Fd + 2) * 2 * 4;
            DFB_PROF("k_conv_in[df_conv0]", sa);
            k_conv_in<2><<<grid, 256, smem, sa>>>(d_feat_spec, w, bb, f.c0, T, Fd, c.inp_kt, c.conv_lookahead, Tsx, Tx, 0);
            DFB_LAUNCH_CHECK();
            DFB_CUDA(cudaEventRecord(L.ev_c0, sa));
        }
        p = mk(f.c0, Fd, (int64_t)Fd * kCh, f.c1, Fd / 2, (int64_t)Fd / 2 * kCh, c.conv_kt);
        if ((rc = blk("enc.df_conv1", p))) return rc;
        if (pw_sw && gl_tc) {  // c1 only feeds df_fc_emb: write its BF16 planes instead of the fp32 tensor
            p.out = nullptr; p.out_hi = pl_c1.hi; p.out_lo = pl_c1.lo; pl_c1.ok = true;
            m->dbg.erase("c1");
        }
        if ((rc = run_dwpw<DW_S2>(sa, p, B, pw_sw))) return rc;
        DFB_CUDA(cudaEventRecord(L.ev_join_enc, sa));
        // DF pathway conv (needs c0 only; its result is consumed by the very last DF-decoder kernel): on the
        // low-priority stream, so its CTAs only take SMs that the critical path -- the encoder convs now, the GRU
        // clusters later -- leaves idle (timeline: on the auxiliary stream it delayed df_fc_emb by 1.8 ms)
        // (also measured with a saturated device -- 512 x 10 s --: on the DF branch's encoder stream it slows df_fc_emb by
        // as much as it gains at the tail, 49.4 vs 45.2 ms per step)
        DFB_CUDA(cudaStreamWaitEvent(sl, L.ev_c0, 0));
        const int O2 = 2 * c.df_order;
        const float *w1, *w2, *bb;
        if ((rc = need(m, "df_dec.df_convp.w1", (int64_t)c.df_pathway_kt * O2 * (kCh / 2), &w1)) ||
            (rc = need(m, "df_dec.df_convp.w2", O2 * O2, &w2)) || (rc = need(m, "df_dec.df_convp.b", O2, &bb)))
            return rc;
        if (c.df_order != 5 || c.df_pathway_kt != 5)
            return fail(DFB_ERR_UNSUPPORTED, "df_order %d / df_pathway_kernel_size_t %d (built kernels: 5, 5)", c.df_order,
                        c.df_pathway_kt);
        if (Fd % 2) return fail(DFB_ERR_UNSUPPORTED, "df pathway conv: odd nb_df");
        dim3 grid((unsigned)((Fd + 2 * kCpWarps - 1) / (2 * kCpWarps)), (unsigned)((T + kCpChunk - 1) / kCpChunk), (unsigned)B);
        const float *w_sw = m->conv_tc ? m->get("df_dec.df_convp.w_sw") : nullptr;
        if (w_sw) {  // channel contraction on tcgen05 (BF16x3), shifted adds + 1x1 conv in the epilogue
            if ((rc = launch_df_convp_tc(sl, f.c0, w_sw, w2, bb, d_coefs, B, T, Fd))) return rc;
        } else {
            DFB_PROF("k_df_convp", sl);
            const int smem = kCpWarps * kCpSlots * (512 + 8);
            k_df_convp<5, 5, 3><<<grid, 32 * kCpWarps, smem, sl>>>(f.c0, w1, w2, bb, d_coefs, T, Fd);
            DFB_LAUNCH_CHECK();
        }
        DFB_CUDA(cudaEventRecord(L.ev_convp, sl));
    }
    {
        DwPwParams p = mk(f.e0, E, (int64_t)E * kCh, f.e1, E / 2, (int64_t)E / 2 * kCh, c.conv_kt);
        if ((rc = blk("enc.erb_conv1", p)) || (rc = run_dwpw<DW_S2>(s, p, B, pw_sw))) return rc;
        p = mk(f.e1, E / 2, (int64_t)E / 2 * kCh, f.e2, E / 4, (int64_t)E / 4 * kCh, c.conv_kt);
        if ((rc = blk("enc.erb_conv2", p)) || (rc = run_dwpw<DW_S2>(s, p, B, pw_sw))) return rc;
        p = mk(f.e2, E / 4, (int64_t)E / 4 * kCh, f.e3, E / 4, e3_fs, c.conv_kt);
        if ((rc = blk("enc.erb_conv3", p))) return rc;
        if (pw_sw && gl_tc && c.enc_concat) { p.out_hi = pl_embin.hi; p.out_lo = pl_embin.lo; }  // DFN2: e3 is the first half of emb_in
        if ((rc = run_dwpw<DW_S1>(s, p, B, pw_sw))) return rc;

    }
    DFB_CUDA(cudaStreamWaitEvent(s, L.ev_join_enc, 0));  // c0 / c1 ready
    {
        // cemb = relu(df_fc_emb(c1 flat)); emb_in = e3 flat + cemb  (DFN2: concat)
        const int I = Fd / 2 * kCh;
        const bool e3_planes = pw_sw && gl_tc && c.enc_concat;
        if (c.enc_concat) {
            rc = gl(s, "enc.df_fc_emb.gl", f.c1, I, &pl_c1, c.g_df_fc_emb, I, ED, ACT_RELU, nullptr, 0, f.emb_in + ED, emb_in_dim,
                    &pl_embin, ED);
            pl_embin.ok = pl_embin.ok && e3_planes;  // both halves must have been written as planes
        } else {
            rc = gl(s, "enc.df_fc_emb.gl", f.c1, I, &pl_c1, c.g_df_fc_emb, I, ED, ACT_RELU, f.e3, ED, f.emb_in, emb_in_dim, &pl_embin);
        }
        if (rc) return rc;
    }
    {
        // enc.emb_gru: linear_in + ReLU -> GRU -> [linear_out + ReLU]
        if ((rc = gl(s, "enc.emb_gru.in.gl", f.emb_in, emb_in_dim, &pl_embin, c.g_enc_in, emb_in_dim, H, ACT_RELU, nullptr, 0, f.g_a, H,
                     &pl_ga))) return rc;
        float *gout = c.g_enc_out ? f.g_b : f.emb;
        Pl &pl_gout = c.g_enc_out ? pl_gb : pl_emb;
        if ((rc = run_gru(m, s, "enc.emb_gru", c.enc_gru_layers, H, f.g_a, H, nullptr, gout, f.xproj, f.g_h, B, T, f.ga_hi, f.ga_lo,
                          f.gh_hi, f.gh_lo, 0, gl_tc ? pl_gout.hi : nullptr, gl_tc ? pl_gout.lo : nullptr, &pl_gout.ok, cx ? &ck_enc : nullptr))) return rc;
        if (c.g_enc_out) {
            if ((rc = gl(s, "enc.emb_gru.out.gl", f.g_b, H, &pl_gb, c.g_enc_out, H, ED, ACT_RELU, nullptr, 0, f.emb, emb_dim, &pl_emb)))
                return rc;
        }
        // the decoders read emb's planes on two streams: make sure they exist before the fork
        if (gl_tc && (rc = ensure_planes(s, f.emb, emb_dim, emb_dim, pl_emb))) return rc;
        if (d_lsnr) {
            const float *lw, *lb;
            if ((rc = need(m, "enc.lsnr.w", emb_dim, &lw)) || (rc = need(m, "enc.lsnr.b", 1, &lb))) return rc;
            if ((rc = run_gl(s, f.emb, emb_dim, lw, lb, nullptr, 0, d_lsnr, 1, M, 1, emb_dim, 1, ACT_SIGMOID, c.lsnr_scale, c.lsnr_offset))) return rc;
        }
    }
    // fork: the two decoders only share read-only encoder outputs
    // the encoder phase is done (ev_fork also tells the next time chunk that it may start); the decoder phase runs on the
    // lane's greatest-priority streams and, in the chunk pipeline, after the previous chunk's decoder has finished
    DFB_CUDA(cudaEventRecord(L.ev_fork, s));
    if (!serial) { s = L.dhi; sa = L.daux; DFB_CUDA(cudaStreamWaitEvent(s, L.ev_fork, 0)); }
    DFB_CUDA(cudaStreamWaitEvent(sa, L.ev_fork, 0));
    if (cx && cx->wait_dec) {
        DFB_CUDA(cudaStreamWaitEvent(s, cx->wait_dec, 0));
        DFB_CUDA(cudaStreamWaitEvent(sa, cx->wait_dec, 0));
    }
    // DFN3's grouped-linear skip around the DF GRU does not depend on the recurrence: evaluate it here (the ERB
    // branch has the slack) and let the last GRU layer add it as its output residual, instead of a kernel on the
    // DF branch's tail, which is the critical path of the decoder phase
    // the two decoders' recurrences run concurrently and at most 15 clusters of 8 CTAs are co-resident: the DF branch uses 32
    // streams per cluster for batches above 64, the ERB branch 16
    const int wide_df = 1, wide_erb = 0;
    const bool early_skip = c.g_df_skip && c.model_kind != 2;
    if (early_skip) {
        if ((rc = gl(s, "df_dec.df_skip.gl", f.emb, emb_dim, &pl_emb, c.g_df_skip, emb_dim, Hd, ACT_NONE, nullptr, 0, f.dfskip, Hd, nullptr)))
            return rc;
        DFB_CUDA(cudaEventRecord(L.ev_skip, s));
    }
    // ---- DF decoder (deepfilternet3.py:323-331), on the auxiliary stream (forked after the encoder)
    {
        cudaStream_t s = sa;  // shadows the caller stream inside this block
        if ((rc = gl(s, "df_dec.df_gru.in.gl", f.emb, emb_dim, &pl_emb, c.g_df_in, emb_dim, Hd, ACT_RELU, nullptr, 0, f.g_a2, Hd, &pl_ga2)))
            return rc;
        const float *res = c.model_kind == 2 ? f.g_a2 : (early_skip ? f.dfskip : nullptr);
        if (early_skip) DFB_CUDA(cudaStreamWaitEvent(s, L.ev_skip, 0));
        if ((rc = run_gru(m, s, "df_dec.df_gru", c.df_gru_layers, Hd, f.g_a2, Hd, res, f.dfc, f.xproj2, f.g_h2, B, T, f.ga2_hi, f.ga2_lo,
                          f.gh2_hi, f.gh2_lo, wide_df, gl_tc ? pl_dfc.hi : nullptr, gl_tc ? pl_dfc.lo : nullptr, &pl_dfc.ok, cx ? &ck_df : nullptr))) return rc;
        if (c.g_df_skip && !early_skip) {
            if ((rc = gl(s, "df_dec.df_skip.gl", f.emb, emb_dim, &pl_emb, c.g_df_skip, emb_dim, Hd, ACT_NONE, f.dfc, Hd, f.dfc, Hd, nullptr)))
                return rc;
            pl_dfc.ok = false;
        }
        if (d_alpha && c.model_kind == 2) {  // alpha = sigmoid(df_fc_a(c)), deepfilternet2.py:368
            const float *aw, *ab;
            if ((rc = need(m, "df_dec.df_fc_a.w", Hd, &aw)) || (rc = need(m, "df_dec.df_fc_a.b", 1, &ab))) return rc;
            if ((rc = run_gl(s, f.dfc, Hd, aw, ab, nullptr, 0, d_alpha, 1, M, 1, Hd, 1, ACT_SIGMOID))) return rc;
        }
        const int O2 = 2 * c.df_order;
        // coefs = tanh(df_out(c)) + df_convp(c0); the pathway term was written by k_df_convp on the low-priority stream
        DFB_CUDA(cudaStreamWaitEvent(s, L.ev_convp, 0));
        if ((rc = gl(s, "df_dec.df_out.gl", f.dfc, Hd, &pl_dfc, c.g_df_out, Hd, Fd * O2, ACT_TANH, d_coefs, (int64_t)Fd * O2, d_coefs,
                     (int64_t)Fd * O2, nullptr))) return rc;
    }
    DFB_CUDA(cudaEventRecord(L.ev_join, sa));
    // ---- ERB decoder (deepfilternet3.py:245-254)
    {
        if ((rc = gl(s, "erb_dec.emb_gru.in.gl", f.emb, emb_dim, &pl_emb, c.g_erb_in, emb_dim, H, ACT_RELU, nullptr, 0, f.g_a, H, &pl_ga)))
            return rc;
        // DFN2 (SqueezedGRU): identity skip around the GRU, y = GRU(x) + x  (modules.py:695-697)
        const float *res = c.model_kind == 2 ? f.g_a : nullptr;
        pl_gb.ok = false;
        if ((rc = run_gru(m, s, "erb_dec.emb_gru", c.erb_gru_layers, H, f.g_a, H, res, f.g_b, f.xproj, f.g_h, B, T, f.ga_hi, f.ga_lo,
                          f.gh_hi, f.gh_lo, wide_erb, gl_tc ? pl_gb.hi : nullptr, gl_tc ? pl_gb.lo : nullptr, &pl_gb.ok, cx ? &ck_erb : nullptr))) return rc;
        if ((rc = gl(s, "erb_dec.emb_gru.out.gl", f.g_b, H, &pl_gb, c.g_erb_out, H, ED, ACT_RELU, nullptr, 0, f.dec_emb, ED, nullptr)))
            return rc;
        if (cx && cx->dec_tail && c.conv_kt > 1) {
            // kt = 2 decoder convs look one frame back into the halo, where this window's recurrence did not run: restore
            // dec_emb there from the previous chunk, then keep this window's last frames for the next one
            const size_t fb = sizeof(float) * ED;
            const int nl = cx->Rc < cx->dec_tail_n ? cx->Rc : cx->dec_tail_n;
            if (cx->have_state && nl > 0)
                DFB_CUDA(cudaMemcpy2DAsync(f.dec_emb + (size_t)(cx->Rc - nl) * ED, fb * T, cx->dec_tail + (size_t)(kHalo - nl) * ED,
                                           fb * kHalo, fb * nl, B, cudaMemcpyDeviceToDevice, s));
            const int ns = T < kHalo ? T : kHalo;
            DFB_CUDA(cudaMemcpy2DAsync(cx->dec_tail + (size_t)(kHalo - ns) * ED, fb * kHalo, f.dec_emb + (size_t)(T - ns) * ED, fb * T,
                                       fb * ns, B, cudaMemcpyDeviceToDevice, s));
            cx->dec_tail_n = ns;
        }
        auto path = [&](DwPwParams &p, const char *pn, const float *pt, int64_t pfs) -> int {
            std::string n(pn);
            p.path = pt; p.path_fs = pfs;
            int r;
            if ((r = need(m, (n + ".s").c_str(), kCh, &p.ps)) || (r = need(m, (n + ".b").c_str(), kCh, &p.pb))) return r;
            return DFB_OK;
        };
        DwPwParams p = mk(f.dec_emb, E / 4, ED, f.d3, E / 4, ED, c.conv_kt);
        if ((rc = blk("erb_dec.convt3", p)) || (rc = path(p, "erb_dec.conv3p", f.e3, e3_fs)) || (rc = run_dwpw<DW_S1>(s, p, B, pw_sw))) return rc;
        p = mk(f.d3, E / 4, ED, f.d2, E / 2, (int64_t)E / 2 * kCh, 1);
        if ((rc = blk("erb_dec.convt2", p)) || (rc = path(p, "erb_dec.conv2p", f.e2, (int64_t)E / 4 * kCh)) || (rc = run_dwpw<DW_T2>(s, p, B, pw_sw))) return rc;
        const float *ps, *pb, *w, *bb;
        if ((rc = need(m, "erb_dec.conv0p.s", kCh, &ps)) || (rc = need(m, "erb_dec.conv0p.b", kCh, &pb)) ||
            (rc = need(m, "erb_dec.conv0_out.w", c.conv_kt * 3 * kCh, &w)) || (rc = need(m, "erb_dec.conv0_out.b", 1, &bb)))
            return rc;
        p = mk(f.d2, E / 2, (int64_t)E / 2 * kCh, f.d1, E, (int64_t)E * kCh, 1);
        if ((rc = blk("erb_dec.convt1", p)) || (rc = path(p, "erb_dec.conv1p", f.e1, (int64_t)E / 2 * kCh))) return rc;
        // kt = 1 models on the tensor-core path: the mask head is evaluated in convt1's epilogue and d1 never leaves the SM
        const bool fused_mask = pw_sw && c.conv_kt == 1 && 128 % E == 0;
        if (fused_mask) {
            p.mk_e0 = f.e0; p.mk_ps = ps; p.mk_pb = pb; p.mk_w = w; p.mk_bias = bb; p.mk_out = d_m;
            p.out = nullptr;
            m->dbg.erase("d1");
        }
        if ((rc = run_dwpw<DW_T2>(s, p, B, pw_sw))) return rc;
        if (fused_mask) return finish();
        static PerDeviceOnce attr_once;
        int smem = (kMaskWarps * 2 * (E + 2) * kMaskLd + c.conv_kt * 3 * kCh) * 4;
        if (auto once_guard = attr_once.first()) {  // sized for the largest supported configuration (nb_erb 64, kt 2)
            DFB_CUDA(cudaFuncSetAttribute(k_mask_out, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          (kMaskWarps * 2 * (64 + 2) * kMaskLd + 2 * 3 * kCh) * 4));
        }
        int per_cta = kMaskWarps * kMaskChunk;
        dim3 grid((unsigned)((T + per_cta - 1) / per_cta), (unsigned)B);
        DFB_PROF("k_mask_out", s);
        k_mask_out<<<grid, 32 * kMaskWarps, smem, s>>>(f.e0, f.d1, ps, pb, w, bb, d_m, T, E, c.conv_kt);
        DFB_LAUNCH_CHECK();
    }
    return finish();
}

// ------------------------------------------------------------------ DeepFilterNet v1 ----
// deepfilternet.py:64-279.  Same kernels as the other models where the layer shapes coincide (input convs, separable conv
// blocks, GRU recurrence + projections, mask head); what differs is expressed around them:
//   * convkxf pads (k - 1 - lookahead, lookahead) frames inside the conv (modules.py:151-154): k_conv_in with tp_min =
//     -lookahead, the depthwise prologue with p.lookahead
//   * pathway convs are full 1x1 convs (depthwise 1x1 + 1x1 + BN + ReLU): the separable kernel with a one-tap depthwise
//   * decoder transposed convs have two time taps (reversed on upload)
//   * GroupedLinear (bias, shuffle) / GroupedGRU (G = 8, shuffle between layers, add_outputs): FFMA grouped linear with bias;
//     every GroupedGRULayer runs as ONE dense H-wide recurrence with block-diagonal weights (the shuffle of its input folded
//     into W_ih), the re-orderings and the sum of layer outputs are k_gather_sum passes
//   * df_fc_out is a dense H -> nb_df * 2 O linear (BF16x3 GEMM), tanh and the 1x1 pathway conv are added by k_convp_v1
//   * DfOp blends the deep-filtered DF bins with the masked spectrum by alpha (apply kernel)
// One window = the whole signal (pick_chunk): the in-conv look-ahead makes the zero padding at the END of the signal part of
// every layer, which a window that stops short of it cannot reproduce.
static int forward_v1(dfb_model *m, Arena &arena, const float *d_feat_erb, const float *d_feat_spec, int B, int T,
                      float *d_m, float *d_coefs, float *d_lsnr, float *d_alpha, cudaStream_t s_in, ChunkCtx *cx) {
    const dfb_model_config &c = m->cfg;
    if (cx && (cx->Rc != 0 || cx->have_state)) return fail(DFB_ERR_UNSUPPORTED, "DeepFilterNet v1 runs as one window per signal");
    const int Tsx = cx ? cx->Tsx : T, Tx = cx ? cx->Tx : T;
    static const bool serial = getenv("DFB_SERIAL") && atoi(getenv("DFB_SERIAL"));
    dfb_model::Lane &L = m->lanes[cx ? cx->lane : 0];
    cudaStream_t s = serial ? s_in : L.hi, sa = serial ? s_in : L.aux;
    if (!serial) {
        DFB_CUDA(cudaEventRecord(L.ev_in, s_in));
        DFB_CUDA(cudaStreamWaitEvent(s, L.ev_in, 0));
    }
    const int64_t M = (int64_t)B * T;
    const int E = c.nb_erb, Fd = c.nb_df, H = c.emb_hidden, O2 = 2 * c.df_order, kt = c.conv_kt;
    int rc;
    FwdBufsV1 f{};
    fwd_plan_v1(c, (size_t)M, &arena, &f);
    if (!f.scr_lo) return fail(DFB_ERR_OOM, "forward workspace exhausted for %lld frames", (long long)M);
    m->dbg.clear();
    m->dbg["e0"] = {f.e0, M * E * kCh}; m->dbg["e1"] = {f.e1, M * (E / 2) * kCh}; m->dbg["e2"] = {f.e2, M * (E / 4) * kCh};
    m->dbg["e3"] = {f.e3, M * (E / 4) * kCh}; m->dbg["c0"] = {f.c0, M * Fd * kCh}; m->dbg["c1"] = {f.c1, M * (Fd / 2) * kCh};
    m->dbg["cemb"] = {f.cemb, M * H}; m->dbg["emb_in"] = {f.emb, M * H}; m->dbg["emb"] = {f.embo, M * H};
    m->dbg["dec_emb"] = {f.dec, M * H}; m->dbg["d3"] = {f.d3, M * (E / 4) * kCh}; m->dbg["d2"] = {f.d2, M * (E / 2) * kCh};
    m->dbg["d1"] = {f.d1, M * E * kCh}; m->dbg["dfc"] = {f.dfc, M * H}; m->dbg["y0"] = {f.y[0], M * H};
    const bool tc = m->conv_tc != 0;
    const float *ones, *zeros;
    if ((rc = need(m, "v1.ones", kCh, &ones)) || (rc = need(m, "v1.zeros", kCh, &zeros))) return rc;
    auto table = [&](const char *name, int n, const int **out) -> int {
        const float *t;
        int r = need(m, name, n, &t);
        *out = reinterpret_cast<const int *>(t);
        return r;
    };
    const int *idx_c1, *idx_e3, *idx_shuf, *idx_id, *idx_dec, *idx_gshuf;
    if ((rc = table("v1.idx_c1", Fd / 2 * kCh, &idx_c1)) || (rc = table("v1.idx_e3", H, &idx_e3)) || (rc = table("v1.idx_shuf", H, &idx_shuf)) ||
        (rc = table("v1.idx_id", H, &idx_id)) || (rc = table("v1.idx_dec", H, &idx_dec)) || (rc = table("v1.idx_gshuf", H, &idx_gshuf)))
        return rc;
    auto gather = [&](cudaStream_t st, int n, const float *const *src, const int64_t *ld, const int *const *idx, int K, int relu,
                      float *out, unsigned short *hi, unsigned short *lo) -> int {
        GatherParams g{};
        for (int i = 0; i < n; i++) { g.src[i] = src[i]; g.ld[i] = ld[i]; g.idx[i] = idx[i]; }
        g.n = n; g.out = out; g.ldo = K; g.hi = hi; g.lo = lo; g.ldp = K; g.K = K; g.relu = relu;
        DFB_PROF("k_gather_sum", st);
        k_gather_sum<<<(unsigned)M, 256, 0, st>>>(g);
        DFB_LAUNCH_CHECK();
        return DFB_OK;
    };
    // separable block `name`: depthwise (kt x 3, look-ahead la) -> 1x1 -> BN -> ReLU, input = in (+ path)
    auto block = [&](cudaStream_t st, const char *name, int mode, const float *in, int Fin, float *out, int Fout, int bkt, int la,
                     const float *path) -> int {
        DwPwParams p{};
        std::string n(name);
        int r;
        if ((r = need(m, (n + ".dw").c_str(), bkt * 3 * kCh, &p.dw)) || (r = need(m, (n + ".pw").c_str(), kCh * kCh, &p.pw)) ||
            (r = need(m, (n + ".b").c_str(), kCh, &p.bias)))
            return r;
        p.in = in; p.Fin = Fin; p.in_fs = (int64_t)Fin * kCh; p.out = out; p.Fout = Fout; p.out_fs = (int64_t)Fout * kCh; p.kt = bkt; p.T = T;
        p.lookahead = la;
        if (path) { p.path = path; p.path_fs = p.in_fs; p.ps = ones; p.pb = zeros; }   // the pathway tensor is already >= 0
        // tensor-core version where it is built: no look-ahead, transposed blocks with one time tap only
        const float *w_sw = nullptr;
        if (tc && la == 0 && !(mode == DW_T2 && bkt != 1) && (r = need(m, (n + ".pw_sw").c_str(), kCh * kCh, &w_sw))) return r;
        if (mode == DW_S1) return run_dwpw<DW_S1>(st, p, B, w_sw);
        if (mode == DW_S2) return run_dwpw<DW_S2>(st, p, B, w_sw);
        return run_dwpw<DW_T2>(st, p, B, w_sw);
    };
    // ---- encoder, deepfilternet.py:122-141
    DFB_CUDA(cudaEventRecord(L.ev_fork_enc, s));
    DFB_CUDA(cudaStreamWaitEvent(sa, L.ev_fork_enc, 0));
    {
        const float *w, *bb;
        if ((rc = need(m, "enc.erb_conv0.w", c.inp_kt * 3 * kCh, &w)) || (rc = need(m, "enc.erb_conv0.b", kCh, &bb))) return rc;
        dim3 grid((unsigned)((T + kInFrames - 1) / kInFrames), (unsigned)B);
        const int la = c.conv_lookahead > 0 ? 1 : 0;
        {
            DFB_PROF("k_conv_in[erb_conv0]", s);
            k_conv_in<1><<<grid, 256, (kInFrames + c.inp_kt - 1) * (E + 2) * 4, s>>>(d_feat_erb, w, bb, f.e0, T, E, c.inp_kt, la, Tsx, Tx, -la);
            DFB_LAUNCH_CHECK();
        }
        if ((rc = need(m, "enc.df_conv0.w", c.inp_kt * 3 * 2 * kCh, &w)) || (rc = need(m, "enc.df_conv0.b", kCh, &bb))) return rc;
        DFB_PROF("k_conv_in[df_conv0]", sa);
        k_conv_in<2><<<grid, 256, (kInFrames + c.inp_kt - 1) * (Fd + 2) * 2 * 4, sa>>>(d_feat_spec, w, bb, f.c0, T, Fd, c.inp_kt, c.conv_lookahead,
                                                                                      Tsx, Tx, -c.conv_lookahead);
        DFB_LAUNCH_CHECK();
    }
    if ((rc = block(sa, "enc.df_conv1", DW_S2, f.c0, Fd, f.c1, Fd / 2, kt, 0, nullptr))) return rc;
    {   // cemb = df_fc_emb(c1 channel-major), pre-shuffle order
        const float *src[1] = {f.c1}; const int64_t ld[1] = {(int64_t)Fd / 2 * kCh}; const int *ix[1] = {idx_c1};
        if ((rc = gather(sa, 1, src, ld, ix, Fd / 2 * kCh, 0, f.c1g, nullptr, nullptr))) return rc;
        const float *w, *bb;
        const int I = Fd / 2 * kCh;
        if ((rc = need(m, "enc.df_fc_emb.gl", (int64_t)I * H / c.g_df_fc_emb, &w)) || (rc = need(m, "enc.df_fc_emb.bias", H, &bb))) return rc;
        if ((rc = run_gl(sa, f.c1g, I, w, bb, nullptr, 0, f.cemb, H, M, c.g_df_fc_emb, I, H, ACT_NONE))) return rc;
    }
    DFB_CUDA(cudaEventRecord(L.ev_join_enc, sa));
    if ((rc = block(s, "enc.erb_conv1", DW_S2, f.e0, E, f.e1, E / 2, kt, c.conv_lookahead > 1 ? 1 : 0, nullptr)) ||
        (rc = block(s, "enc.erb_conv2", DW_S2, f.e1, E / 2, f.e2, E / 4, kt, c.conv_lookahead > 2 ? 1 : 0, nullptr)) ||
        (rc = block(s, "enc.erb_conv3", DW_S1, f.e2, E / 4, f.e3, E / 4, kt, 0, nullptr)))
        return rc;
    DFB_CUDA(cudaStreamWaitEvent(s, L.ev_join_enc, 0));
    {   // emb = e3 (channel-major flatten) + shuffle(cemb)
        const float *src[2] = {f.e3, f.cemb}; const int64_t ld[2] = {H, H}; const int *ix[2] = {idx_e3, idx_shuf};
        if ((rc = gather(s, 2, src, ld, ix, H, 0, f.emb, f.emb_hi, f.emb_lo))) return rc;
    }
    // GroupedGRU: layer l as a dense recurrence, out = sum_l shuffle(y_l) (l < last) + y_last
    auto ggru = [&](cudaStream_t st, const char *name, int layers, const float *x, unsigned short *x_hi, unsigned short *x_lo, float **y,
                    unsigned short **y_hi, unsigned short **y_lo, float *xproj, float *hbase, float *out, unsigned short *out_hi,
                    unsigned short *out_lo) -> int {
        const float *cur = x;
        unsigned short *ch = x_hi, *cl = x_lo;
        for (int l = 0; l < layers; l++) {
            const std::string nm = std::string(name) + ".g" + std::to_string(l);
            GruChunk ck{hbase ? hbase + (int64_t)l * B * H : nullptr, false, 0};
            bool ok = false;
            int r = run_gru(m, st, nm.c_str(), 1, H, cur, H, nullptr, y[l], xproj, nullptr, B, T, ch, cl, f.scr_hi, f.scr_lo, 0, y_hi[l], y_lo[l], &ok,
                            hbase ? &ck : nullptr);
            if (r) return r;
            cur = y[l]; ch = y_hi[l]; cl = y_lo[l];
        }
        const float *src[3]; int64_t ld[3]; const int *ix[3];
        for (int l = 0; l < layers; l++) { src[l] = y[l]; ld[l] = H; ix[l] = l == layers - 1 ? idx_id : idx_gshuf; }
        return gather(st, layers, src, ld, ix, H, 0, out, out_hi, out_lo);
    };
    if (c.enc_gru_layers > 3 || c.df_gru_layers > 2) return fail(DFB_ERR_UNSUPPORTED, "DeepFilterNet v1: more GRU layers than built (3 / 2)");
    if ((rc = ggru(s, "enc.emb_gru", c.enc_gru_layers, f.emb, f.emb_hi, f.emb_lo, f.y, f.y_hi, f.y_lo, f.xproj, cx ? cx->h_enc : nullptr, f.embo,
                   f.embo_hi, f.embo_lo)))
        return rc;
    if (d_lsnr) {
        const float *lw, *lb;
        if ((rc = need(m, "enc.lsnr.w", H, &lw)) || (rc = need(m, "enc.lsnr.b", 1, &lb))) return rc;
        if ((rc = run_gl(s, f.embo, H, lw, lb, nullptr, 0, d_lsnr, 1, M, 1, H, 1, ACT_SIGMOID, c.lsnr_scale, c.lsnr_offset))) return rc;
    }
    DFB_CUDA(cudaEventRecord(L.ev_fork, s));
    if (!serial) { s = L.dhi; sa = L.daux; DFB_CUDA(cudaStreamWaitEvent(s, L.ev_fork, 0)); }
    DFB_CUDA(cudaStreamWaitEvent(sa, L.ev_fork, 0));
    // ---- DF decoder, deepfilternet.py:219-229 (auxiliary stream)
    {
        if ((rc = ggru(sa, "df_dec.df_gru", c.df_gru_layers, f.embo, f.embo_hi, f.embo_lo, f.z, f.z_hi, f.z_lo, f.xproj2, cx ? cx->h_df : nullptr, f.dfc,
                       f.dfc_hi, f.dfc_lo)))
            return rc;
        if (d_alpha) {
            const float *aw, *ab;
            if ((rc = need(m, "df_dec.df_fc_a.w", H, &aw)) || (rc = need(m, "df_dec.df_fc_a.b", 1, &ab))) return rc;
            if ((rc = run_gl(sa, f.dfc, H, aw, ab, nullptr, 0, d_alpha, 1, M, 1, H, 1, ACT_SIGMOID))) return rc;
        }
        const float *w_t, *bb, *w_hi, *w_lo;
        const int N = Fd * O2;
        if ((rc = need(m, "df_dec.df_fc_out.w_t", (int64_t)H * N, &w_t)) || (rc = need(m, "df_dec.df_fc_out.b", N, &bb))) return rc;
        rc = DFB_ERR_UNSUPPORTED;
        if (m->proj_tc && m->get("df_dec.df_fc_out.w_hi")) {
            if ((rc = need(m, "df_dec.df_fc_out.w_hi", (int64_t)H * N / 2, &w_hi)) || (rc = need(m, "df_dec.df_fc_out.w_lo", (int64_t)H * N / 2, &w_lo))) return rc;
            rc = launch_gemm_bf16x3(sa, f.dfc_hi, f.dfc_lo, H, w_hi, w_lo, bb, d_coefs, N, M, N, H);
        }
        if (rc == DFB_ERR_UNSUPPORTED) rc = run_gl(sa, f.dfc, H, w_t, bb, nullptr, 0, d_coefs, N, M, 1, H, N, ACT_NONE);
        if (rc) return rc;
        const float *pw, *pb;
        if ((rc = need(m, "df_dec.df_convp.w", kCh * O2, &pw)) || (rc = need(m, "df_dec.df_convp.b", O2, &pb))) return rc;
        const long long rows = (long long)M * Fd;
        DFB_PROF("k_convp_v1", sa);
        k_convp_v1<10><<<(unsigned)((rows + 127) / 128), 128, 0, sa>>>(f.c0, pw, pb, d_coefs, rows);
        DFB_LAUNCH_CHECK();
    }
    DFB_CUDA(cudaEventRecord(L.ev_join, sa));
    // ---- ERB decoder, deepfilternet.py:179-189
    {
        const float *w, *bb;
        if ((rc = need(m, "erb_dec.fc_emb.gl", (int64_t)H * H / c.g_erb_in, &w)) || (rc = need(m, "erb_dec.fc_emb.bias", H, &bb))) return rc;
        if ((rc = run_gl(s, f.embo, H, w, bb, nullptr, 0, f.dec_old, H, M, c.g_erb_in, H, H, ACT_RELU))) return rc;
        const float *src[1] = {f.dec_old}; const int64_t ld[1] = {H}; const int *ix[1] = {idx_dec};
        if ((rc = gather(s, 1, src, ld, ix, H, 0, f.dec, nullptr, nullptr))) return rc;
        if ((rc = block(s, "erb_dec.conv3p", DW_S1, f.e3, E / 4, f.p3, E / 4, 1, 0, nullptr)) ||
            (rc = block(s, "erb_dec.conv2p", DW_S1, f.e2, E / 4, f.p2, E / 4, 1, 0, nullptr)) ||
            (rc = block(s, "erb_dec.conv1p", DW_S1, f.e1, E / 2, f.p1, E / 2, 1, 0, nullptr)) ||
            (rc = block(s, "erb_dec.conv0p", DW_S1, f.e0, E, f.p0, E, 1, 0, nullptr)))
            return rc;
        if ((rc = block(s, "erb_dec.convt3", DW_S1, f.dec, E / 4, f.d3, E / 4, kt, 0, f.p3)) ||
            (rc = block(s, "erb_dec.convt2", DW_T2, f.d3, E / 4, f.d2, E / 2, kt, 0, f.p2)) ||
            (rc = block(s, "erb_dec.convt1", DW_T2, f.d2, E / 2, f.d1, E, kt, 0, f.p1)))
            return rc;
        if ((rc = need(m, "erb_dec.conv0_out.w", kt * 3 * kCh, &w)) || (rc = need(m, "erb_dec.conv0_out.b", 1, &bb))) return rc;
        static PerDeviceOnce attr_once;
        const int smem = (kMaskWarps * 2 * (E + 2) * kMaskLd + kt * 3 * kCh) * 4;
        if (auto once_guard = attr_once.first()) {
            DFB_CUDA(cudaFuncSetAttribute(k_mask_out, cudaFuncAttributeMaxDynamicSharedMemorySize, (kMaskWarps * 2 * (64 + 2) * kMaskLd + 2 * 3 * kCh) * 4));
        }
        const int per_cta = kMaskWarps * kMaskChunk;
        dim3 grid((unsigned)((T + per_cta - 1) / per_cta), (unsigned)B);
        DFB_PROF("k_mask_out", s);
        k_mask_out<<<grid, 32 * kMaskWarps, smem, s>>>(f.p0, f.d1, ones, zeros, w, bb, d_m, T, E, kt);
        DFB_LAUNCH_CHECK();
    }
    DFB_CUDA(cudaStreamWaitEvent(s, L.ev_join, 0));
    if (!serial) {
        DFB_CUDA(cudaEventRecord(L.ev_out, s));
        DFB_CUDA(cudaStreamWaitEvent(s_in, L.ev_out, 0));
    }
    return DFB_OK;
}

// Chunk pipeline of dfb_enhance / dfb_enhance_host: signals of at least 64 * chunks frames are cut into >= `chunks` time
// chunks (device-pointer / host-pointer entry point); lanes = 2 overlaps the encoder phase of chunk c + 1 with the decoder
// phase of chunk c, lanes = 1 runs the chunks back to back.  Defaults auto / 4 / 2 (DFB_DEVICE_CHUNKS, DFB_HOST_CHUNKS,
// DFB_LANES at dfb_model_create); device_chunks = 0 (auto) is 3 chunks up to 8 streams, 2 up to 256, else 1.
extern "C" int dfb_model_set_chunking(dfb_model *m, int device_chunks, int host_chunks, int lanes) {
    if (!m || device_chunks < 0 || host_chunks < 1 || lanes < 1 || lanes > 2) return fail(DFB_ERR_INVALID, "bad chunking parameters");
    m->dev_chunks = device_chunks; m->host_chunks = host_chunks; m->n_lanes = lanes;
    return DFB_OK;
}

// The workspace is sized from the model's band layout but the DSP kernels index with the state's: they must agree.
static int check_state(const dfb_model *m, const dfb_state *st) {
    if (m->device != st->device) return fail(DFB_ERR_INVALID, "model and state live on different devices");
    if (m->cfg.nb_df > st->tb.F)
        return fail(DFB_ERR_INVALID, "nb_df = %d exceeds the %d frequency bins of fft_size %d", m->cfg.nb_df, st->tb.F, st->fft);
    if (st->tb.E != m->cfg.nb_erb)
        return fail(DFB_ERR_INVALID, "DF state has %d ERB bands, the model was built for %d", st->tb.E, m->cfg.nb_erb);
    if (!m->erb_widths.empty())
        for (int i = 0; i < m->cfg.nb_erb; i++)
            if (m->erb_widths[i] != st->erb[i])
                return fail(DFB_ERR_INVALID, "DF state's ERB band %d is %lld bins wide, the model was built for %lld", i,
                            (long long)st->erb[i], (long long)m->erb_widths[i]);
    return DFB_OK;
}

// The time-chunked executor carries one hop of STFT memory and one frame of overlap-add tail per stream, which is the
// whole state only when hop == fft / 2 (every DeepFilterNet config).
static int check_half_overlap(const dfb_state *st) {
    if (st->hop * 2 != st->fft)
        return fail(DFB_ERR_UNSUPPORTED, "enhance / streaming need hop_size == fft_size / 2 (got fft_size %d, hop_size %d); "
                    "use analysis, DfNet.forward and synthesis for other hops", st->fft, st->hop);
    return DFB_OK;
}

static int apply_mode(const dfb_model *m) { return m->cfg.model_kind == 3 ? 1 : 2; }   // v1 / v2 filter the masked spectrum
static void apply_options(const dfb_model *m, dfb::ApplyParams &p) {
    p.pf = m->post_filter; p.pf_beta = m->pf_beta; p.mask_only = m->mask_only;
}

// init_df(post_filter=..., mask_only=...) (df/enhance.py:101-187): the post filter of deepfilternet3.py:448-454 (beta =
// pf_beta) or, for DeepFilterNet2, Mask.pf on the ERB gains (modules.py:234-245, beta fixed at 0.02); mask_only = the
// model built with run_df = False (checkpoint.py:32): no deep filtering stage.
extern "C" int dfb_model_set_options(dfb_model *m, int post_filter, float pf_beta, int mask_only) {
    if (!m) return fail(DFB_ERR_INVALID, "null model");
    m->post_filter = post_filter ? 1 : 0;
    m->pf_beta = pf_beta;
    m->mask_only = mask_only ? 1 : 0;
    return DFB_OK;
}

static int apply_impl(dfb_model *m, dfb_state *st, const float *d_spec, const float *d_m, const float *d_coefs, const float *d_alpha,
                      int64_t B, int64_t T, float *d_spec_e, void *stream);
extern "C" int dfb_apply(dfb_model *m, dfb_state *st, const float *d_spec, const float *d_m, const float *d_coefs,
                         int64_t B, int64_t T, float *d_spec_e, void *stream) {
    if (m && m->cfg.model_kind == 1 && !m->mask_only)
        return fail(DFB_ERR_UNSUPPORTED, "DeepFilterNet v1 blends with df_alpha: use dfb_model_forward_full / dfb_enhance");
    return apply_impl(m, st, d_spec, d_m, d_coefs, nullptr, B, T, d_spec_e, stream);
}
static int apply_impl(dfb_model *m, dfb_state *st, const float *d_spec, const float *d_m, const float *d_coefs, const float *d_alpha,
                      int64_t B, int64_t T, float *d_spec_e, void *stream) {
    if (!m || !st || !d_spec || !d_m || !d_coefs || !d_spec_e) return fail(DFB_ERR_INVALID, "null argument");
    if (int rcs = check_state(m, st)) return rcs;
    DFB_CUDA(cudaSetDevice(m->device));
    dfb::ApplyParams p{};
    p.spec = (const float2 *)d_spec; p.m = d_m; p.coefs = d_coefs; p.audio = nullptr; p.spec_out = (float2 *)d_spec_e;
    p.Tf = (int)T; p.mode = apply_mode(m); p.nb_df = m->cfg.nb_df; p.order = m->cfg.df_order; p.lookahead = m->cfg.df_lookahead;
    p.alpha = d_alpha;
    apply_options(m, p);
    return launch_apply_synthesis(st, p, B, (cudaStream_t)stream);
}

extern "C" int dfb_model_forward_full(dfb_model *m, dfb_state *st, const float *d_spec, const float *d_feat_erb,
                                      const float *d_feat_spec, int64_t B, int64_t T, float *d_spec_e, float *d_m,
                                      float *d_lsnr, float *d_coefs, float *d_alpha, void *stream) {
    if (!m || !st || !d_spec || !d_feat_erb || !d_feat_spec || !d_spec_e) return fail(DFB_ERR_INVALID, "null argument");
    if (int rcs = check_state(m, st)) return rcs;
    DFB_CUDA(cudaSetDevice(m->device));
    const int64_t M = B * T;
    const int O2 = 2 * m->cfg.df_order;
    if (B <= 0 || T <= 0) return DFB_OK;
    if (B > 65535) return fail(DFB_ERR_INVALID, "more than 65535 streams per call");
    size_t extra = ((size_t)M * m->cfg.nb_erb + (size_t)M * m->cfg.nb_df * O2 + (size_t)M) * 4 + 8192;
    int rc = m->arena.reserve(fwd_plan(m->cfg, (size_t)M, nullptr, nullptr) + extra);
    if (rc) return rc;
    m->arena.reset();
    float *mm = d_m ? d_m : m->arena.take<float>((size_t)M * m->cfg.nb_erb);
    float *cc = d_coefs ? d_coefs : m->arena.take<float>((size_t)M * m->cfg.nb_df * O2);
    float *aa = d_alpha;
    if (!aa && m->cfg.model_kind == 1) aa = m->arena.take<float>((size_t)M);
    rc = forward_impl(m, m->arena, d_feat_erb, d_feat_spec, (int)B, (int)T, mm, cc, d_lsnr, aa, (cudaStream_t)stream);
    if (rc) { m->arena.reset(); return rc; }
    rc = apply_impl(m, st, d_spec, mm, cc, m->cfg.model_kind == 1 ? aa : nullptr, B, T, d_spec_e, stream);
    m->arena.reset();
    return rc;
}

extern "C" int64_t dfb_enhance_out_len(const dfb_state *st, int64_t T, int pad) {
    if (!st) return -1;
    return pad ? T : (T / st->hop) * st->hop;
}

// enhance(): df/enhance.py:206-250.  Streams are processed in groups so that the workspace stays
// below the model's workspace cap (64 GB by default; dfb_model_set_max_workspace / DFB_MAX_WORKSPACE_MB); streams
// are independent (per-channel state reset, pyDF/src/lib.rs:56-58).
extern "C" int dfb_model_set_max_workspace(dfb_model *m, int64_t bytes) {
    if (!m || bytes <= 0) return fail(DFB_ERR_INVALID, "bad workspace cap");
    m->max_workspace = (size_t)bytes;
    return DFB_OK;
}


// ============================================================== time-chunked executor ====
// enhance() (df/enhance.py:206-250) and the streaming API run the path in TIME CHUNKS with carried per-stream state
// (SURVEY.md Appendix D): memory is proportional to the chunk, not the signal; host copies of one chunk overlap the
// compute of the next; and the frame-incremental API of the reference (libDF/src/tract.rs:509-642) is the same code
// with a chunk of a few frames.  Per chunk the window [W0, d1) of DNN frames = kHalo already finished frames (their
// feed-forward activations are recomputed from the carried feature history; receptive field <= 6 frames) + the new
// frames [d0, d1); the recurrences run over the new frames only, from the carried hidden states.
struct StreamState {
    int B = 0;
    int64_t a1 = 0, d1 = 0, e1 = 0;     // frames analysed / through the DNN / emitted as audio so far (absolute)
    bool started = false, dnn_started = false;   // first analysis / first DNN chunk done (states are valid)
    float *slab = nullptr;              // one allocation holding everything below
    float *ana_mem = nullptr;           // [B][hop]       last input hop (streaming API; the batch path reads resident audio)
    float *erb_state = nullptr, *unit_state = nullptr;   // [B][E], [B][Fd]  EMA states of the feature normalisation
    float *h_enc = nullptr, *h_erb = nullptr, *h_df = nullptr;   // [layers][B][H]
    float *t_spec = nullptr, *t_fe = nullptr, *t_fs = nullptr;   // last Hf = kHalo + Lmax frames of spec / features, right aligned
    float *t_m = nullptr, *t_c = nullptr;                        // last kMcTail frames of m / coefs, right aligned
    float *t_l = nullptr;                                        // ... and of lsnr (stage gating)
    float *t_dec = nullptr;                                      // (conv_kt == 2) last kHalo frames of dec_emb
    int n_feat = 0, n_mc = 0, n_dec = 0;                         // valid frames in the tails
};
constexpr int kMcTail = 6;   // >= lag + 3 (see run_chunk)

struct ChunkGeom { int Lmax, lag, Hf; };
static ChunkGeom chunk_geom(const dfb_model_config &c) {
    ChunkGeom g;
    g.Lmax = c.conv_lookahead > c.df_lookahead ? c.conv_lookahead : c.df_lookahead;
    // DeepFilterNet2 filters the MASKED spectrum: frame t needs the masks of frames <= t + df_lookahead, so its audio
    // trails the DNN frames by df_lookahead (deepfilternet2.py:494-503)
    g.lag = c.model_kind != 3 ? c.df_lookahead : 0;
    g.Hf = kHalo + g.Lmax;
    return g;
}

static size_t state_floats(const dfb_model_config &c, const dfb_state *st, int B, size_t off[16]) {
    const ChunkGeom g = chunk_geom(c);
    const int E = c.nb_erb, Fd = c.nb_df, O2 = 2 * c.df_order, F = st->tb.F, ED = E / 4 * kCh;
    size_t n = 0;
    auto add = [&](int i, size_t k) { off[i] = n; n += (k + 63) & ~size_t(63); };
    add(0, (size_t)B * st->hop); add(1, (size_t)B * E); add(2, (size_t)B * Fd);
    add(3, (size_t)c.enc_gru_layers * B * c.emb_hidden); add(4, (size_t)c.erb_gru_layers * B * c.emb_hidden);
    add(5, (size_t)c.df_gru_layers * B * c.df_hidden);
    add(6, (size_t)B * g.Hf * 2 * F); add(7, (size_t)B * g.Hf * E); add(8, (size_t)B * g.Hf * 2 * Fd);
    add(9, (size_t)B * kMcTail * E); add(10, (size_t)B * kMcTail * Fd * O2);
    add(11, c.conv_kt > 1 ? (size_t)B * kHalo * ED : 0);
    add(12, (size_t)B * kMcTail);
    return n;
}
static void state_bind(StreamState &S, float *base, const size_t off[16], int B) {
    S.B = B; S.slab = base;
    S.ana_mem = base + off[0]; S.erb_state = base + off[1]; S.unit_state = base + off[2];
    S.h_enc = base + off[3]; S.h_erb = base + off[4]; S.h_df = base + off[5];
    S.t_spec = base + off[6]; S.t_fe = base + off[7]; S.t_fs = base + off[8];
    S.t_m = base + off[9]; S.t_c = base + off[10]; S.t_dec = base + off[11]; S.t_l = base + off[12];
    S.a1 = S.d1 = S.e1 = 0; S.started = S.dnn_started = false; S.n_feat = S.n_mc = S.n_dec = 0;
}

// last n frames of buf [B][T][fe] -> tail [B][cap][fe] (right aligned), and back into frames [dst_t, dst_t + n) of a buffer
static int save_tail(cudaStream_t s, const float *buf, int T, size_t fe, int n, float *tail, int cap, int B) {
    if (n <= 0) return DFB_OK;
    DFB_CUDA(cudaMemcpy2DAsync(tail + (size_t)(cap - n) * fe, sizeof(float) * fe * cap, buf + (size_t)(T - n) * fe, sizeof(float) * fe * T,
                               sizeof(float) * fe * n, B, cudaMemcpyDeviceToDevice, s));
    return DFB_OK;
}
static int load_tail(cudaStream_t s, float *buf, int T, size_t fe, int n, const float *tail, int cap, int dst_t, int B) {
    if (n <= 0) return DFB_OK;
    DFB_CUDA(cudaMemcpy2DAsync(buf + (size_t)dst_t * fe, sizeof(float) * fe * T, tail + (size_t)(cap - n) * fe, sizeof(float) * fe * cap,
                               sizeof(float) * fe * n, B, cudaMemcpyDeviceToDevice, s));
    return DFB_OK;
}

// bytes of workspace one window of Tw DNN frames needs per stream (features hold Tw + Lmax frames)
static size_t chunk_bytes_per_stream(const dfb_model_config &c, const dfb_state *st, int Tw) {
    const ChunkGeom g = chunk_geom(c);
    const int E = c.nb_erb, Fd = c.nb_df, O2 = 2 * c.df_order, F = st->tb.F;
    return (size_t)(Tw + g.Lmax) * (2 * F + E + 2 * Fd) * 4 + (size_t)Tw * (E + (size_t)Fd * O2 + 2) * 4 + fwd_plan(c, (size_t)Tw, nullptr, nullptr) +
           16384;
}

// Where the audio of one chunk comes from and goes to.
struct ChunkIO {
    const float *audio; int64_t audio_T, audio_stride;  // signal the analysis reads: T samples per row (row pitch audio_stride)
    int64_t audio_frame0;     // absolute frame index of the signal's first frame (0: resident whole signal; a0: streaming chunk)
    const float *init_mem;    // [B][hop] samples before audio[0] (streaming) or null (zeros)
    float *out; int64_t out_stride, out_len;
    int64_t out_sample0;      // absolute synthesis sample (frame * hop + i) that lands at out[0]
    float atten_lim;
    const float *lsnr_th;     // {min_db_thresh, max_db_erb_thresh, max_db_df_thresh} (tract.rs:658-672) or null: no gating
};

// One chunk: analyse frames [S.a1, a1n), run the DNN over [S.d1, d1n), emit audio of frames [S.e1, e1n).
// Tf_end: total frames of the stream when known (features / spectrum beyond it are zero), else -1.
// lane / pipelined: consecutive chunks of a batch call alternate between the model's two lanes (stream sets + arenas);
// chunk c starts when chunk c - 1 has finished its ENCODER phase and its decoder phase waits for chunk c - 1 to finish
// entirely, so encoder(c) overlaps decoder(c - 1).  `s` is the stream the chunk is enqueued on (the lane's main stream
// in the pipeline, the caller's stream otherwise).
static int run_chunk(dfb_model *m, dfb_state *st, StreamState &S, const ChunkIO &io, int64_t a1n, int64_t d1n, int64_t e1n,
                     cudaStream_t s, int lane = 0, bool pipelined = false) {
    Arena &arena = lane ? m->arena1 : m->arena;
    dfb_model::Lane &L = m->lanes[lane], &P = m->lanes[lane ^ 1];
    const bool have_prev = pipelined && S.started;
    if (have_prev) DFB_CUDA(cudaStreamWaitEvent(s, P.ev_fork, 0));   // previous chunk: features + encoder phase done
    const dfb_model_config &c = m->cfg;
    const ChunkGeom g = chunk_geom(c);
    const int B = S.B, E = c.nb_erb, Fd = c.nb_df, O2 = 2 * c.df_order, F = st->tb.F, hop = st->hop, ED = E / 4 * kCh;
    const int64_t W0 = S.d1 > kHalo ? S.d1 - kHalo : 0;
    const int Rc = (int)(S.d1 - W0), Tw = (int)(d1n - W0), Tsb = Tw + g.Lmax;
    const int n_hist = (int)(S.a1 - W0);                 // feature frames of the window that are already known
    const int n_new = (int)(a1n - S.a1), Tv = (int)(a1n - W0);
    if (Tw < Rc || n_hist < 0 || n_hist > S.n_feat || Tv > Tsb || Tsb <= 0)
        return fail(DFB_ERR_INVALID, "inconsistent chunk geometry");
    const bool run_dnn = d1n > S.d1;      // a short streaming call may only add look-ahead frames
    int rc;
    arena.reset();
    float *spec = arena.take<float>((size_t)B * Tsb * F * 2 + 2);
    float *fe = arena.take<float>((size_t)B * Tsb * E);
    float *fs = arena.take<float>((size_t)B * Tsb * Fd * 2);
    float *mm = arena.take<float>((size_t)B * (Tw + 1) * E);
    float *cc = arena.take<float>((size_t)B * (Tw + 1) * Fd * O2);
    float *ll = io.lsnr_th ? arena.take<float>((size_t)B * (Tw + 1)) : nullptr;
    float *aa = c.model_kind == 1 ? arena.take<float>((size_t)B * (Tw + 1)) : nullptr;   // df_alpha (v1)
    if (!cc || (c.model_kind == 1 && !aa)) return fail(DFB_ERR_OOM, "chunk workspace exhausted");
    // ---- features: carried history, then the new frames
    if ((rc = load_tail(s, spec, Tsb, (size_t)2 * F, n_hist, S.t_spec, g.Hf, 0, B)) || (rc = load_tail(s, fe, Tsb, E, n_hist, S.t_fe, g.Hf, 0, B)) ||
        (rc = load_tail(s, fs, Tsb, (size_t)2 * Fd, n_hist, S.t_fs, g.Hf, 0, B)))
        return rc;
    if (n_new > 0) {
        AnaWindow w{(int)(S.a1 - io.audio_frame0), n_new, n_hist, Tsb, io.audio_stride};
        if ((rc = launch_analysis(st, io.audio, B, io.audio_T, spec, fe, s, io.init_mem, &w))) return rc;
        if ((rc = launch_feat_norm(fe + (size_t)n_hist * E, E, E, spec + (size_t)n_hist * 2 * F, Fd, F, B, n_new, c.norm_alpha,
                                   S.started ? S.erb_state : nullptr, S.started ? S.unit_state : nullptr, fe + (size_t)n_hist * E,
                                   fs + (size_t)n_hist * 2 * Fd, s, Tsb, S.erb_state, S.unit_state)))
            return rc;
    }
    {   // carry the feature history right away: the next chunk may start as soon as this chunk's encoder is done
        const int nf = Tv < g.Hf ? Tv : g.Hf;
        // the feature buffers hold Tsb frames per stream of which the first Tv are valid: keep the last nf valid ones
        const size_t fes[3] = {(size_t)2 * F, (size_t)E, (size_t)2 * Fd};
        float *bufs[3] = {spec, fe, fs}, *tails[3] = {S.t_spec, S.t_fe, S.t_fs};
        for (int i = 0; i < 3; i++)
            DFB_CUDA(cudaMemcpy2DAsync(tails[i] + (size_t)(g.Hf - nf) * fes[i], sizeof(float) * fes[i] * g.Hf,
                                       bufs[i] + (size_t)(Tv - nf) * fes[i], sizeof(float) * fes[i] * Tsb, sizeof(float) * fes[i] * nf, B,
                                       cudaMemcpyDeviceToDevice, s));
        S.n_feat = nf;
    }
    // ---- DNN over the window
    if (run_dnn) {
    ChunkCtx cx{Rc, Tsb, Tv, S.h_enc, S.h_erb, S.h_df, S.dnn_started, c.conv_kt > 1 ? S.t_dec : nullptr, S.n_dec, lane,
                have_prev ? P.ev_done : nullptr};
    if ((rc = forward_impl(m, arena, fe, fs, B, Tw, mm, cc, ll, aa, s, &cx))) return rc;
    S.n_dec = cx.dec_tail_n;
    S.dnn_started = true;
    // the halo rows of m / coefs come from skipped recurrences: restore the last finished frames from the previous chunk
    // (the apply kernel re-synthesises frame e0 - 1 for its overlap-add tail; DFN2's masked taps reach 2 frames further back)
    if (Rc > 0 && S.n_mc > 0) {
        const int n = S.n_mc < Rc ? S.n_mc : Rc;
        if ((rc = load_tail(s, mm, Tw, E, n, S.t_m, kMcTail, Rc - n, B)) || (rc = load_tail(s, cc, Tw, (size_t)Fd * O2, n, S.t_c, kMcTail, Rc - n, B)))
            return rc;
        if (ll && (rc = load_tail(s, ll, Tw, 1, n, S.t_l, kMcTail, Rc - n, B))) return rc;
    }
    }
    // ---- apply + synthesis of frames [e0, e1n)
    if (run_dnn && e1n > S.e1) {
        dfb::ApplyParams p{};
        p.spec = (const float2 *)spec; p.m = mm; p.coefs = cc; p.audio = io.out; p.spec_out = nullptr;
        p.out_stride = io.out_stride; p.out_len = io.out_len;
        p.out_offset = io.out_sample0 - W0 * hop;     // g = t_window * hop + i - out_offset
        p.Tf = (int)(e1n - W0); p.spec_T = Tsb; p.Tv = Tv; p.mc_T = Tw; p.t_first = (int)(S.e1 - W0);
        p.mode = apply_mode(m); p.nb_df = Fd; p.order = c.df_order; p.lookahead = c.df_lookahead;
        p.atten_lim = io.atten_lim;
        p.alpha = aa;
        apply_options(m, p);
        if (ll) { p.lsnr = ll; p.th_min = io.lsnr_th[0]; p.th_erb = io.lsnr_th[1]; p.th_df = io.lsnr_th[2]; }
        if ((rc = launch_apply_synthesis(st, p, B, s))) return rc;
    }
    // ---- carry
    {
        if (run_dnn) {
            const int nm = Tw < kMcTail ? Tw : kMcTail;
            if ((rc = save_tail(s, mm, Tw, E, nm, S.t_m, kMcTail, B)) || (rc = save_tail(s, cc, Tw, (size_t)Fd * O2, nm, S.t_c, kMcTail, B))) return rc;
            if (ll && (rc = save_tail(s, ll, Tw, 1, nm, S.t_l, kMcTail, B))) return rc;
            S.n_mc = nm;
        }
    }
    (void)ED;
    if (pipelined) {
        if (!run_dnn) DFB_CUDA(cudaEventRecord(L.ev_fork, s));   // no forward pass recorded it
        DFB_CUDA(cudaEventRecord(L.ev_done, s));
    }
    S.a1 = a1n; S.d1 = d1n; if (run_dnn) S.e1 = e1n;
    S.started = true;
    return DFB_OK;
}

// Chunk length (new DNN frames per chunk) for B streams under the workspace cap; 0 when not even a short chunk fits.
static int pick_chunk(const dfb_model *m, const dfb_state *st, int64_t B, int64_t Tf, int min_chunks) {
    const size_t per_frame = chunk_bytes_per_stream(m->cfg, st, 1024) / 1024 + 1;   // bytes per stream and window frame
    const ChunkGeom g = chunk_geom(m->cfg);
    int64_t tw = (int64_t)(m->max_workspace / ((size_t)B * per_frame)) - g.Lmax - 8;
    int64_t tc = tw - kHalo;
    if (tc > Tf) tc = Tf;
    if (min_chunks > 1 && Tf >= (int64_t)min_chunks * 64) {
        const int64_t t2 = (Tf + min_chunks - 1) / min_chunks;
        if (t2 < tc) tc = t2;
    }
    if (m->cfg.model_kind == 1) return tw >= Tf ? (int)Tf : 0;   // DeepFilterNet v1: one window per signal (forward_v1)
    if (tc < 1) return 0;
    if (tc < Tf && tc < 32) return 0;   // a chunk this short wastes most of its window on the halo: use stream groups
    return (int)tc;
}
// Runs the chunk loop over `nb` streams whose padded signal d_x [nb][Tp] is resident (or becomes resident chunk by chunk:
// `before` / `after` are called around every chunk with the sample ranges it reads / has written).
struct ChunkHooks {
    // analysis of this chunk reads input samples [x0, x1) of every stream; output samples [y0, y1) have been written
    // `cs` is the stream the chunk's compute is enqueued on (must wait for the input / produces the output)
    std::function<int(int64_t x0, int64_t x1, cudaStream_t cs)> before;
    std::function<int(int64_t y0, int64_t y1, cudaStream_t cs)> after;
};

static int enhance_group(dfb_model *m, dfb_state *st, const float *d_x, int64_t nb, int64_t Tp, int64_t in_valid, int pad,
                         float lim, float *d_out, int64_t out_len, int tc, bool pipelined, cudaStream_t s, const ChunkHooks *hooks) {
    const dfb_model_config &c = m->cfg;
    const ChunkGeom g = chunk_geom(c);
    const int hop = st->hop, fft = st->fft;
    const int64_t Tf = Tp / hop;
    size_t off[16];
    const size_t nstate = state_floats(c, st, (int)nb, off);
    float *slab = m->aux_arena.take<float>(nstate);
    if (!slab) return fail(DFB_ERR_OOM, "stream state arena exhausted");
    StreamState S;
    state_bind(S, slab, off, (int)nb);
    int rc = DFB_OK;
    const int64_t delay = pad ? fft - hop : 0;
    if (tc >= Tf) pipelined = false;      // a single chunk
    cudaEvent_t ev_call = nullptr;
    if (pipelined) {  // both lanes start after everything the caller has enqueued so far
        DFB_CUDA(cudaEventCreateWithFlags(&ev_call, cudaEventDisableTiming));
        DFB_CUDA(cudaEventRecord(ev_call, s));
        DFB_CUDA(cudaStreamWaitEvent(m->lanes[0].main, ev_call, 0));
        DFB_CUDA(cudaStreamWaitEvent(m->lanes[1].main, ev_call, 0));
    }
    int chunk = 0, last_lane = 0;
    // Host path: the first chunk's H2D copy and the last chunk's D2H copy are the only ones nothing overlaps, so both end
    // chunks are half as long as the others (128 x 10 s in 4 chunks: 250 / 250 / 250 / 252 frames -> 125 / 250 / 250 / 250 / 127).
    const bool taper = hooks && pipelined && tc < Tf && tc >= 64;
    while (S.d1 < Tf) {
        int64_t step = tc;
        if (taper) {
            const int64_t left = Tf - S.d1;
            if (chunk == 0) step = tc / 2;
            else if (left <= tc + tc / 2 && left - tc / 2 >= tc / 4) step = left - tc / 2;   // leaves a half-length last chunk
        }
        const int64_t d1n = S.d1 + step < Tf ? S.d1 + step : Tf;
        const int64_t a1n = d1n + g.Lmax < Tf ? d1n + g.Lmax : Tf;
        const int64_t e1n = d1n == Tf ? Tf : d1n - g.lag;
        const int lane = pipelined ? (chunk & 1) : 0;
        cudaStream_t cs = pipelined ? m->lanes[lane].main : s;
        if (hooks && hooks->before) {
            int64_t x0 = S.a1 * hop, x1 = a1n * hop;
            if (x1 > in_valid) x1 = in_valid;
            if (x0 < x1 && (rc = hooks->before(x0, x1, cs))) break;
        }
        const int64_t e0 = S.e1;
        ChunkIO io{d_x, Tp, Tp, 0, nullptr, d_out, out_len, out_len, delay, lim, nullptr};
        if ((rc = run_chunk(m, st, S, io, a1n, d1n, e1n > S.e1 ? e1n : S.e1, cs, lane, pipelined))) break;
        if (hooks && hooks->after) {
            int64_t y0 = e0 * hop - delay, y1 = S.e1 * hop - delay;
            if (y0 < 0) y0 = 0;
            if (y1 > out_len) y1 = out_len;
            if (y0 < y1 && (rc = hooks->after(y0, y1, cs))) break;
        }
        last_lane = lane;
        chunk++;
    }
    if (pipelined) {  // hand the result back to the caller's stream (the last chunk finishes after all earlier ones)
        if (chunk > 0) cudaStreamWaitEvent(s, m->lanes[last_lane].ev_done, 0);
        if (chunk > 1) cudaStreamWaitEvent(s, m->lanes[last_lane ^ 1].ev_done, 0);
        if (rc) cudaDeviceSynchronize();
        cudaEventDestroy(ev_call);
    }
    return rc;
}

// enhance(): df/enhance.py:206-250.  Time chunks (above) inside stream groups: a group is as many streams as fit the
// workspace cap with a reasonable chunk; streams are independent (per-channel state reset, pyDF/src/lib.rs:56-58).
static int enhance_plan(dfb_model *m, dfb_state *st, int64_t B, int64_t Tf, int min_chunks, int64_t *group_out, int *tc_out,
                        bool *pipelined_out) {
    // two lanes (DFB_LANES=1 turns the chunk pipeline off): each lane's arena may take half of the workspace cap
    static const bool serial = getenv("DFB_SERIAL") && atoi(getenv("DFB_SERIAL"));
    const bool pipelined = m->n_lanes == 2 && !serial && min_chunks > 1 && Tf >= (int64_t)min_chunks * 64;
    const size_t cap = m->max_workspace;
    if (pipelined) m->max_workspace = cap / 2;
    int64_t group = B > 65535 ? 65535 : B;
    int tc = 0;
    while ((tc = pick_chunk(m, st, group, Tf, min_chunks)) == 0) {
        if (group == 1) { m->max_workspace = cap; return fail(DFB_ERR_OOM, "workspace cap of %zu bytes is too small for a single stream", cap); }
        group = (group + 1) / 2;
    }
    m->max_workspace = cap;
    *group_out = group; *tc_out = tc; *pipelined_out = pipelined && tc < Tf;
    const ChunkGeom g = chunk_geom(m->cfg);
    const size_t bytes = chunk_bytes_per_stream(m->cfg, st, tc + kHalo) * (size_t)group + ((size_t)g.Lmax << 10) + (2 << 20);
    int rc = m->arena.reserve(bytes);
    if (!rc && *pipelined_out) rc = m->arena1.reserve(bytes);
    return rc;
}

extern "C" int dfb_enhance(dfb_model *m, dfb_state *st, const float *d_audio, int64_t B, int64_t T, int pad,
                           float atten_lim_db, float *d_out, void *stream) {
    if (!m || !st || !d_audio || !d_out) return fail(DFB_ERR_INVALID, "null argument");
    if (B <= 0 || T <= 0) return fail(DFB_ERR_INVALID, "empty input");
    if (int rcs = check_state(m, st)) return rcs;
    if (int rch = check_half_overlap(st)) return rch;
    DFB_CUDA(cudaSetDevice(m->device));
    cudaStream_t s = (cudaStream_t)stream;
    const int hop = st->hop, fft = st->fft;
    // pad = True appends fft zeros (enhance.py:230-233): Tf = (T + fft) / hop
    const int64_t Tp = pad ? T + fft : T;
    const int64_t Tf = Tp / hop;
    if (Tf <= 0) return fail(DFB_ERR_INVALID, "input shorter than one hop");
    const int64_t out_len = dfb_enhance_out_len(st, T, pad);
    int64_t group = 0;
    int tc = 0, rc;
    bool pipelined = false;
    // measured (profiles/r02_chunk_sweep.txt, 128 x 10 s): cutting a device-resident batch into pipelined chunks costs more
    // (persistent kernels re-pay their prologues, short grids leave partial waves: 13.6 -> 14.1 ms for 4 chunks) than the
    // overlap of encoder and decoder phases gains -- except for a few streams, where everything is latency bound
    // (batch 1: RTF 0.00046 -> 0.00040 with 3 chunks).  0 = that policy.
    // (round 2, after the DSP kernels got shorter: 2 chunks gain 17 % at 32 x 10 s, 1.3 % at 128 x 10 s, 1 % at 256 x 10 s _ll
    // and lose 1 % at 512 x 10 s)
    const int dev_chunks = m->dev_chunks > 0 ? m->dev_chunks : (B <= 8 ? 3 : (B <= 256 ? 2 : 1));
    if ((rc = enhance_plan(m, st, B, Tf, dev_chunks, &group, &tc, &pipelined))) return rc;
    const float lim = (atten_lim_db > 0.f) ? powf(10.f, -atten_lim_db / 20.f) : 0.f;
    size_t off[16];
    if ((rc = m->aux_arena.reserve((state_floats(m->cfg, st, (int)group, off) + (pad ? (size_t)group * Tp : 0)) * sizeof(float) + 8192))) return rc;
    for (int64_t b0 = 0; b0 < B && !rc; b0 += group) {
        const int64_t nb = (B - b0 < group) ? B - b0 : group;
        const float *x = d_audio + b0 * T;
        m->aux_arena.reset();
        float *xp = pad ? m->aux_arena.take<float>((size_t)nb * Tp) : nullptr;
        if (pad) {
            rc = cudaMemsetAsync(xp, 0, sizeof(float) * nb * Tp, s) != cudaSuccess ||
                 cudaMemcpy2DAsync(xp, sizeof(float) * Tp, x, sizeof(float) * T, sizeof(float) * T, nb, cudaMemcpyDeviceToDevice, s) != cudaSuccess
                     ? fail(DFB_ERR_CUDA, "padding copy failed") : DFB_OK;
            x = xp;
        }
        if (!rc) rc = enhance_group(m, st, x, nb, Tp, Tp, pad, lim, d_out + b0 * out_len, out_len, tc, pipelined, s, nullptr);
    }
    m->arena.reset();
    m->arena1.reset();
    return rc;
}

// Host buffers: the batch is staged chunk by chunk -- the H2D copy of chunk c + 1 and the D2H copy of chunk c - 1 run on
// their own streams (both copy engines) while chunk c computes.
extern "C" int dfb_enhance_host(dfb_model *m, dfb_state *st, const float *h_audio, int64_t B, int64_t T, int pad,
                                float atten_lim_db, float *h_out) {
    if (!m || !st || !h_audio || !h_out) return fail(DFB_ERR_INVALID, "null argument");
    if (B <= 0 || T <= 0) return fail(DFB_ERR_INVALID, "empty input");
    if (int rcs = check_state(m, st)) return rcs;
    if (int rch = check_half_overlap(st)) return rch;
    DFB_CUDA(cudaSetDevice(m->device));
    const int hop = st->hop, fft = st->fft;
    const int64_t Tp = pad ? T + fft : T, Tf = Tp / hop;
    if (Tf <= 0) return fail(DFB_ERR_INVALID, "input shorter than one hop");
    const int64_t out_len = dfb_enhance_out_len(st, T, pad);
    int64_t group = 0;
    int tc = 0, rc;
    bool pipelined = false;
    if ((rc = enhance_plan(m, st, B, Tf, m->host_chunks, &group, &tc, &pipelined))) return rc;
    const float lim = (atten_lim_db > 0.f) ? powf(10.f, -atten_lim_db / 20.f) : 0.f;
    size_t off[16];
    if ((rc = m->aux_arena.reserve(state_floats(m->cfg, st, (int)group, off) * sizeof(float) + 8192))) return rc;
    if ((rc = st->arena.reserve(sizeof(float) * (size_t)group * (Tp + out_len) + 4096))) return rc;
    st->arena.reset();
    float *d_in = st->arena.take<float>((size_t)group * Tp), *d_out = st->arena.take<float>((size_t)group * out_len);
    cudaStream_t sc = m->stream, sh = m->h2d, sd = m->d2h;
    std::vector<cudaEvent_t> evs;
    auto new_event = [&]() { cudaEvent_t e = nullptr; cudaEventCreateWithFlags(&e, cudaEventDisableTiming); evs.push_back(e); return e; };
    for (int64_t b0 = 0; b0 < B && !rc; b0 += group) {
        const int64_t nb = (B - b0 < group) ? B - b0 : group;
        const float *hx = h_audio + b0 * T;
        float *hy = h_out + b0 * out_len;
        // the previous group's D2H copies read d_out and its compute read d_in: order this group's first writes after them
        cudaEvent_t e0 = new_event();
        DFB_CUDA(cudaEventRecord(e0, sd));
        DFB_CUDA(cudaStreamWaitEvent(sc, e0, 0));
        cudaEvent_t e1 = new_event();
        DFB_CUDA(cudaEventRecord(e1, sc));
        DFB_CUDA(cudaStreamWaitEvent(sh, e1, 0));
        if (pad)  // zero tail of the padded rows (enhance.py:233)
            DFB_CUDA(cudaMemset2DAsync(d_in + T, sizeof(float) * Tp, 0, sizeof(float) * (Tp - T), nb, sh));
        ChunkHooks hooks;
        hooks.before = [&](int64_t x0, int64_t x1, cudaStream_t cs) -> int {
            if (x1 > T) x1 = T;
            if (x0 < x1)
                DFB_CUDA(cudaMemcpy2DAsync(d_in + x0, sizeof(float) * Tp, hx + x0, sizeof(float) * T, sizeof(float) * (x1 - x0), nb,
                                           cudaMemcpyHostToDevice, sh));
            cudaEvent_t e = new_event();
            DFB_CUDA(cudaEventRecord(e, sh));
            DFB_CUDA(cudaStreamWaitEvent(cs, e, 0));
            return DFB_OK;
        };
        hooks.after = [&](int64_t y0, int64_t y1, cudaStream_t cs) -> int {
            cudaEvent_t e = new_event();
            DFB_CUDA(cudaEventRecord(e, cs));
            DFB_CUDA(cudaStreamWaitEvent(sd, e, 0));
            DFB_CUDA(cudaMemcpy2DAsync(hy + y0, sizeof(float) * out_len, d_out + y0, sizeof(float) * out_len, sizeof(float) * (y1 - y0), nb,
                                       cudaMemcpyDeviceToHost, sd));
            return DFB_OK;
        };
        m->aux_arena.reset();
        rc = enhance_group(m, st, d_in, nb, Tp, T, pad, lim, d_out, out_len, tc, pipelined, sc, &hooks);
    }
    cudaError_t e1 = cudaStreamSynchronize(sc), e2 = cudaStreamSynchronize(sd), e3 = cudaStreamSynchronize(sh);
    for (cudaEvent_t e : evs) cudaEventDestroy(e);
    m->arena.reset();
    m->arena1.reset();
    if (rc) return rc;
    if (e1 != cudaSuccess || e2 != cudaSuccess || e3 != cudaSuccess)
        return fail(DFB_ERR_CUDA, "enhance_host failed: %s", cudaGetErrorString(e1 != cudaSuccess ? e1 : (e2 != cudaSuccess ? e2 : e3)));
    return DFB_OK;
}

// ============================================================== streaming API ====
// Frame-incremental processing with carried state: the batched counterpart of the reference's single-stream runtime
// (libDF/src/tract.rs:509-642 `DfTract::process`, C ABI libDF/src/capi.rs:83-253 df_create / df_process_frame / df_free).
// Every call feeds n >= 1 hops per stream and returns n hops; the output trails the input by `latency` frames
// (max(conv_lookahead, df_lookahead), + df_lookahead for DeepFilterNet2) on top of the STFT's own fft - hop samples,
// i.e. the concatenated output equals enhance(pad=False) of the concatenated input delayed by latency * hop samples.
struct dfb_stream {
    dfb_model *m;
    dfb_state *st;
    int B;
    float lim;
    StreamState S;
    float *slab = nullptr;
    bool gating = false;
    float th[3] = {-10.f, 30.f, 20.f};                 // tract.rs:180-185 defaults
    float *stage_in = nullptr, *stage_out = nullptr;   // device staging of the *_host entry point
    size_t stage_cap = 0;
};

extern "C" int dfb_stream_create(dfb_stream **out, dfb_model *m, dfb_state *st, int64_t B, float atten_lim_db) {
    if (!out || !m || !st || B <= 0 || B > 65535) return fail(DFB_ERR_INVALID, "bad argument");
    *out = nullptr;
    if (int rcs = check_state(m, st)) return rcs;
    if (int rch = check_half_overlap(st)) return rch;
    if (m->cfg.model_kind == 1)
        return fail(DFB_ERR_UNSUPPORTED, "DeepFilterNet v1 runs as one window per signal (forward_v1): no frame-incremental API");
    DFB_CUDA(cudaSetDevice(m->device));
    dfb_stream *h = new dfb_stream();
    h->m = m; h->st = st; h->B = (int)B;
    h->lim = (atten_lim_db > 0.f) ? powf(10.f, -atten_lim_db / 20.f) : 0.f;
    size_t off[16];
    const size_t n = state_floats(m->cfg, st, (int)B, off);
    if (cudaMalloc(&h->slab, n * sizeof(float)) != cudaSuccess) { delete h; return fail(DFB_ERR_OOM, "stream state allocation failed"); }
    cudaMemset(h->slab, 0, n * sizeof(float));
    state_bind(h->S, h->slab, off, (int)B);
    *out = h;
    return DFB_OK;
}

extern "C" void dfb_stream_free(dfb_stream *h) {
    if (!h) return;
    cudaSetDevice(h->m->device);
    if (h->slab) cudaFree(h->slab);
    if (h->stage_in) cudaFree(h->stage_in);
    if (h->stage_out) cudaFree(h->stage_out);
    delete h;
}

extern "C" int dfb_stream_reset(dfb_stream *h) {
    if (!h) return fail(DFB_ERR_INVALID, "null stream");
    size_t off[16];
    state_floats(h->m->cfg, h->st, h->B, off);
    state_bind(h->S, h->slab, off, h->B);
    return DFB_OK;
}

// LSNR stage gating of the Rust runtime (libDF/src/tract.rs:658-672; thresholds tract.rs:180-185, DfParams of
// deep-filter / capi.rs).  Off by default: the Python path this library mirrors does not gate.  DeepFilterNet3 only.
extern "C" int dfb_stream_set_lsnr_thresholds(dfb_stream *h, int enable, float min_db_thresh, float max_db_erb_thresh,
                                              float max_db_df_thresh) {
    if (!h) return fail(DFB_ERR_INVALID, "null stream");
    if (enable && h->m->cfg.model_kind != 3) return fail(DFB_ERR_UNSUPPORTED, "LSNR stage gating: DeepFilterNet3 topologies only");
    h->gating = enable != 0;
    h->th[0] = min_db_thresh; h->th[1] = max_db_erb_thresh; h->th[2] = max_db_df_thresh;
    return DFB_OK;
}

extern "C" int64_t dfb_stream_latency_frames(const dfb_stream *h) {
    if (!h) return -1;
    const ChunkGeom g = chunk_geom(h->m->cfg);
    return g.Lmax + g.lag;
}
extern "C" int64_t dfb_stream_frame_length(const dfb_stream *h) { return h ? h->st->hop : -1; }  // capi.rs df_get_frame_length

static int stream_step(dfb_stream *h, const float *d_in, int64_t n, bool flush, float *d_out, cudaStream_t s) {
    dfb_model *m = h->m;
    dfb_state *st = h->st;
    StreamState &S = h->S;
    const ChunkGeom g = chunk_geom(m->cfg);
    const int hop = st->hop, B = h->B;
    const int64_t Ltot = g.Lmax + g.lag;
    const int64_t n_out = flush ? Ltot : n;
    const int64_t a0 = S.a1, a1n = a0 + (flush ? 0 : n);
    int64_t d1n = flush ? a1n : a1n - g.Lmax, e1n = flush ? a1n : d1n - g.lag;
    if (d1n < S.d1) d1n = S.d1;
    if (e1n < S.e1) e1n = S.e1;
    // the window of this call: halo + new DNN frames (+ look-ahead)
    const int64_t W0 = S.d1 > kHalo ? S.d1 - kHalo : 0;
    const int Tw = (int)(d1n - W0);
    int rc = m->arena.reserve(chunk_bytes_per_stream(m->cfg, st, Tw + 1) * (size_t)B + (2 << 20));
    if (rc) return rc;
    // output slot j (hop j of d_out) carries frame a0 - Ltot + j (flush: a1 - Ltot + j); frames < 0 are silence
    const int64_t f0 = (flush ? S.a1 : a0) - Ltot;
    if (f0 < 0 || e1n <= S.e1) DFB_CUDA(cudaMemsetAsync(d_out, 0, sizeof(float) * B * n_out * hop, s));
    ChunkIO io{d_in, (flush ? 0 : n) * hop, (flush ? 0 : n) * hop, a0, S.started ? S.ana_mem : nullptr, d_out, n_out * hop, n_out * hop,
               f0 * hop, h->lim, h->gating ? h->th : nullptr};
    if (!flush && a1n > a0) {
        // zero analysis memory before the very first frame
        if (!S.started) DFB_CUDA(cudaMemsetAsync(S.ana_mem, 0, sizeof(float) * B * hop, s));
        io.init_mem = S.ana_mem;
    }
    if ((rc = run_chunk(m, st, S, io, a1n, d1n, e1n, s))) return rc;
    if (!flush)  // carried analysis memory: the last hop of this call's input
        DFB_CUDA(cudaMemcpy2DAsync(S.ana_mem, sizeof(float) * hop, d_in + (n - 1) * hop, sizeof(float) * n * hop, sizeof(float) * hop, B,
                                   cudaMemcpyDeviceToDevice, s));
    m->arena.reset();
    return DFB_OK;
}

// d_in [B][n_frames * hop] -> d_out [B][n_frames * hop] (device pointers, asynchronous on `stream`)
extern "C" int dfb_stream_process(dfb_stream *h, const float *d_in, int64_t n_frames, float *d_out, void *stream) {
    if (!h || !d_in || !d_out || n_frames <= 0) return fail(DFB_ERR_INVALID, "bad argument");
    DFB_CUDA(cudaSetDevice(h->m->device));
    return stream_step(h, d_in, n_frames, false, d_out, (cudaStream_t)stream);
}

// End of the stream: the `latency` frames still in flight, computed with zero look-ahead exactly like the end of a
// batch enhance(); d_out [B][latency * hop].  The stream must be reset before it is fed again.
extern "C" int dfb_stream_flush(dfb_stream *h, float *d_out, void *stream) {
    if (!h || !d_out) return fail(DFB_ERR_INVALID, "bad argument");
    DFB_CUDA(cudaSetDevice(h->m->device));
    if (dfb_stream_latency_frames(h) == 0) return DFB_OK;
    return stream_step(h, nullptr, 0, true, d_out, (cudaStream_t)stream);
}

// host-pointer variant (synchronous): h_in / h_out [B][n_frames * hop]; h_in == NULL flushes into h_out [B][latency * hop]
extern "C" int dfb_stream_process_host(dfb_stream *h, const float *h_in, int64_t n_frames, float *h_out) {
    if (!h || !h_out || (h_in && n_frames <= 0)) return fail(DFB_ERR_INVALID, "bad argument");
    DFB_CUDA(cudaSetDevice(h->m->device));
    const bool flush = h_in == nullptr;
    const int64_t nf = flush ? dfb_stream_latency_frames(h) : n_frames;
    if (nf == 0) return DFB_OK;
    const size_t bytes = sizeof(float) * (size_t)h->B * nf * h->st->hop;
    if (bytes > h->stage_cap) {
        if (h->stage_in) cudaFree(h->stage_in);
        if (h->stage_out) cudaFree(h->stage_out);
        h->stage_in = h->stage_out = nullptr; h->stage_cap = 0;
        if (cudaMalloc(&h->stage_in, bytes) != cudaSuccess || cudaMalloc(&h->stage_out, bytes) != cudaSuccess)
            return fail(DFB_ERR_OOM, "stream staging allocation failed");
        h->stage_cap = bytes;
    }
    cudaStream_t s = h->m->stream;
    if (!flush) DFB_CUDA(cudaMemcpyAsync(h->stage_in, h_in, bytes, cudaMemcpyHostToDevice, s));
    int rc = stream_step(h, h->stage_in, nf, flush, h->stage_out, s);
    if (rc) return rc;
    DFB_CUDA(cudaMemcpyAsync(h_out, h->stage_out, bytes, cudaMemcpyDeviceToHost, s));
    DFB_CUDA(cudaStreamSynchronize(s));
    return DFB_OK;
}
