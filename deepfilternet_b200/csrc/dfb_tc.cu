// dfb_tc.cu -- 5th-generation tensor-core (tcgen05) kernels for the dense contractions of the path.
//
//   k_gemm_bf16x3: GRU input projections W_ih x + b_ih (torch.nn.GRU inside SqueezedGRU[_S], modules.py:684,723)
//   k_dwpw_bx:     fused depthwise (+pathway) -> 1x1 conv -> ReLU blocks (Conv2dNormAct / ConvTranspose2dNormAct)
//   k_gru_tc:      the GRU recurrence W_hh h with the weights resident in tensor memory
// All three reach fp32-level accuracy on the BF16 tensor pipe by splitting both operands into BF16 hi + lo planes
// (x = hi + lo to ~2^-17) and issuing hi*hi + lo*hi + hi*lo with fp32 accumulation in TMEM.
#include <cooperative_groups.h>
#include <map>
#include <mutex>
#include <cuda.h>
#include <cuda_bf16.h>

#include "dfb_common.cuh"
#include "dfb_dwpw.cuh"
#include "dfb_ptx.cuh"

namespace dfb {

// ----------------------------------------------------------------------------- PTX helpers ----





// ------------------------------------------------------------- BF16x3 GEMM (projections) ----
// Y[M,N] = X[M,K] . W[N,K]^T + bias with fp32-level accuracy on the BF16 tensor pipe: both operands
// are stored as BF16 hi/lo planes (x = hi + lo to ~2^-17; X planes written by the producing kernel's
// epilogue, W planes split on the host) and every product is hi*hi + lo*hi + hi*lo with fp32
// accumulation in TMEM.
// W-stationary, transposed: a persistent CTA owns 128 output columns; its W slice [128 n][K <= 256] sits in
// TENSOR MEMORY for the whole kernel (hi | lo planes, 256 columns) and is the MMA's A operand (TS mode), the
// X tiles (128 rows x 64 k per stage, hi + lo = 32 KB) stream through a 6-stage TMA ring as the B operand,
// and the accumulator D[n][m] (two 128-column TMEM buffers) comes out transposed: TMEM lane = output column,
// so every epilogue store instruction writes 128 contiguous bytes of one output row.
// History (ncu): one CTA per 128 x 64 tile re-read the X tile 12 times -- 2.3 GB of L2 -> SM traffic per
// projection, lts-bound at 6 TB/s, IPC 0.24; an X-stationary version could keep only 80 KB of W in flight
// next to its 128 KB X tile and was latency bound.  Here all of shared memory is the in-flight ring.
// warps 0-7 = W load (0-3), then epilogue (lane quarter = warp % 4, column half = warp / 4; two warps per
// scheduler -- with four the epilogue's dependent address / store chain was the bottleneck, ncu: 80 % of the
// samples); warp 8 = TMA producer; warp 9 = MMA issuer (elect.sync issue).
constexpr int kBxBM = 128 /* x rows per tile (MMA N) */, kBxBN = 128 /* output columns per CTA (MMA M) */, kBxBK = 64,
              kBxStages = 6, kBxMaxK = 256;

struct BxSmem {
    alignas(1024) unsigned char x[kBxStages][2][kBxBM * 128];  // [stage][hi|lo][128 rows x 64 bf16], 128B swizzle
    alignas(8) uint64_t full[kBxStages];
    uint64_t empty[kBxStages];
    uint64_t tmem_full[2], tmem_empty[2];
    uint32_t tmem_base;
};


constexpr int kBxThreads = 320;
__global__ void __launch_bounds__(kBxThreads, 1)
k_gemm_bf16x3(const __grid_constant__ CUtensorMap tmXhi, const __grid_constant__ CUtensorMap tmXlo,
              const unsigned short *__restrict__ w_hi, const unsigned short *__restrict__ w_lo /* [N][K] BF16 */,
              const float *__restrict__ bias, float *__restrict__ Y, int64_t ldy, int M, int N, int K, int ldw, int k0,
              int accumulate) {
    // K > 256 (H = 512 projections) runs as passes over K slices of 256 (the W slice of one pass fills the tensor memory):
    // this launch covers columns [k0, k0 + K) of X and W (W row pitch ldw) and, when `accumulate`, adds to Y
    extern __shared__ __align__(1024) unsigned char tc_smem_raw[];
    BxSmem &sm = *reinterpret_cast<BxSmem *>(((uintptr_t)tc_smem_raw + 1023) & ~uintptr_t(1023));
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n0 = blockIdx.x * kBxBN;
    const int nkb = K / kBxBK, wcols = K / 2;             // TMEM columns of one W plane
    const int ntiles = (M + kBxBM - 1) / kBxBM;
    const uint32_t dcol = 2 * (kBxMaxK / 2);              // accumulators behind the two W planes
    if (threadIdx.x == 0) {
        for (int s = 0; s < kBxStages; s++) { mbar_init(&sm.full[s], 1); mbar_init(&sm.empty[s], 1); }
        for (int i = 0; i < 2; i++) { mbar_init(&sm.tmem_full[i], 1); mbar_init(&sm.tmem_empty[i], 8); }
        fence_barrier_init();
    }
    if (warp == 0) tmem_alloc(&sm.tmem_base, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = sm.tmem_base;
    if (warp < 4) {
        // ---- W slice -> TMEM: lane = output column n0 + 32 warp + lane, column j of a plane = k elements (2 j, 2 j + 1)
        const int n = n0 + warp * 32 + lane;
        for (int cb = 0; cb < nkb; cb++) {  // 64 k elements = 32 columns per store
            uint32_t vh[32], vl[32];
            const uint4 *ph = reinterpret_cast<const uint4 *>(w_hi + (int64_t)n * ldw + k0 + cb * 64);
            const uint4 *pl = reinterpret_cast<const uint4 *>(w_lo + (int64_t)n * ldw + k0 + cb * 64);
#pragma unroll
            for (int i = 0; i < 8; i++) {
                const uint4 a = n < N ? __ldg(ph + i) : make_uint4(0, 0, 0, 0), c = n < N ? __ldg(pl + i) : make_uint4(0, 0, 0, 0);
                vh[4 * i] = a.x; vh[4 * i + 1] = a.y; vh[4 * i + 2] = a.z; vh[4 * i + 3] = a.w;
                vl[4 * i] = c.x; vl[4 * i + 1] = c.y; vl[4 * i + 2] = c.z; vl[4 * i + 3] = c.w;
            }
            const uint32_t ta = tmem + ((uint32_t)(warp * 32) << 16) + cb * 32;
            tmem_st32(ta, vh);
            tmem_st32(ta + wcols, vl);
        }
        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (warp == 8) {
        // ===== TMA producer: X tiles of this CTA's row groups
        if (lane == 0) {
            tma_prefetch_desc(&tmXhi); tma_prefetch_desc(&tmXlo);
            int it = 0;
            for (int tile = blockIdx.y; tile < ntiles; tile += gridDim.y)
                for (int kb = 0; kb < nkb; kb++, it++) {
                    const int s = it % kBxStages, n = it / kBxStages;
                    if (n > 0) mbar_wait(&sm.empty[s], (n - 1) & 1);
                    mbar_expect_tx(&sm.full[s], 2 * kBxBM * 128);
                    tma_load_2d(sm.x[s][0], &tmXhi, k0 + kb * kBxBK, tile * kBxBM, &sm.full[s]);
                    tma_load_2d(sm.x[s][1], &tmXlo, k0 + kb * kBxBK, tile * kBxBM, &sm.full[s]);
                }
        }
    } else if (warp == 9) {
        // ===== MMA issuer (whole warp, elected lane issues): D[n][m] += W[n][k] . X[m][k]
        constexpr uint32_t idesc = umma_idesc_bf16(kBxBN, kBxBM);
        const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem, 0);
        int it = 0, li = 0;
        for (int tile = blockIdx.y; tile < ntiles; tile += gridDim.y, li++) {
            const int buf = li & 1;
            if (li >= 2) mbar_wait(&sm.tmem_empty[buf], ((li >> 1) - 1) & 1);
            tc_fence_after();
            const uint32_t d = tmem_u + dcol + buf * kBxBM;
            for (int kb = 0; kb < nkb; kb++, it++) {
                const int s = it % kBxStages, n = it / kBxStages;
                mbar_wait(&sm.full[s], n & 1);
                tc_fence_after();
                const uint64_t xh = umma_desc_sw128(smem_u32(sm.x[s][0])), xl = umma_desc_sw128(smem_u32(sm.x[s][1]));
#pragma unroll
                for (int k = 0; k < kBxBK / 16; k++) {  // K step 16: 8 TMEM columns of W, 32 bytes inside the swizzle row of X
                    const uint32_t wh = tmem_u + kb * 32 + k * 8;
                    umma_bf16_ts_elect(d, wh, xh + 2 * k, idesc, (kb | k) != 0);
                    umma_bf16_ts_elect(d, wh + wcols, xh + 2 * k, idesc, 1u);
                    umma_bf16_ts_elect(d, wh, xl + 2 * k, idesc, 1u);
                }
                umma_commit_elect(&sm.empty[s]);
            }
            umma_commit_elect(&sm.tmem_full[buf]);
        }
    } else {
        // ===== epilogue: warp w owns TMEM lanes [32 (w % 4), +32) = output columns n0 + 32 (w % 4) + lane and the
        //       accumulator columns (= rows of Y) [64 (w / 4), +64) of every tile
        const int q = warp & 3, half = warp >> 2;
        const int n = n0 + q * 32 + lane;
        const float bn = (bias && n < N) ? __ldg(bias + n) : 0.f;
        int li = 0;
        for (int tile = blockIdx.y; tile < ntiles; tile += gridDim.y, li++) {
            const int buf = li & 1;
            mbar_wait(&sm.tmem_full[buf], (li >> 1) & 1);
            tc_fence_after();
            const uint32_t ta = tmem + ((uint32_t)(q * 32) << 16) + dcol + buf * kBxBM + half * 64;
            const int m0 = tile * kBxBM + half * 64;
            float v0[32], v1[32];
            tmem_ld32(ta, v0);
            tmem_ld32(ta + 32, v1);
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&sm.tmem_empty[buf]);  // accumulator read: hand the buffer back before the stores
            float *dst = Y + (int64_t)m0 * ldy + n;
            if (accumulate && n < N) {
                // second K pass: Y += D.  All loads of a half first (independent), then the stores: as separate
                // load / add / store triples the compiler must assume aliasing and serialises 64 DRAM round trips
                const bool full = m0 + 64 <= M;
#pragma unroll
                for (int j = 0; j < 32; j++) v0[j] += (full || m0 + j < M) ? dst[(int64_t)j * ldy] : 0.f;
#pragma unroll
                for (int j = 0; j < 32; j++) if (full || m0 + j < M) dst[(int64_t)j * ldy] = v0[j];
                float *dst1 = dst + 32 * ldy;
#pragma unroll
                for (int j = 0; j < 32; j++) v1[j] += (full || m0 + 32 + j < M) ? dst1[(int64_t)j * ldy] : 0.f;
#pragma unroll
                for (int j = 0; j < 32; j++) if (full || m0 + 32 + j < M) dst1[(int64_t)j * ldy] = v1[j];
            } else if (m0 + 64 <= M && n < N) {
#pragma unroll
                for (int j = 0; j < 32; j++) { *dst = v0[j] + bn; dst += ldy; }
#pragma unroll
                for (int j = 0; j < 32; j++) { *dst = v1[j] + bn; dst += ldy; }
            } else if (n < N) {
#pragma unroll
                for (int j = 0; j < 32; j++) { if (m0 + j < M) *dst = v0[j] + bn; dst += ldy; }
#pragma unroll
                for (int j = 0; j < 32; j++) { if (m0 + 32 + j < M) *dst = v1[j] + bn; dst += ldy; }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 512);
}

// ------------------------------------------- fused depthwise -> 1x1 (tcgen05) -> ReLU ----
// Tensor-core version of k_dwpw (dfb_model.cu) at fp32-level accuracy (BF16x3): one CTA per 128-row tile.
//   0. thread 0 asks the TMA engine for every raw input (and pathway) frame of the tile -- one contiguous
//      Fin * 256-byte bulk copy per frame -- plus the pre-swizzled 16 KB weight image: the CTA's whole input is
//      in flight at once without passing through registers;
//   1. all 256 threads run the depthwise (+pathway) prologue out of shared memory (thread = channel quad x 8
//      consecutive rows), split the result x = hi + lo into BF16 planes and write them in the UMMA K-major
//      128B-swizzle layout (a row of 64 channels is exactly one 128-byte swizzle row);
//   2. warp 0 issues 12 tcgen05.mma (M128 N64 K16; hi*hi + lo*hi + hi*lo), fp32 accumulator in 64 TMEM columns;
//   3. all 8 warps read their TMEM lane quarter / column half (tcgen05.ld), add bias, ReLU and stage the fp32
//      tile in the (now free) operand planes with an XOR chunk swizzle -- conflict free for row-per-lane writes;
//   4. the CTA streams the staged tile out with coalesced 256-byte half-warp stores.
// Two CTAs per SM overlap each other's load / MMA / store phases.  Shared memory (1024-byte aligned base):
//   [0, 32K) A hi | lo planes (later the fp32 staging tile)   [32K, 48K) W hi | lo   [48K, 48K + raw) raw frames
//   then bias[64], two mbarriers, the TMEM base address.
constexpr int kDxThreads = 256;
constexpr uint32_t kDxW = 32768, kDxRaw = 49152, kDxTail = 64 * 4 + 32;


// MASK = 1 (last ERB decoder block of the kt = 1 models): the tile holds whole frames, so the mask head
//   m[t,f] = sigmoid(sum_{df,c} w[df][c] * (relu(e0 * ps + pb) + out)[t][f+df-1][c] + bias)
// (conv0_out(conv0p(e0) + convt1(...)), deepfilternet3.py:253) is evaluated right on the staged fp32 tile and
// `out` itself never goes to HBM (p.out may be null).
template <int MODE, int KT, int PATH, int MASK>
__global__ void __launch_bounds__(kDxThreads, 2)
k_dwpw_bx(DwPwParams p, const float *__restrict__ w_sw /* [hi | lo] x [64 n][64 k] BF16, 128B-swizzled rows */) {
    extern __shared__ __align__(1024) unsigned char tc_smem_raw[];
    const uint32_t sb = smem_u32(tc_smem_raw);
    if (sb & 1023u) __trap();  // the swizzled operand planes need a 1024-byte aligned base
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int b = blockIdx.y, t0 = blockIdx.x * p.NF;
    const int nf = min(p.NF, p.T - t0);
    const int R = nf * p.Fout;  // rows actually present
    const int tq0 = t0 - (KT - 1);
    const uint32_t fbytes = (uint32_t)p.Fin * kCh * 4;
    const uint32_t raw_in = sb + kDxRaw, raw_path = raw_in + (uint32_t)(p.NF + KT - 1) * fbytes;
    const uint32_t raw_e0 = raw_in + (uint32_t)(p.NF + KT - 1) * fbytes * (PATH ? 2u : 1u);  // MASK: [NF][Fout][64]
    const uint32_t obytes = (uint32_t)p.Fout * kCh * 4;
    const uint32_t tail = raw_e0 + (MASK ? (uint32_t)p.NF * obytes : 0u);
    const uint32_t s_bias = tail, bar_mma = tail + 256, bar_raw = tail + 264, s_tmem = tail + 272;
    const uint32_t s_mask = raw_in;  // MASK: ps | pb | w[3][64], written over the raw input frames once they are converted
    if (tid == 0) {
        mbar_init_a(bar_mma, 1);
        mbar_init_a(bar_raw, 1);
        fence_barrier_init();
        const int ta = max(tq0, 0), tb = t0 + nf;  // frames [ta, tb)
        mbar_expect_tx_a(bar_raw, (uint32_t)(tb - ta) * fbytes * (PATH ? 2u : 1u) + 2u * kCh * 128u + (MASK ? (uint32_t)nf * obytes : 0u));
        if (MASK)
            for (int t = t0; t < tb; t++)
                bulk_load(raw_e0 + (uint32_t)(t - t0) * obytes, p.mk_e0 + ((int64_t)b * p.T + t) * p.Fout * kCh, obytes, bar_raw);
        for (int t = ta; t < tb; t++) {
            bulk_load(raw_in + (uint32_t)(t - tq0) * fbytes, p.in + ((int64_t)b * p.T + t) * p.in_fs, fbytes, bar_raw);
            if (PATH) bulk_load(raw_path + (uint32_t)(t - tq0) * fbytes, p.path + ((int64_t)b * p.T + t) * p.path_fs, fbytes, bar_raw);
        }
        bulk_load(sb + kDxW, w_sw, 2 * kCh * 128, bar_raw);
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(s_tmem), "r"(kCh) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (tid < kCh / 4) sts128(s_bias + tid * 16, __ldg(reinterpret_cast<const float4 *>(p.bias) + tid));
    // ---- depthwise taps of this thread's channel quad, pathway affine
    const int cq = tid & 15, slot = tid >> 4;
    float4 wd[KT][3], ps4, pb4;
#pragma unroll
    for (int dt = 0; dt < KT; dt++)
#pragma unroll
        for (int df = 0; df < 3; df++) wd[dt][df] = __ldg(reinterpret_cast<const float4 *>(p.dw + (dt * 3 + df) * kCh) + cq);
    if (PATH) {
        ps4 = __ldg(reinterpret_cast<const float4 *>(p.ps) + cq);
        pb4 = __ldg(reinterpret_cast<const float4 *>(p.pb) + cq);
    }
    // rows r = 8 slot + i: (frame fr, bin fo) by multiply-shift division (exact for r < 128), then incrementally
    int fr = (8 * slot * p.fo_magic) >> 16, fo = 8 * slot - fr * p.Fout;
    __syncthreads();  // barriers initialised before anyone waits on them
    mbar_wait_a(bar_raw, 0);
    // ---- prologue
    auto rd = [&](uint32_t a) -> float4 {
        float4 x = lds128(a);
        if (PATH) {
            const float4 e = lds128(a + (raw_path - raw_in));
            x.x += fmaxf(fmaf(e.x, ps4.x, pb4.x), 0.f); x.y += fmaxf(fmaf(e.y, ps4.y, pb4.y), 0.f);
            x.z += fmaxf(fmaf(e.z, ps4.z, pb4.z), 0.f); x.w += fmaxf(fmaf(e.w, ps4.w, pb4.w), 0.f);
        }
        return x;
    };
    const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int i = 0; i < 8; i++) {
        const int r = 8 * slot + i;
        float4 acc = zero4;
        if (r < R) {
#pragma unroll
            for (int dt = 0; dt < KT; dt++) {
                // tap dt reads frame t - (KT-1-dt) = raw frame fr + dt; before the start of the stream it is zero padding
                if (KT > 1 && tq0 + fr + dt < 0) continue;
                const uint32_t fb = raw_in + (uint32_t)(fr + dt) * fbytes + cq * 16;
                if (MODE == DW_S1) {
                    const uint32_t a = fb + (uint32_t)fo * 256;
                    if (fo > 0) acc = f4_fma(rd(a - 256), wd[dt][0], acc);
                    acc = f4_fma(rd(a), wd[dt][1], acc);
                    if (fo + 1 < p.Fin) acc = f4_fma(rd(a + 256), wd[dt][2], acc);
                } else if (MODE == DW_S2) {
                    const uint32_t a = fb + (uint32_t)fo * 512;
                    if (fo > 0) acc = f4_fma(rd(a - 256), wd[dt][0], acc);
                    acc = f4_fma(rd(a), wd[dt][1], acc);
                    acc = f4_fma(rd(a + 256), wd[dt][2], acc);
                } else {  // DW_T2: out[2j] = w1 x[j]; out[2j+1] = w2 x[j] + w0 x[j+1]
                    const uint32_t a = fb + (uint32_t)(fo >> 1) * 256;
                    if ((fo & 1) == 0) {
                        acc = f4_fma(rd(a), wd[dt][1], acc);
                    } else {
                        acc = f4_fma(rd(a), wd[dt][2], acc);
                        if ((fo >> 1) + 1 < p.Fin) acc = f4_fma(rd(a + 256), wd[dt][0], acc);
                    }
                }
            }
        }
        uint32_t h0, l0, h1, l1;
        bf16x2_split(acc.x, acc.y, h0, l0);
        bf16x2_split(acc.z, acc.w, h1, l1);
        const uint32_t off = sb + sw128_off(r, cq >> 1) + (cq & 1) * 8;
        sts64(off, h0, h1);
        sts64(off + 16384, l0, l1);
        if (++fo == p.Fout) { fo = 0; fr++; }
    }
    fence_proxy_async();  // generic-proxy smem writes -> visible to the tensor core (async proxy)
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = lds32(s_tmem);
    if (MASK && tid >= 64 && tid < 64 + 80) {  // ps | pb | w[3][64] as 80 float4
        const int i = tid - 64;
        const float4 *src = i < 16 ? reinterpret_cast<const float4 *>(p.mk_ps) + i
                          : i < 32 ? reinterpret_cast<const float4 *>(p.mk_pb) + (i - 16)
                                   : reinterpret_cast<const float4 *>(p.mk_w) + (i - 32);
        sts128(s_mask + i * 16, __ldg(src));
    }
    if (warp == 0) {
        constexpr uint32_t idesc = umma_idesc_bf16(128, kCh);
        const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem, 0);
        const uint64_t ah = umma_desc_sw128(sb), al = umma_desc_sw128(sb + 16384);
        const uint64_t bh = umma_desc_sw128(sb + kDxW), bl = umma_desc_sw128(sb + kDxW + 8192);
#pragma unroll
        for (int k = 0; k < kCh / 16; k++) {  // 32 bytes per K step inside the 128-byte swizzle row
            umma_bf16_ss_elect(tmem_u, ah + 2 * k, bh + 2 * k, idesc, k != 0);
            umma_bf16_ss_elect(tmem_u, al + 2 * k, bh + 2 * k, idesc, 1u);
            umma_bf16_ss_elect(tmem_u, ah + 2 * k, bl + 2 * k, idesc, 1u);
        }
        asm volatile(
            "{\n\t"
            ".reg .pred e;\n\t"
            "elect.sync _|e, 0xffffffff;\n\t"
            "@e tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t"
            "}\n" ::"r"(bar_mma)
            : "memory");
    }
    mbar_wait_a(bar_mma, 0);
    tc_fence_after();
    // ---- accumulator -> bias + ReLU -> staging tile (row r, 16-byte chunk j at r * 256 + ((j ^ (r & 15)) << 4))
    {
        const int q = warp & 3, ch = warp >> 2;  // TMEM lane quarter, column half
        float v[32];
        tmem_ld32(tmem + ((uint32_t)(q * 32) << 16) + ch * 32, v);
        const int r = q * 32 + lane;
        const uint32_t row = sb + r * 256;
#pragma unroll
        for (int jj = 0; jj < 8; jj++) {
            const float4 bv = lds128(s_bias + (ch * 8 + jj) * 16);
            sts128(row + (((ch * 8 + jj) ^ (r & 15)) << 4),
                   make_float4(fmaxf(v[jj * 4] + bv.x, 0.f), fmaxf(v[jj * 4 + 1] + bv.y, 0.f), fmaxf(v[jj * 4 + 2] + bv.z, 0.f),
                               fmaxf(v[jj * 4 + 3] + bv.w, 0.f)));
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem, kCh);
    if (MASK) {
        // thread = (channel quad j, 8 consecutive rows of one frame): X = relu(e0 * ps + pb) + out is formed once per
        // (row, quad), each row feeds the three taps of its neighbours, and the 16 quads are reduced with shuffles
        const int j = tid & 15, r0 = 8 * slot;
        const int fr = (r0 * p.fo_magic) >> 16, f0 = r0 - fr * p.Fout;   // Fout % 8 == 0: the 8 rows share a frame
        const float4 s4 = lds128(s_mask + j * 16), b4 = lds128(s_mask + 256 + j * 16);
        const float4 w0 = lds128(s_mask + 512 + j * 16), w1 = lds128(s_mask + 512 + 256 + j * 16), w2 = lds128(s_mask + 512 + 512 + j * 16);
        float part[8];
#pragma unroll
        for (int i = 0; i < 8; i++) part[i] = 0.f;
        if (r0 < R) {
#pragma unroll
            for (int i = -1; i <= 8; i++) {
                const int f2 = f0 + i, r2 = r0 + i;
                if (f2 < 0 || f2 >= p.Fout) continue;
                const float4 d = lds128(sb + r2 * 256 + ((j ^ (r2 & 15)) << 4));
                const float4 e = lds128(raw_e0 + r2 * 256 + j * 16);
                float4 x;
                x.x = fmaxf(fmaf(e.x, s4.x, b4.x), 0.f) + d.x; x.y = fmaxf(fmaf(e.y, s4.y, b4.y), 0.f) + d.y;
                x.z = fmaxf(fmaf(e.z, s4.z, b4.z), 0.f) + d.z; x.w = fmaxf(fmaf(e.w, s4.w, b4.w), 0.f) + d.w;
                // row r2 is tap df = 0 of output r2 + 1, tap 1 of r2, tap 2 of r2 - 1
                if (i + 1 < 8) part[i + 1 < 0 ? 0 : i + 1] += x.x * w0.x + x.y * w0.y + x.z * w0.z + x.w * w0.w;
                if (i >= 0 && i < 8) part[i < 0 ? 0 : (i > 7 ? 7 : i)] += x.x * w1.x + x.y * w1.y + x.z * w1.z + x.w * w1.w;
                if (i - 1 >= 0) part[i - 1 > 7 ? 7 : i - 1] += x.x * w2.x + x.y * w2.y + x.z * w2.z + x.w * w2.w;
            }
        }
#pragma unroll
        for (int i = 0; i < 8; i++) {
            float v = part[i];
            v += __shfl_xor_sync(0xffffffffu, v, 1);
            v += __shfl_xor_sync(0xffffffffu, v, 2);
            v += __shfl_xor_sync(0xffffffffu, v, 4);
            v += __shfl_xor_sync(0xffffffffu, v, 8);
            part[i] = v;
        }
        if (r0 < R && j < 8) {
            float z = part[0];
#pragma unroll
            for (int i = 1; i < 8; i++) z = j == i ? part[i] : z;
            z += __ldg(p.mk_bias);
            p.mk_out[((int64_t)b * p.T + t0 + fr) * p.Fout + f0 + j] = 1.f / (1.f + expf(-z));
        }
    }
    // ---- coalesced write-out: half a warp per 256-byte row, 8 consecutive rows per thread
    if (p.out || p.out_hi) {
        const int j = tid & 15;
        int fr2 = (8 * slot * p.fo_magic) >> 16, fo2 = 8 * slot - fr2 * p.Fout;
        int64_t off = ((int64_t)b * p.T + t0 + fr2) * p.out_fs + fo2 * kCh + j * 4;
#pragma unroll
        for (int i = 0; i < 8; i++) {
            const int r = 8 * slot + i;
            if (r < R) {
                const float4 v = lds128(sb + r * 256 + ((j ^ (r & 15)) << 4));
                if (p.out) *reinterpret_cast<float4 *>(p.out + off) = v;
                if (p.out_hi) {
                    uint32_t h0, l0, h1, l1;
                    bf16x2_split(v.x, v.y, h0, l0);
                    bf16x2_split(v.z, v.w, h1, l1);
                    *reinterpret_cast<uint2 *>(p.out_hi + off) = make_uint2(h0, h1);
                    *reinterpret_cast<uint2 *>(p.out_lo + off) = make_uint2(l0, l1);
                }
            }
            off += kCh;
            if (++fo2 == p.Fout) { fo2 = 0; off += p.out_fs - (int64_t)p.Fout * kCh; }
        }
    }
}

template <int MODE, int KT, int PATH, int MASK = 0>
static int launch_dwpw_bx(cudaStream_t s, const DwPwParams &p, const float *w_sw, int B) {
    static int attr_smem[64] = {0};  // per device: largest dynamic shared memory size set so far
    int dev = 0;
    cudaGetDevice(&dev);
    dev &= 63;
    const int raw = (p.NF + KT - 1) * p.Fin * kCh * 4 * (PATH ? 2 : 1) + (MASK ? p.NF * p.Fout * kCh * 4 : 0);
    const int smem = (int)kDxRaw + raw + (int)kDxTail;
    if (smem > 227 * 1024) return fail(DFB_ERR_UNSUPPORTED, "dwpw tile needs %d bytes of shared memory", smem);
    if (smem > attr_smem[dev]) {
        DFB_CUDA(cudaFuncSetAttribute(k_dwpw_bx<MODE, KT, PATH, MASK>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        attr_smem[dev] = smem;
    }
    dim3 grid((unsigned)((p.T + p.NF - 1) / p.NF), (unsigned)B);
    DFB_PROF("k_dwpw_bx", s);
    k_dwpw_bx<MODE, KT, PATH, MASK><<<grid, kDxThreads, smem, s>>>(p, w_sw);
    DFB_LAUNCH_CHECK();
    return DFB_OK;
}

template <int MODE>
int launch_dwpw_tc(cudaStream_t s, DwPwParams p, const float *w_sw, int B) {
    p.NF = 128 / p.Fout;
    if (p.NF < 1) p.NF = 1;
    if (p.NF * p.Fout > 128) return fail(DFB_ERR_UNSUPPORTED, "dwpw tile: Fout = %d", p.Fout);
    p.fo_magic = (65536 + p.Fout - 1) / p.Fout;
    for (int r = 0; r < 128; r++)
        if (((r * p.fo_magic) >> 16) != r / p.Fout) return fail(DFB_ERR_UNSUPPORTED, "dwpw tile: Fout = %d", p.Fout);
    if ((p.in_fs * 4) % 16 || (p.path && (p.path_fs * 4) % 16)) return fail(DFB_ERR_UNSUPPORTED, "dwpw: unaligned frame stride");
    const bool path = p.path != nullptr;
    if (MODE == DW_S1) {
        if (p.kt == 1) return path ? launch_dwpw_bx<DW_S1, 1, 1>(s, p, w_sw, B) : launch_dwpw_bx<DW_S1, 1, 0>(s, p, w_sw, B);
        if (p.kt == 2) return path ? launch_dwpw_bx<DW_S1, 2, 1>(s, p, w_sw, B) : launch_dwpw_bx<DW_S1, 2, 0>(s, p, w_sw, B);
    } else if (MODE == DW_S2 && !path) {
        if (p.kt == 1) return launch_dwpw_bx<DW_S2, 1, 0>(s, p, w_sw, B);
        if (p.kt == 2) return launch_dwpw_bx<DW_S2, 2, 0>(s, p, w_sw, B);
    } else if (MODE == DW_T2 && path && p.kt == 1) {
        if (p.mk_e0) {
            return launch_dwpw_bx<DW_T2, 1, 1, 1>(s, p, w_sw, B);
        }
        return launch_dwpw_bx<DW_T2, 1, 1>(s, p, w_sw, B);
    }
    return fail(DFB_ERR_UNSUPPORTED, "dwpw tensor-core path: mode %d kt %d path %d", MODE, p.kt, (int)path);
}
template int launch_dwpw_tc<DW_S1>(cudaStream_t, DwPwParams, const float *, int);
template int launch_dwpw_tc<DW_S2>(cudaStream_t, DwPwParams, const float *, int);
template int launch_dwpw_tc<DW_T2>(cudaStream_t, DwPwParams, const float *, int);

// ---------------------------------------------------------- DF pathway conv on tensor cores ----
// coefs[b,t,f,:] = relu( pw( conv_t(c0) ) + b )  (df_convp, deepfilternet3.py:293-295: grouped (2) temporal conv 64 -> 10
// with kernel (5,1), 1x1 conv 10 x 10, BN, ReLU).  The FFMA kernel (k_df_convp, dfb_model.cu) is instruction-issue bound
// (~250 warp instructions per frame and bin pair: 1.4 ms of issue slots per 128 x 10 s, measured 2.2 ms = 0.25 of the HBM
// roofline, and a deeper load ring did not change it).  Here the channel contraction runs on tcgen05:
//   Y[t, g*32 + dt*5 + o] = sum_{c in group g} w1[dt][g*5+o][c] * c0[t, f, c]        (one [128 t x 64 c] x [64 c x 64] product)
//   z[t, g*5 + o]         = sum_dt Y[t - 4 + dt, g*32 + dt*5 + o]                     (shifted adds out of shared memory)
//   coefs[t, f, :]        = relu(z . w2 + b)
// One CTA = (stream, bin f, 124 output frames): its 128 time rows of c0[., f, :] (4 frames of history) arrive as two TMA
// tensor boxes (rows 24.5 KB apart in HBM, 2 x 128 B per row, 128-byte swizzle), are split into BF16 hi / lo operand planes
// (BF16x3: fp32-level accuracy), 12 tcgen05.mma (M128 N64 K16) leave Y in 64 TMEM columns, the epilogue stages Y in shared
// memory (row stride 65 floats) and 128 threads (one per time row) do the shifted sums, the 1x1 conv and the 40-byte store.
constexpr int kCvThreads = 256, kCvOut = 124, kCvYld = 51 /* 2 x 25 used columns + 1 */, kCvBins = 8;
// shared memory: [0, 32K) A hi | lo planes, [32K, 48K) W hi | lo, [48K, 80K) raw fp32 boxes of the current bin,
// [80K, +26112) the staged Y tile, then w2 | bias, barriers, the TMEM address
constexpr uint32_t kCvW = 32768, kCvRawOff = 49152, kCvYs = kCvRawOff + 32768, kCvTail = kCvYs + 128 * kCvYld * 4;

struct CvParams {
    const float *w_sw;   // [hi | lo] x [64 n][64 k] BF16, 128B-swizzled rows: n = g*32 + dt*5 + o, k = channel
    const float *w2;     // [10 in][10 out]
    const float *bias;   // [10]
    float *coefs;        // [B,T,Fd,10]
    int T, Fd;
};

// One CTA = (stream, kCvBins consecutive bins, 124 output frames): the weight image, the TMEM allocation and the barrier
// set-up are paid once per CTA, and the TMA load of the next bin's rows is issued as soon as the current bin's rows have
// been converted, so it overlaps the MMA and the epilogue (the first version ran one bin per CTA: 0.39 of HBM).
template <int ORDER, int KTP>
__global__ void __launch_bounds__(kCvThreads, 2) k_df_convp_tc(const __grid_constant__ CUtensorMap tmC0, CvParams p) {
    constexpr int O2 = 2 * ORDER, NY = KTP * ORDER;
    extern __shared__ __align__(1024) unsigned char tc_smem_raw[];
    const uint32_t sb = (smem_u32(tc_smem_raw) + 1023u) & ~1023u;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int f_begin = blockIdx.x * kCvBins, f_end = min(f_begin + kCvBins, p.Fd);
    const int b = blockIdx.z, t0 = blockIdx.y * kCvOut, r0 = t0 - (KTP - 1);
    const uint32_t s_w2 = sb + kCvTail, bar_raw = s_w2 + 512, bar_mma = bar_raw + 8, bar_w = bar_mma + 8, s_tmem = bar_w + 8;
    const int row = b * p.T + r0;   // may be negative for the first stream: out-of-bounds rows arrive as zeros
    auto load_bin = [&](int f) {    // thread 0 only
        mbar_expect_tx_a(bar_raw, 32768);
        asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                     ::"r"(sb + kCvRawOff), "l"((uint64_t)&tmC0), "r"(f * 64), "r"(row), "r"(bar_raw) : "memory");
        asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                     ::"r"(sb + kCvRawOff + 16384), "l"((uint64_t)&tmC0), "r"(f * 64 + 32), "r"(row), "r"(bar_raw) : "memory");
    };
    if (tid == 0) {
        mbar_init_a(bar_raw, 1);
        mbar_init_a(bar_mma, 1);
        mbar_init_a(bar_w, 1);
        fence_barrier_init();
        mbar_expect_tx_a(bar_w, 16384);
        bulk_load(sb + kCvW, p.w_sw, 16384, bar_w);
        load_bin(f_begin);
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(s_tmem), "r"(64) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    for (int i = tid; i < O2 * O2 + O2; i += kCvThreads)
        asm volatile("st.shared.f32 [%0], %1;" ::"r"(s_w2 + 4 * i), "f"(i < O2 * O2 ? __ldg(p.w2 + i) : __ldg(p.bias + i - O2 * O2)) : "memory");
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = lds32(s_tmem);
    mbar_wait_a(bar_w, 0);
    const int r = tid & 127, half = tid >> 7;
    const bool zero = r0 + r < 0;   // before the start of the stream (for b > 0 the box holds the previous stream's rows)
    for (int f = f_begin, it = 0; f < f_end; f++, it++) {
        const uint32_t par = (uint32_t)(it & 1);
        mbar_wait_a(bar_raw, par);
        {   // fp32 rows -> BF16 hi / lo operand planes: thread = (time row, channel half)
            const uint32_t src = sb + kCvRawOff + (uint32_t)half * 16384u + (uint32_t)r * 128u;
            // all eight loads first: the shared-memory accesses are volatile asm statements, so a load placed after a store
            // in program order also waits for it -- as one loop every chunk paid the load latency (short-scoreboard was the
            // top stall of this kernel)
            float4 xs[8];
#pragma unroll
            for (int c = 0; c < 8; c++) xs[c] = lds128(src + (uint32_t)((c ^ (r & 7)) << 4));
#pragma unroll
            for (int c = 0; c < 8; c++) {
                float4 x = xs[c];
                if (zero) x = make_float4(0.f, 0.f, 0.f, 0.f);
                uint32_t h0, l0, h1, l1;
                bf16x2_split(x.x, x.y, h0, l0);
                bf16x2_split(x.z, x.w, h1, l1);
                const int cq = half * 8 + c;
                const uint32_t off = sb + sw128_off(r, cq >> 1) + (cq & 1) * 8;
                sts64(off, h0, h1);
                sts64(off + 16384, l0, l1);
            }
        }
        fence_proxy_async();
        tc_fence_before();
        __syncthreads();     // planes complete (and the raw boxes free; the previous bin's epilogue has left the Y tile)
        tc_fence_after();
        if (tid == 0 && f + 1 < f_end) load_bin(f + 1);   // overlaps the MMA and the epilogue below
        if (warp == 0) {
            constexpr uint32_t idesc = umma_idesc_bf16(128, 64);
            const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem, 0);
            const uint64_t ah = umma_desc_sw128(sb), al = umma_desc_sw128(sb + 16384);
            const uint64_t bh = umma_desc_sw128(sb + kCvW), bl = umma_desc_sw128(sb + kCvW + 8192);
#pragma unroll
            for (int k = 0; k < 4; k++) {
                umma_bf16_ss_elect(tmem_u, ah + 2 * k, bh + 2 * k, idesc, k != 0);
                umma_bf16_ss_elect(tmem_u, al + 2 * k, bh + 2 * k, idesc, 1u);
                umma_bf16_ss_elect(tmem_u, ah + 2 * k, bl + 2 * k, idesc, 1u);
            }
            asm volatile("{\n\t.reg .pred e;\n\telect.sync _|e, 0xffffffff;\n\t"
                         "@e tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}\n" ::"r"(bar_mma) : "memory");
        }
        mbar_wait_a(bar_mma, par);
        tc_fence_after();
        {   // Y -> shared memory: warp w holds TMEM lanes [32 (w % 4), +32) = time rows, columns [32 (w / 4), +32) = group w / 4
            const int q = warp & 3, g = warp >> 2;
            float v[32];
            tmem_ld32(tmem + ((uint32_t)(q * 32) << 16) + g * 32, v);
            const uint32_t dst = sb + kCvYs + (uint32_t)((q * 32 + lane) * kCvYld + g * NY) * 4u;
#pragma unroll
            for (int j = 0; j < NY; j++) asm volatile("st.shared.f32 [%0], %1;" ::"r"(dst + 4 * j), "f"(v[j]) : "memory");
        }
        tc_fence_before();
        __syncthreads();     // Y staged; the accumulator may be overwritten by the next bin's MMAs
        if (tid < 128) {
            const int t = r0 + tid;
            if (tid >= KTP - 1 && tid < KTP - 1 + kCvOut && t < p.T) {
                float z[O2];
#pragma unroll
                for (int g = 0; g < 2; g++)
#pragma unroll
                    for (int o = 0; o < ORDER; o++) {
                        float a = 0.f;
#pragma unroll
                        for (int dt = 0; dt < KTP; dt++) {
                            float y;
                            asm volatile("ld.shared.f32 %0, [%1];" : "=f"(y) : "r"(sb + kCvYs + (uint32_t)((tid - (KTP - 1) + dt) * kCvYld + g * NY + dt * ORDER + o) * 4u));
                            a += y;
                        }
                        z[g * ORDER + o] = a;
                    }
                float outv[O2];
#pragma unroll
                for (int qo = 0; qo < O2; qo++) {
                    float a;
                    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(a) : "r"(s_w2 + 4 * (O2 * O2 + qo)));
#pragma unroll
                    for (int k = 0; k < O2; k++) {
                        float w;
                        asm volatile("ld.shared.f32 %0, [%1];" : "=f"(w) : "r"(s_w2 + 4 * (k * O2 + qo)));
                        a = fmaf(z[k], w, a);
                    }
                    outv[qo] = fmaxf(a, 0.f);
                }
                float *dst = p.coefs + (((int64_t)b * p.T + t) * p.Fd + f) * O2;   // 40-byte rows: 8-byte aligned
#pragma unroll
                for (int qo = 0; qo < O2; qo += 2) *reinterpret_cast<float2 *>(dst + qo) = make_float2(outv[qo], outv[qo + 1]);
            }
        }
        // the next iteration's conversion writes the operand planes (read by the MMAs that completed above) and its
        // __syncthreads orders this bin's shifted sums before the next Y tile is staged
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem, 64);
}

// ================================================================ tensor-core GRU recurrence ====
// torch.nn.GRU cell (DeepFilterNet/df/modules.py:684,723), hidden size 256.  A cluster of 8 CTAs owns
// up to 16 streams for the whole sequence.  CTA `rank` keeps the W_hh rows of its 32 hidden units
// (3 gates x 32 rows x 256) resident in TENSOR MEMORY for the whole kernel as a BF16 hi/lo split
// (W = hi + lo to ~2^-17; lane = row, 2 x 128 columns); the hidden state of the group is the B
// operand in shared memory ([16 streams][256], BF16 hi/lo, K-major core matrices ordered so that a
// CTA's 32 units are one contiguous 2 KB piece).  Per time step one warp issues 48 tcgen05.mma
// (TS mode: A from TMEM, B from smem; M128 N16 K16, kind::f16: hi*hi + lo*hi + hi*lo, fp32
// accumulate in TMEM); eight warps read the pre-activations from TMEM, apply the gates in fp32,
// store the CTA's slice of the new state to a global scratch piece, and one thread asks the TMA
// engine for a multicast bulk copy of that piece into the operand buffer of every CTA of the
// cluster (itself included), which completes bytes on each CTA's mbarrier -- no cluster barrier
// on the step's critical path.  The fp32 hidden state of a CTA's own units stays in registers;
// only the MMA operand is BF16.
// Measured step timeline (clock64, 16 streams, profiles/r02_gru_anatomy.txt): 48 MMAs 450 cycles, commit ->
// gates 135, TMEM load + gates 645, fence 39, barrier + multicast through L2 + global stores 984  =>  2090 cycles / step
// (round 1, DSMEM exchange: 2380; the FFMA kernel k_gru: 4700).  History of the issue loop: `if (lane == 0)` around each
// MMA ~50 cycles per instruction (ptxas wrapped each in an ELECT / R2UR / BRA.U.ANY loop); every lane executing every
// call with a per-call elect 16.7; one elected lane running the whole loop 9.6 (the tensor pipe's rate at N = 16).
namespace cg = cooperative_groups;

constexpr int kGtU = 32, kGtRows = 3 * kGtU;   // hidden units / W_hh rows per CTA (both hidden sizes)
// gate threads: one per (unit pair, stream) item = 16 * NS; plus the MMA warp
// h operand (B, K-major, no swizzle) as 8 x 16 B core matrices ordered [k core matrix][row group][hi|lo]:
// a CTA's 32 units (4 k core matrices) are one contiguous piece (2 KB for 16 streams) -> one multicast bulk copy.
// NS = streams per cluster (MMA N): 16 (lowest step latency) or 32 (half as many clusters: the DF decoder's
// recurrence uses it for large batches so that it is co-resident with the ERB decoder's -- at most 15 clusters
// of 8 CTAs fit on the device, and two launches of 8 clusters made the second one run in two waves).
// HH = hidden size: 256 (cluster of 8, W_hh hi | lo both in tensor memory) or 512 (DeepFilterNet3_ll: cluster of 16
// -- non-portable size --, W_hh hi in tensor memory (256 columns), W_hh lo in shared memory as a second A operand).
template <int NS, int HH>
struct GtCfg {
    static constexpr int kC = HH / kGtU;              // CTAs per cluster: 8 / 16
    static constexpr int kGateThreads = 16 * NS;      // 256 / 512
    static constexpr int kGateWarps = kGateThreads / 32;
    static constexpr int kThreads = kGateThreads + 32;
    static constexpr int kMmaWarp = kGateThreads / 32;
    static constexpr int kLbo = (NS / 8) * 256;       // stride between K-adjacent core matrices
    static constexpr int kSbo = 256;                  // stride between 8-stream row groups
    static constexpr int kPlane = 128;                // hi -> lo
    static constexpr int kPiece = 4 * kLbo;           // one CTA's slice
    static constexpr int kBuf = (HH / 8) * kLbo;      // one buffer (16 KB / 32 KB at 256; 32 KB at 512 x 16)
    static constexpr int kWCols = HH / 2;             // TMEM columns of one W plane: 2 bf16 per 32-bit column
    // W_hh lo plane: K elements [0, kLoTmemK) live in tensor memory behind the hi plane, the rest (H = 512: the upper half;
    // 512 columns cannot hold hi + lo + accumulator) in shared memory as a second A operand (SS form)
    // (448, not 256, at H = 512: the accumulator needs only NS <= 32 of the 512 columns, and an SS-form MMA costs 40 cycles of
    // the tensor pipe against 16 for the TS form -- profiles/microbench/mma_rate.cu -- so 4 instead of 16 of the step's 96 MMAs
    // read their A operand from shared memory)
    static constexpr int kLoTmemK = HH > 256 ? 448 : HH;
    static constexpr bool kLoSmem = kLoTmemK < HH;
    static constexpr int kDCol = kWCols + kLoTmemK / 2;   // accumulator columns behind W_hi | W_lo[0, kLoTmemK): 256 / 384
    static constexpr int kWloBytes = kLoSmem ? ((HH - kLoTmemK) / 8) * 16 * 128 : 16;   // [k core matrix][16 row groups][8 x 16 B]
    static constexpr int kWloLbo = 16 * 128;          // stride between K-adjacent core matrices of the smem W_lo operand
};

template <int NS, int HH>
struct GruTcSmem {
    alignas(1024) unsigned char h[2][GtCfg<NS, HH>::kBuf];   // [buffer][k core matrix][row group][hi|lo][8 rows x 16 B]
    alignas(128) unsigned char wlo[GtCfg<NS, HH>::kWloBytes];  // (HH = 512) W_hh lo plane, K-major core matrices, 128 rows
    float pre[3][kGtU][NS + 1];
    alignas(8) uint64_t bar_h[2];
    uint64_t t_full;
    uint32_t tmem_base;
};

struct GruTcParams {
    const float *xproj;  // [B,T,3H]
    const float *whh;    // [3H][H]
    const float *bhh;    // [3H]
    const float *res;    // optional [B,T,H], added to the OUTPUT only
    float *hout;         // [B,T,H]
    unsigned short *hout_hi, *hout_lo;  // optional BF16 hi/lo planes of hout (A operand of the next projection GEMM)
    int planes_res;      // 1: the planes hold hout + res (input of a grouped linear), 0: the residual-free h
    // time-chunked execution: steps t = 0 .. T-1 are frames t0 + t of buffers holding Ts frames per stream; the
    // recurrence starts from h0 [B][H] (null: zeros) and leaves its final state in hT [B][H] (may alias h0)
    const float *h0;
    float *hT;
    int t0, Ts;
    int B, T, Bc;
    long long *dbg;      // optional [T][8] clock64 stamps of CTA 0 (0-3: MMA thread, 4-7: gate thread 0)
    unsigned char *xbuf; // exchange scratch in global memory [cluster][2][CTA][kPiece]
};


// The new state travels through L2 instead of SM to SM: per-peer DSMEM copies (15 x 4 KB out and in per CTA and step at
// H = 512 / 32 streams, ~20 B/cycle on the SM-to-SM network: more than half of the step) become one 4 KB read that the
// crossbar replicates.
template <int NS, int HH>
__global__ void __launch_bounds__(GtCfg<NS, HH>::kThreads, 1) k_gru_tc(GruTcParams p) {
    using Cfg = GtCfg<NS, HH>;
    constexpr int kGtThreads = Cfg::kThreads;
    constexpr int kGtH = HH, kGtC = Cfg::kC, kGtWCols = Cfg::kWCols, kGtDCol = Cfg::kDCol;
    extern __shared__ __align__(1024) unsigned char tc_smem_raw[];
    GruTcSmem<NS, HH> &sm = *reinterpret_cast<GruTcSmem<NS, HH> *>(((uintptr_t)tc_smem_raw + 1023) & ~uintptr_t(1023));
    cg::cluster_group cluster = cg::this_cluster();
    const int rank = (int)cluster.block_rank();
    const int group = blockIdx.x / kGtC;
    const int b0 = group * p.Bc;
    const int nb = min(p.Bc, p.B - b0);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int H = kGtH, T = p.T;
    for (int i = tid; i < (int)sizeof(sm.h) / 16; i += kGtThreads) reinterpret_cast<uint4 *>(&sm.h[0][0])[i] = make_uint4(0, 0, 0, 0);  // h0 = 0
    if (tid == 0) {
        mbar_init(&sm.bar_h[0], 1);   // MMA thread's expect_tx arrive
        mbar_init(&sm.bar_h[1], 1);
        mbar_init(&sm.t_full, 1);
        fence_barrier_init();
    }
    if (warp == 0) tmem_alloc(&sm.tmem_base, 512);
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = sm.tmem_base;
    const uint32_t tmem_d = tmem + kGtDCol;   // accumulator [128 lanes][NS columns]
    if (p.h0) {  // carried state: every CTA builds the whole operand h_{-1} of its streams in buffer 0
        for (int i = tid; i < nb * (kGtH / 2); i += kGtThreads) {
            const int s = i / (kGtH / 2), gu = (i - s * (kGtH / 2)) * 2;
            const float2 hv = *reinterpret_cast<const float2 *>(p.h0 + (int64_t)(b0 + s) * kGtH + gu);
            unsigned short h0b, l0b, h1b, l1b;
            bf16_split(hv.x, h0b, l0b);
            bf16_split(hv.y, h1b, l1b);
            const uint32_t off = (uint32_t)((gu >> 3) * Cfg::kLbo + (s >> 3) * Cfg::kSbo + (s & 7) * 16 + (gu & 7) * 2);
            *reinterpret_cast<uint32_t *>(sm.h[0] + off) = h0b | (uint32_t)h1b << 16;
            *reinterpret_cast<uint32_t *>(sm.h[0] + off + Cfg::kPlane) = l0b | (uint32_t)l1b << 16;
        }
        fence_proxy_async();
    }
    // ---- W_hh slice -> TMEM as BF16 hi | lo planes: lane = row rho (gate * 32 + unit; lanes 96..127 zero),
    //      column j of a plane = elements (2 j, 2 j + 1).  Warps 0-3 own lane quarters 0-3.
    if (warp < 4) {
        const int rho = warp * 32 + lane;
        const int g = rho / kGtU, u = rho - g * kGtU;
        const float *src = p.whh + ((int64_t)g * H + rank * kGtU + u) * H;
        for (int cb = 0; cb < kGtWCols / 32; cb++) {  // 32 columns = 64 elements per store
            uint32_t vh[32], vl[32];
#pragma unroll
            for (int i = 0; i < 32; i += 2) {
                float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
                if (rho < kGtRows) x = *reinterpret_cast<const float4 *>(src + cb * 64 + i * 2);
                unsigned short h0, l0, h1, l1, h2, l2, h3, l3;
                bf16_split(x.x, h0, l0); bf16_split(x.y, h1, l1); bf16_split(x.z, h2, l2); bf16_split(x.w, h3, l3);
                vh[i] = h0 | (uint32_t)h1 << 16; vh[i + 1] = h2 | (uint32_t)h3 << 16;
                vl[i] = l0 | (uint32_t)l1 << 16; vl[i + 1] = l2 | (uint32_t)l3 << 16;
            }
            const uint32_t ta = tmem + ((uint32_t)(warp * 32) << 16) + cb * 32;
            tmem_st32(ta, vh);
            if (cb * 64 < Cfg::kLoTmemK) {
                tmem_st32(ta + kGtWCols, vl);
            } else {
                // row rho, elements [64 cb, +64) = 8 core-matrix rows of 16 bytes: core matrix (k - kLoTmemK) / 8, row group rho / 8
                const uint32_t base = smem_u32(sm.wlo) + (uint32_t)(rho >> 3) * 128u + (uint32_t)(rho & 7) * 16u;
#pragma unroll
                for (int j = 0; j < 8; j++)
                    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(base + (uint32_t)(cb * 8 + j - Cfg::kLoTmemK / 8) * Cfg::kWloLbo),
                                 "r"(vl[4 * j]), "r"(vl[4 * j + 1]), "r"(vl[4 * j + 2]), "r"(vl[4 * j + 3]) : "memory");
            }
        }
        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
        if (Cfg::kLoSmem) fence_proxy_async();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    cluster.sync();  // every CTA's barriers are initialised and its h buffers zeroed before any remote copy
    const uint32_t step_bytes = (uint32_t)(kGtC * Cfg::kPiece);  // one piece from each CTA of the cluster, itself included

    if (warp == Cfg::kMmaWarp) {
        // ================================================================= MMA issuer (whole warp, elected lane issues)
        // ONE elected lane runs the whole time loop.  Inside an `if (elect_one())` region the compiler knows that a single lane
        // is active: the tcgen05.mma operands (tensor-memory addresses, shared-memory descriptors) stay in uniform registers
        // from step to step.  The earlier form -- all 32 lanes execute every call, each call elects its issuing lane -- made
        // it move four operands per MMA from vector to uniform registers under the elect predicate: 11-17 SASS instructions
        // and 16.7 cycles per MMA, against 9.6 cycles of tensor pipe at N = 16 (profiles/r02_mma_rate.txt).
        constexpr uint32_t idesc = umma_idesc_bf16(128, NS);
        if (elect_one()) {
            const uint32_t tmem_u = tmem, tmem_du = tmem_d;
            const uint64_t bd0 = umma_desc_interleave(smem_u32(sm.h[0]), Cfg::kLbo, Cfg::kSbo);
            const uint64_t bd1 = umma_desc_interleave(smem_u32(sm.h[1]), Cfg::kLbo, Cfg::kSbo);
            const uint64_t wlo_desc = umma_desc_interleave(smem_u32(sm.wlo), Cfg::kWloLbo, 128);
            (void)wlo_desc;
            const bool dbg_on = p.dbg && blockIdx.x == 0;
            for (int t = 0; t < T; t++) {
                const int cur = t & 1;
                if (dbg_on) p.dbg[t * 8 + 0] = clock64();
                if (t + 1 < T) mbar_expect_tx(&sm.bar_h[cur ^ 1], step_bytes);
                if (t > 0) mbar_wait(&sm.bar_h[cur], (uint32_t)(((t - 1) >> 1) & 1));
                if (dbg_on) p.dbg[t * 8 + 1] = clock64();
                fence_proxy_async();
                tc_fence_after();
                const uint64_t bb = cur ? bd1 : bd0;
#pragma unroll
                for (int combo = 0; combo < 3; combo++) {
                    const int wa = (combo == 1) ? 1 : 0, hb = (combo == 2) ? 1 : 0;  // hi*hi, lo*hi, hi*lo
#pragma unroll
                    for (int ks = 0; ks < kGtH / 16; ks++) {  // K step of 16: 8 TMEM columns of W, two core matrices of h
                        const uint64_t bdesc = bb + (uint64_t)((ks * 2 * Cfg::kLbo + hb * Cfg::kPlane) >> 4);
                        if (wa && ks * 16 >= Cfg::kLoTmemK) {   // tail of W_lo from shared memory (SS form): two core matrices per K step
                            umma_bf16_ss(tmem_du, wlo_desc + (uint64_t)(((ks - Cfg::kLoTmemK / 16) * 2 * Cfg::kWloLbo) >> 4), bdesc, idesc, 1u);
                        } else {
                            umma_bf16_ts(tmem_du, tmem_u + wa * kGtWCols + ks * 8, bdesc, idesc, (combo == 0 && ks == 0) ? 0u : 1u);
                        }
                    }
                }
                if (dbg_on) p.dbg[t * 8 + 2] = clock64();
                umma_commit(&sm.t_full);
            }
        }
        __syncwarp();
    } else {
        // ================================================================= gate warps (16 NS threads)
        // one item per thread: unit pair up = tid % 16 (units 2 up, 2 up + 1 of this CTA), stream s = tid / 16.
        // (The first 32-stream version kept 256 gate threads with two items each: 4550 cycles per step instead of 2600.)
        const int up = tid & 15, s = tid >> 4;
        const bool active = s < nb;
        const int gu = rank * kGtU + 2 * up;       // first of the two global hidden units of this thread
        float hprev0 = 0.f, hprev1 = 0.f;
        if (p.h0 && active) {
            const float2 hv = *reinterpret_cast<const float2 *>(p.h0 + (int64_t)(b0 + s) * H + gu);
            hprev0 = hv.x; hprev1 = hv.y;
        }
        const float2 bhr = *reinterpret_cast<const float2 *>(p.bhh + gu), bhz = *reinterpret_cast<const float2 *>(p.bhh + H + gu),
                     bhn = *reinterpret_cast<const float2 *>(p.bhh + 2 * H + gu);
        // byte offset of this (stream, unit pair) inside an h buffer (hi plane): core matrix gu / 8, row group s / 8
        const uint32_t hoff = (uint32_t)((gu >> 3) * Cfg::kLbo + (s >> 3) * Cfg::kSbo + (s & 7) * 16 + (gu & 7) * 2);
        const uint32_t piece0 = (uint32_t)(rank * Cfg::kPiece);  // this CTA's slice of a buffer
        // TMEM loaders: warp w reads lane quarter w % 4 (gates r, z, n = quarters 0-2), streams [16 (w / 4), +16)
        const bool loader = (warp & 3) < 3 && (warp >> 2) < NS / 16;
        for (int t = 0; t < T; t++) {
            const int cur = t & 1;
            float2 xr = make_float2(0.f, 0.f), xz = xr, xn = xr;
            uint32_t vhi = 0, vlo = 0;
            if (active) {
                const float *xp = p.xproj + ((int64_t)(b0 + s) * p.Ts + p.t0 + t) * (3 * H) + gu;
                xr = *reinterpret_cast<const float2 *>(xp);
                xz = *reinterpret_cast<const float2 *>(xp + H);
                xn = *reinterpret_cast<const float2 *>(xp + 2 * H);
                // xproj streams from HBM (3 KB per frame and stream, used once).  These loads are issued one MMA phase before
                // the gates need them; since that phase shrank to ~460 cycles (elected-lane issue) a load that misses L2 under
                // the feed-forward kernels' traffic arrived late (step 2070 cycles alone, 2525 inside the 128-stream pipeline).
                // Pull the rows of frame t + 3 into L2 now: no registers, and the load above becomes an L2 hit.
                if (t + 3 < T && (up & 7) == 0) {   // two requests per 128-byte line (16 threads x 8 bytes cover a gate's 32 units)
                    const float *xq = xp + 3 * (3 * H);
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(xq));
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(xq + H));
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(xq + 2 * H));
                }
            }
            const bool gdbg = p.dbg && blockIdx.x == 0 && tid == 0;
            if (gdbg) p.dbg[t * 8 + 4] = clock64();
            mbar_wait(&sm.t_full, (uint32_t)(t & 1));
            if (gdbg) p.dbg[t * 8 + 5] = clock64();
            tc_fence_after();
            if (loader) {  // TMEM lanes 32 g + u hold gate g of unit u; columns = streams
                const int g = warp & 3, q = warp >> 2;
                float v[16];
                tmem_ld16(tmem_d + ((uint32_t)(g * 32) << 16) + 16 * q, v);
#pragma unroll
                for (int ss = 0; ss < 16; ss++) sm.pre[g][lane][16 * q + ss] = v[ss];
            }
            tc_fence_before();
            asm volatile("bar.sync 1, %0;" ::"n"(Cfg::kGateThreads) : "memory");  // the gate warps only
            if (active) {
                const int u0 = 2 * up;
                const float r0 = gt_sigmoid(xr.x + sm.pre[0][u0][s] + bhr.x), r1 = gt_sigmoid(xr.y + sm.pre[0][u0 + 1][s] + bhr.y);
                const float z0 = gt_sigmoid(xz.x + sm.pre[1][u0][s] + bhz.x), z1 = gt_sigmoid(xz.y + sm.pre[1][u0 + 1][s] + bhz.y);
                const float n0 = gt_tanh(xn.x + r0 * (sm.pre[2][u0][s] + bhn.x)), n1 = gt_tanh(xn.y + r1 * (sm.pre[2][u0 + 1][s] + bhn.y));
                hprev0 = (1.f - z0) * n0 + z0 * hprev0;
                hprev1 = (1.f - z1) * n1 + z1 * hprev1;
                unsigned short h0, l0, h1, l1;
                bf16_split(hprev0, h0, l0);
                bf16_split(hprev1, h1, l1);
                vhi = h0 | (uint32_t)h1 << 16;
                vlo = l0 | (uint32_t)l1 << 16;
                if (t + 1 < T) {   // own piece of the scratch buffer (same layout as the shared-memory slice)
                    unsigned char *xp = p.xbuf + ((size_t)(group * 2 + (cur ^ 1)) * kGtC + rank) * Cfg::kPiece + (hoff - piece0);
                    *reinterpret_cast<uint32_t *>(xp) = vhi;
                    *reinterpret_cast<uint32_t *>(xp + Cfg::kPlane) = vlo;
                }
            }
            if (gdbg) p.dbg[t * 8 + 6] = clock64();
            if (t + 1 < T) {
                // own slice (generic stores) -> visible to the bulk-copy proxy
                fence_proxy_async_global();
                if (gdbg) p.dbg[t * 8 + 3] = clock64();
                asm volatile("bar.sync 1, %0;" ::"n"(Cfg::kGateThreads) : "memory");
                if (tid == 0) {
                    const unsigned char *xp = p.xbuf + ((size_t)(group * 2 + (cur ^ 1)) * kGtC + rank) * Cfg::kPiece;
                    bulk_load_multicast(smem_u32(sm.h[cur ^ 1]) + piece0, xp, Cfg::kPiece, smem_u32(&sm.bar_h[cur ^ 1]),
                                        (uint16_t)((1u << kGtC) - 1u));
                }
            } else {
                asm volatile("bar.sync 1, %0;" ::"n"(Cfg::kGateThreads) : "memory");
            }
            if (active) {  // global result last: nothing on the recurrence's critical path waits for it
                const int64_t o = ((int64_t)(b0 + s) * p.Ts + p.t0 + t) * H + gu;
                float2 ov = make_float2(hprev0, hprev1);
                if (p.hT && t + 1 == T) *reinterpret_cast<float2 *>(p.hT + (int64_t)(b0 + s) * H + gu) = ov;
                if (p.res) { const float2 rv = *reinterpret_cast<const float2 *>(p.res + o); ov.x += rv.x; ov.y += rv.y; }
                *reinterpret_cast<float2 *>(p.hout + o) = ov;
                if (p.hout_hi) {  // residual-free h (the next layer's projection input) or the layer output
                    if (p.planes_res && p.res) bf16x2_split(ov.x, ov.y, vhi, vlo);
                    *reinterpret_cast<uint32_t *>(p.hout_hi + o) = vhi;
                    *reinterpret_cast<uint32_t *>(p.hout_lo + o) = vlo;
                }
            }
            if (gdbg) p.dbg[t * 8 + 7] = clock64();
            // sm.pre is rewritten only after the next t_full, i.e. after every CTA's copies of this step
        }
    }
    tc_fence_before();
    __syncthreads();
    cluster.sync();  // no CTA exits while peers may still address its shared memory
    if (warp == 0) tmem_dealloc(tmem, 512);
}

// exchange scratch of the recurrence: one buffer per (device, stream) -- launches on one stream are serialised, the two
// decoders' recurrences run on different streams
static unsigned char *gru_xbuf(cudaStream_t s, size_t bytes) {
    struct Ent { unsigned char *p = nullptr; size_t cap = 0; };
    static std::mutex mu;
    static std::map<std::pair<int, cudaStream_t>, Ent> pool;
    int dev = 0;
    cudaGetDevice(&dev);
    std::lock_guard<std::mutex> lk(mu);
    Ent &e = pool[{dev, s}];
    if (e.cap < bytes) {
        if (e.p) { cudaDeviceSynchronize(); cudaFree(e.p); e.p = nullptr; e.cap = 0; }
        const size_t want = (bytes + (1u << 20)) & ~size_t((1u << 20) - 1);
        if (cudaMalloc(&e.p, want) != cudaSuccess) { e.p = nullptr; return nullptr; }
        e.cap = want;
    }
    return e.p;
}

template <int NS, int HH>
static int launch_gru_tc_n(cudaStream_t s, GruTcParams p) {
    using Cfg = GtCfg<NS, HH>;
    static PerDeviceOnce attr_once;
    // the kernel allocates all 512 TMEM columns (W_hh lives there), so only one CTA may be resident per SM: request more
    // than half of the shared memory to enforce it.  (Tried: 256 + 32 columns, half the registers and 115 KB so that
    // feed-forward CTAs could share the SMs a recurrence occupies but hardly uses -- no gain at 128 or 512 streams.)
    const int need = (int)sizeof(GruTcSmem<NS, HH>) + 1024;
    // (also tried: the whole 227 KB carve-out, so that no feed-forward CTA can sit next to a recurrence CTA and wait in
    // tcgen05.alloc -- no change at 128 x 10 s with 1 .. 4 device chunks, 512 x 10 s: 45.2 vs 45.3 ms)
    const int smem = need > 120 * 1024 ? need : 120 * 1024;
    if (auto once_guard = attr_once.first()) {
        if (Cfg::kC > 8) DFB_CUDA(cudaFuncSetAttribute(k_gru_tc<NS, HH>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
        DFB_CUDA(cudaFuncSetAttribute(k_gru_tc<NS, HH>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    }
    cudaLaunchConfig_t cfg{};
    cfg.blockDim = dim3(Cfg::kThreads);
    cfg.dynamicSmemBytes = smem;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = Cfg::kC; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    p.Bc = NS;
    const int ngroups = (p.B + NS - 1) / NS;
    cfg.gridDim = dim3((unsigned)(ngroups * Cfg::kC));
    cfg.stream = s;
    p.xbuf = gru_xbuf(s, (size_t)ngroups * 2 * Cfg::kC * Cfg::kPiece);
    if (!p.xbuf) return fail(DFB_ERR_OOM, "GRU exchange scratch");
    DFB_PROF(HH == 256 ? "k_gru_tc" : "k_gru_tc512", s);
    DFB_CUDA(cudaLaunchKernelEx(&cfg, k_gru_tc<NS, HH>, p));
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return DFB_OK;
}

// wide != 0: 32 streams per cluster when the batch needs more than 4 clusters of 16 (see GtCfg).  H = 512: clusters of
// 16 CTAs with 16 or 32 streams.
int launch_gru_tc(cudaStream_t s, const float *xproj, const float *whh, const float *bhh, const float *res, float *hout,
                  unsigned short *hout_hi, unsigned short *hout_lo, int B, int T, long long *dbg, int wide, int planes_res,
                  const GruWindow *w, int H) {
    GruTcParams p{xproj, whh, bhh, res, hout, hout_hi, hout_lo, planes_res, w ? w->h0 : nullptr, w ? w->hT : nullptr,
                  w ? w->t0 : 0, w ? w->Ts : T, B, T, 0, dbg};
    // (Tried: a "ping-pong" kernel in which a cluster owns 2 or 3 independent sub-batches of 16 streams -- own state buffers,
    // accumulator columns, barriers and 8 gate warps each, one MMA warp serving them in turn -- so that one sub-batch's
    // MMAs fill the other's gate / exchange latency.  Correct (parity tests green), but 48 MMAs of N = 16 take ~800 cycles to
    // issue (16.7 per instruction, twice their math time), so two sub-batches keep the MMA warp busy 1800 of the 2650-cycle
    // chain and the chain itself stretches: 3127 cycles per step for 2 x 16 streams vs 3050 for one N = 32 batch, 3947 for
    // 3 x 16; 128 x 10 s 11.75 vs 11.31 ms.)
    // exchange through L2 + multicast instead of per-peer DSMEM copies, measured: H = 512 256 x 10 s 60.8 -> 51.0 ms,
    // 32 x 10 s 12.0 -> 9.5 ms; H = 256 / 32 streams: 512 x 10 s 43.9 -> 41.6 ms; H = 256 / 16 streams: 128 x 10 s
    // 11.88 -> 11.34 ms, 32 x 10 s 5.57 -> 5.09 ms, batch 1 3.79 -> 3.62 ms.
    if (H == 512) return B > 128 ? launch_gru_tc_n<32, 512>(s, p) : launch_gru_tc_n<16, 512>(s, p);
    if (H != 256) return fail(DFB_ERR_UNSUPPORTED, "tensor-core recurrence: hidden size %d", H);
    // 16 streams per cluster have the shortest step (2600 cycles vs 3830 for 32) but 36 % more cluster time per stream:
    // from 256 streams on a launch needs several waves of the 15 co-resident clusters anyway, and 32 per cluster are faster
    // (512 x 10 s DeepFilterNet2: 48.1 -> 45.3 ms per step)
    const bool use32 = (wide && B > 64) || B >= 256;
    // beyond 15 x 32 streams a launch of 32-stream clusters needs a second wave of the 15 co-resident clusters (512 streams:
    // 16 clusters -> twice the time); 48 streams per cluster (N = 48, 768 gate threads) keep 512 streams in one wave
    if (use32 && B > 15 * 32) return launch_gru_tc_n<48, 256>(s, p);
    return use32 ? launch_gru_tc_n<32, 256>(s, p) : launch_gru_tc_n<16, 256>(s, p);
}

int cached_map_f32_sw128(CUtensorMap *out, const void *base, int64_t rows, int64_t cols, int64_t ld, int box_rows);

// c0 [B,T,Fd,64] -> coefs [B,T,Fd,10] (pathway term), tensor-core version; w_sw: host-packed operand image (weights.py)
int launch_df_convp_tc(cudaStream_t s, const float *c0, const float *w_sw, const float *w2, const float *bias, float *coefs, int B, int T,
                       int Fd) {
    if ((int64_t)B * T >= (int64_t(1) << 31) - 256 || B > 65535) return fail(DFB_ERR_UNSUPPORTED, "df pathway conv: batch too large for one launch");
    CUtensorMap mc;
    int rc;
    if ((rc = cached_map_f32_sw128(&mc, c0, (int64_t)B * T, (int64_t)Fd * kCh, (int64_t)Fd * kCh, 128))) return rc;
    const int smem = 1024 + (int)kCvTail + 512 + 64;
    static PerDeviceOnce attr_once;
    if (auto once_guard = attr_once.first())
        DFB_CUDA(cudaFuncSetAttribute(k_df_convp_tc<5, 5>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    CvParams p{w_sw, w2, bias, coefs, T, Fd};
    dim3 grid((unsigned)((Fd + kCvBins - 1) / kCvBins), (unsigned)((T + kCvOut - 1) / kCvOut), (unsigned)B);
    DFB_PROF("k_df_convp_tc", s);
    k_df_convp_tc<5, 5><<<grid, kCvThreads, smem, s>>>(mc, p);
    DFB_LAUNCH_CHECK();
    return DFB_OK;
}

// ------------------------------------------------------------------------------- host side ----
int cached_map_bf16(CUtensorMap *out, const void *base, int64_t rows, int64_t cols, int64_t ld, int box_rows);  // dfb_gl.cu

// Y[M,N] = X . W^T + bias with X, W given as BF16 hi/lo planes (X: [M][K] pitch ldx, W: [N][K] pitch K)
int launch_gemm_bf16x3(cudaStream_t s, const void *x_hi, const void *x_lo, int64_t ldx, const void *w_hi, const void *w_lo,
                       const float *bias, float *y, int64_t ldy, int64_t M, int N, int K) {
    if (N % kBxBN || K % kBxBK || (K > kBxMaxK && K % kBxMaxK) || (ldx % 8) || M <= 0 || ((uintptr_t)w_hi & 15) || ((uintptr_t)w_lo & 15))
        return fail(DFB_ERR_UNSUPPORTED, "bf16x3 GEMM shape M=%lld N=%d K=%d", (long long)M, N, K);
    CUtensorMap mxh, mxl;
    int rc;
    // (cached per (base, shape): the arenas hand out the same addresses call after call)
    if ((rc = cached_map_bf16(&mxh, x_hi, M, K, ldx, kBxBM)) || (rc = cached_map_bf16(&mxl, x_lo, M, K, ldx, kBxBM))) return rc;
    static PerDeviceOnce attr_once;
    const int smem = (int)sizeof(BxSmem) + 1024;
    if (auto once_guard = attr_once.first()) DFB_CUDA(cudaFuncSetAttribute(k_gemm_bf16x3, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    int dev = 0, num_sms = 0;
    DFB_CUDA(cudaGetDevice(&dev));
    DFB_CUDA(cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev));
    // persistent: one CTA per SM; blockIdx.x = column slice (fastest, so the CTAs that stream the same X tiles are
    // co-scheduled and share them through L2), blockIdx.y = row group
    const int nslices = N / kBxBN;
    const int ntiles = (int)((M + kBxBM - 1) / kBxBM);
    int groups = num_sms / nslices;
    if (groups < 1) groups = 1;
    if (groups > ntiles) groups = ntiles;
    dim3 grid((unsigned)nslices, (unsigned)groups);
    const int kpass = K > kBxMaxK ? kBxMaxK : K;
    for (int k0 = 0; k0 < K; k0 += kpass) {
        DFB_PROF("k_gemm_bf16x3[gru_proj]", s);
        k_gemm_bf16x3<<<grid, kBxThreads, smem, s>>>(mxh, mxl, reinterpret_cast<const unsigned short *>(w_hi),
                                                  reinterpret_cast<const unsigned short *>(w_lo), bias, y, ldy, (int)M, N, kpass, K, k0,
                                                  k0 > 0 ? 1 : 0);
        DFB_LAUNCH_CHECK();
    }
    return DFB_OK;
}

}  // namespace dfb
