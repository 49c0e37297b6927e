// dfb_fft.cuh -- fp32 FFT building blocks for the real transforms of the DeepFilterNet analysis /
// synthesis kernels (sm_100a): the specialised 960-point transform of the shipped models and a
// runtime mixed-radix transform for every other supported fft_size (end of this file).
//
// The reference computes these with realfft 3.3.0 / rustfft 6.2.0 (libDF/src/lib.rs:117-118,
// :385-388, :398-405): an unnormalised real DFT of length N = fft_size and its inverse.
// Here: N-point real transform = N/2-point complex transform + split post/pre-processing;
// the N/2 = 480-point complex transform is a two-pass (20 x 24) Cooley-Tukey held by one warp:
// every lane runs a 20- resp. 24-point DFT entirely in registers (compile-time generated
// radix-{2,3,4,5} butterflies with literal twiddles) and the transpose between the two passes
// goes through a per-warp shared-memory tile.
//
// Everything below is __host__ __device__ so that tests/host/fft_host_test.cu and
// tests/host/fft_any_host_test.cu can emulate the 32 lanes on the CPU and check the index algebra
// against a double-precision DFT.
#pragma once
#include <cuda_runtime.h>

#include <utility>

#define DFB_HD __host__ __device__ __forceinline__
#define DFB_CX __host__ __device__ constexpr

namespace dfb {

// ---------------------------------------------------------------- compile-time trig ----
constexpr double kPi = 3.14159265358979323846264338327950288;

DFB_CX double cx_sin_small(double x) {  // |x| <= pi/4
    double term = x, sum = x, x2 = x * x;
    for (int i = 1; i < 14; i++) {
        term *= -x2 / double((2 * i) * (2 * i + 1));
        sum += term;
    }
    return sum;
}
DFB_CX double cx_cos_small(double x) {
    double term = 1, sum = 1, x2 = x * x;
    for (int i = 1; i < 14; i++) {
        term *= -x2 / double((2 * i - 1) * (2 * i));
        sum += term;
    }
    return sum;
}
// cos / sin of 2*pi*k/n with exact integer octant reduction
DFB_CX long cx_mod(long k, long n) { return ((k % n) + n) % n; }
DFB_CX int cx_quadrant(long k, long n) { return int((8 * cx_mod(k, n) + n) / (2 * n)) % 4; }  // round(4k/n)
DFB_CX double cx_resid(long k, long n) {
    long km = cx_mod(k, n);
    long q = (8 * km + n) / (2 * n);
    return 2.0 * kPi * double(4 * km - q * n) / double(4 * n);
}
DFB_CX double cx_cos2pi(long k, long n) {
    int q = cx_quadrant(k, n);
    double r = cx_resid(k, n);
    return q == 0 ? cx_cos_small(r) : q == 1 ? -cx_sin_small(r) : q == 2 ? -cx_cos_small(r) : cx_sin_small(r);
}
DFB_CX double cx_sin2pi(long k, long n) {
    int q = cx_quadrant(k, n);
    double r = cx_resid(k, n);
    return q == 0 ? cx_sin_small(r) : q == 1 ? cx_cos_small(r) : q == 2 ? -cx_sin_small(r) : -cx_cos_small(r);
}

// --------------------------------------------------------------------- complex helpers ----
DFB_HD float2 cadd(float2 a, float2 b) { return make_float2(a.x + b.x, a.y + b.y); }
DFB_HD float2 csub(float2 a, float2 b) { return make_float2(a.x - b.x, a.y - b.y); }
DFB_HD float2 cmul(float2 a, float2 b) { return make_float2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x); }
DFB_HD float2 cconj(float2 a) { return make_float2(a.x, -a.y); }
DFB_HD float2 cscale(float2 a, float s) { return make_float2(a.x * s, a.y * s); }
// multiply by -i (forward) or +i (inverse)
template <bool INV>
DFB_HD float2 cmul_mi(float2 a) {
    return INV ? make_float2(-a.y, a.x) : make_float2(a.y, -a.x);
}

// a * e^{-+ 2 pi i K / N}   (minus sign for the forward transform)
template <int N, int K, bool INV>
DFB_HD float2 twmul(float2 a) {
    constexpr int k = ((K % N) + N) % N;
    if constexpr (k == 0) {
        return a;
    } else if constexpr (2 * k == N) {
        return make_float2(-a.x, -a.y);
    } else if constexpr (4 * k == N) {
        return cmul_mi<INV>(a);
    } else if constexpr (4 * k == 3 * N) {
        return cmul_mi<!INV>(a);
    } else {
        constexpr float c = float(cx_cos2pi(k, N));
        constexpr float s = float(INV ? cx_sin2pi(k, N) : -cx_sin2pi(k, N));
        return make_float2(a.x * c - a.y * s, a.x * s + a.y * c);
    }
}

// --------------------------------------------------- in-register DFT<N>, natural order ----
template <int N, bool INV>
struct Dft;

template <bool INV>
struct Dft<1, INV> {
    static DFB_HD void run(float2 (&)[1]) {}
};

template <bool INV>
struct Dft<2, INV> {
    static DFB_HD void run(float2 (&v)[2]) {
        float2 a = v[0], b = v[1];
        v[0] = cadd(a, b);
        v[1] = csub(a, b);
    }
};

template <bool INV>
struct Dft<3, INV> {
    static DFB_HD void run(float2 (&v)[3]) {
        constexpr float s3 = float(cx_sin2pi(1, 3));  // sqrt(3)/2
        float2 s = cadd(v[1], v[2]), d = csub(v[1], v[2]);
        float2 m = make_float2(v[0].x - 0.5f * s.x, v[0].y - 0.5f * s.y);
        float2 q = cmul_mi<INV>(cscale(d, s3));  // -+ i * s3 * d
        v[0] = cadd(v[0], s);
        v[1] = cadd(m, q);
        v[2] = csub(m, q);
    }
};

template <bool INV>
struct Dft<4, INV> {
    static DFB_HD void run(float2 (&v)[4]) {
        float2 t0 = cadd(v[0], v[2]), t1 = csub(v[0], v[2]);
        float2 t2 = cadd(v[1], v[3]), t3 = cmul_mi<INV>(csub(v[1], v[3]));
        v[0] = cadd(t0, t2);
        v[2] = csub(t0, t2);
        v[1] = cadd(t1, t3);
        v[3] = csub(t1, t3);
    }
};

template <bool INV>
struct Dft<5, INV> {
    static DFB_HD void run(float2 (&v)[5]) {
        constexpr float c1 = float(cx_cos2pi(1, 5)), c2 = float(cx_cos2pi(2, 5));
        constexpr float s1 = float(cx_sin2pi(1, 5)), s2 = float(cx_sin2pi(2, 5));
        float2 a1 = cadd(v[1], v[4]), a2 = cadd(v[2], v[3]);
        float2 d1 = csub(v[1], v[4]), d2 = csub(v[2], v[3]);
        float2 p1 = make_float2(v[0].x + c1 * a1.x + c2 * a2.x, v[0].y + c1 * a1.y + c2 * a2.y);
        float2 p2 = make_float2(v[0].x + c2 * a1.x + c1 * a2.x, v[0].y + c2 * a1.y + c1 * a2.y);
        float2 q1 = cmul_mi<INV>(make_float2(s1 * d1.x + s2 * d2.x, s1 * d1.y + s2 * d2.y));
        float2 q2 = cmul_mi<INV>(make_float2(s2 * d1.x - s1 * d2.x, s2 * d1.y - s1 * d2.y));
        v[0] = cadd(v[0], cadd(a1, a2));
        v[1] = cadd(p1, q1);
        v[4] = csub(p1, q1);
        v[2] = cadd(p2, q2);
        v[3] = csub(p2, q2);
    }
};

template <bool INV>
struct Dft<7, INV> {
    static DFB_HD void run(float2 (&v)[7]) {
        constexpr float c1 = float(cx_cos2pi(1, 7)), c2 = float(cx_cos2pi(2, 7)), c3 = float(cx_cos2pi(3, 7));
        constexpr float s1 = float(cx_sin2pi(1, 7)), s2 = float(cx_sin2pi(2, 7)), s3 = float(cx_sin2pi(3, 7));
        float2 a1 = cadd(v[1], v[6]), a2 = cadd(v[2], v[5]), a3 = cadd(v[3], v[4]);
        float2 d1 = csub(v[1], v[6]), d2 = csub(v[2], v[5]), d3 = csub(v[3], v[4]);
        // X[k] = v0 + sum_m cos(2 pi k m / 7) a_m -+ i sum_m sin(2 pi k m / 7) d_m,  X[7-k] with the opposite sign
        float2 p1 = make_float2(v[0].x + c1 * a1.x + c2 * a2.x + c3 * a3.x, v[0].y + c1 * a1.y + c2 * a2.y + c3 * a3.y);
        float2 p2 = make_float2(v[0].x + c2 * a1.x + c3 * a2.x + c1 * a3.x, v[0].y + c2 * a1.y + c3 * a2.y + c1 * a3.y);
        float2 p3 = make_float2(v[0].x + c3 * a1.x + c1 * a2.x + c2 * a3.x, v[0].y + c3 * a1.y + c1 * a2.y + c2 * a3.y);
        float2 q1 = cmul_mi<INV>(make_float2(s1 * d1.x + s2 * d2.x + s3 * d3.x, s1 * d1.y + s2 * d2.y + s3 * d3.y));
        float2 q2 = cmul_mi<INV>(make_float2(s2 * d1.x - s3 * d2.x - s1 * d3.x, s2 * d1.y - s3 * d2.y - s1 * d3.y));
        float2 q3 = cmul_mi<INV>(make_float2(s3 * d1.x - s1 * d2.x + s2 * d3.x, s3 * d1.y - s1 * d2.y + s2 * d3.y));
        v[0] = cadd(v[0], cadd(a1, cadd(a2, a3)));
        v[1] = cadd(p1, q1);
        v[6] = csub(p1, q1);
        v[2] = cadd(p2, q2);
        v[5] = csub(p2, q2);
        v[3] = cadd(p3, q3);
        v[4] = csub(p3, q3);
    }
};

template <int N>
struct Factor {
    static constexpr int P = (N % 4 == 0) ? 4 : (N % 2 == 0) ? 2 : (N % 3 == 0) ? 3 : (N % 5 == 0) ? 5 : N;
    static_assert(P != N || N <= 5, "unsupported DFT size");
};

// decimation in time: X[k + M q] = sum_r w_P^{r q} ( w_N^{r k} Y_r[k] ),  Y_r = DFT_M(x[r + P m])
template <int N, bool INV>
struct Dft {
    static constexpr int P = Factor<N>::P;
    static constexpr int M = N / P;

    template <int K>
    static DFB_HD void combine(float2 (&sub)[P][M], float2 (&v)[N]) {
        float2 t[P];
        comb_load<K>(sub, t, std::make_integer_sequence<int, P>{});
        Dft<P, INV>::run(t);
#pragma unroll
        for (int q = 0; q < P; q++) v[K + M * q] = t[q];
    }
    template <int K, int... R>
    static DFB_HD void comb_load(float2 (&sub)[P][M], float2 (&t)[P], std::integer_sequence<int, R...>) {
        ((t[R] = twmul<N, R * K, INV>(sub[R][K])), ...);
    }
    template <int... K>
    static DFB_HD void combine_all(float2 (&sub)[P][M], float2 (&v)[N], std::integer_sequence<int, K...>) {
        (combine<K>(sub, v), ...);
    }
    static DFB_HD void run(float2 (&v)[N]) {
        float2 sub[P][M];
#pragma unroll
        for (int r = 0; r < P; r++) {
#pragma unroll
            for (int m = 0; m < M; m++) sub[r][m] = v[r + P * m];
            Dft<M, INV>::run(sub[r]);
        }
        combine_all(sub, v, std::make_integer_sequence<int, M>{});
    }
};

// ----------------------------------------------------------- 480-point warp transform ----
// n = 24 n1 + n2 (n1 < 20, n2 < 24),  k = k1 + 20 k2 (k1 < 20, k2 < 24)
//   pass A, lane n2 < 24:  A[k1] = DFT20_{n1}( z[24 n1 + n2] ) * w480^{n2 k1}   -> tile[k1][n2]
//   pass B, lane k1 < 20:  Z[k1 + 20 k2] = DFT24_{n2}( tile[k1][n2] )
constexpr int kC = 480;          // complex length
constexpr int kN1 = 20, kN2 = 24;
constexpr int kTileStride = 25;  // float2 units; 25 keeps the pass-B column reads conflict free
constexpr int kTileFloat2 = kN1 * kTileStride;  // 500 float2 = 4000 B per warp

// Pass A for one lane.  `a` holds z[24 n1 + lane] (n1 = 0..19); `tw` -> w480^{-+ lane k1} (k1 = 0..19), e.g. in shared memory.
template <bool INV>
DFB_HD void fft480_pass_a(float2 (&a)[kN1], const float2* tw, float2* tile, int lane) {
    Dft<kN1, INV>::run(a);
#pragma unroll
    for (int k1 = 0; k1 < kN1; k1++) tile[k1 * kTileStride + lane] = cmul(a[k1], tw[k1]);
}

// Pass B, read phase: lane k1 < 20 gathers its column and transforms it.
template <bool INV>
DFB_HD void fft480_pass_b(float2 (&b)[kN2], const float2* tile, int lane) {
#pragma unroll
    for (int n2 = 0; n2 < kN2; n2++) b[n2] = tile[lane * kTileStride + n2];
    Dft<kN2, INV>::run(b);
}
// Pass B, write phase (after a warp sync): natural order Z[k1 + 20 k2] into buf[0..480)
DFB_HD void fft480_store_natural(const float2 (&b)[kN2], float2* buf, int lane) {
#pragma unroll
    for (int k2 = 0; k2 < kN2; k2++) buf[lane + kN1 * k2] = b[k2];
}

// Split step of the real forward transform of length N = 2 M (960 for the shipped models): from
// Z = DFT_M(x[2n] + i x[2n+1]),
//   X[k] = (Z[k] + conj Z[M-k])/2 - i w_N^k (Z[k] - conj Z[M-k])/2,  Z[M] := Z[0]
// returns X[k] and X[M-k] for one k in [0, M/2]; w = e^{-2 pi i k / N}
DFB_HD void rfft_split(float2 zk, float2 znk, float2 w, float2& xk, float2& xnk) {
    float2 e = make_float2(0.5f * (zk.x + znk.x), 0.5f * (zk.y - znk.y));   // (Z[k] + conj Z[n-k]) / 2
    float2 d = make_float2(0.5f * (zk.x - znk.x), 0.5f * (zk.y + znk.y));   // (Z[k] - conj Z[n-k]) / 2
    float2 o = cmul(make_float2(d.y, -d.x), w);                             // -i d w
    xk = cadd(e, o);
    // X[M-k] = conj(e) - conj(o) ... derived from the same pair:  e' = conj(e), d' = -conj(d), w' = -conj(w)
    xnk = make_float2(e.x - o.x, -(e.y - o.y));
}

// Merge step of the real inverse transform: from X[k], X[M-k] (k in [0, M/2]) build
//   Z[k] = (X[k] + conj X[M-k]) + i w_N^{-k} (X[k] - conj X[M-k])   (unnormalised irfft)
// and Z[M-k]; wc = e^{+2 pi i k / N}
DFB_HD void irfft_merge(float2 xk, float2 xnk, float2 wc, float2& zk, float2& znk) {
    float2 e = make_float2(xk.x + xnk.x, xk.y - xnk.y);
    float2 d = make_float2(xk.x - xnk.x, xk.y + xnk.y);
    float2 o = cmul(make_float2(-d.y, d.x), wc);  // i d wc
    zk = cadd(e, o);
    znk = make_float2(e.x - o.x, -(e.y - o.y));
}

// ------------------------------------------------ runtime mixed-radix transform (any M) ----
// The analysis / synthesis kernels of every other STFT geometry (k_analysis_any, k_apply_synthesis_any) run the
// M = fft_size / 2 point complex transform as a Stockham autosort FFT in shared memory: one pass per radix of the plan
// (fft_next_radix), natural order in and out, ping-pong between two M-point buffers.  One code path serves
// every supported size; the radix of a pass is a runtime switch over the compile-time butterflies above.
constexpr int kAnyMaxM = 2048;     // fft_size <= 4096

// radix of the next pass for the remaining length r (4 first, then 2, 3, 5, 7); 0: a prime factor above 7 is left
DFB_HD int fft_next_radix(int r) {
    return r % 4 == 0 ? 4 : r % 2 == 0 ? 2 : r % 3 == 0 ? 3 : r % 5 == 0 ? 5 : r % 7 == 0 ? 7 : 0;
}
inline bool fft_any_supported(int M) {
    if (M < 1 || M > kAnyMaxM) return false;
    while (M > 1) {
        const int p = fft_next_radix(M);
        if (!p) return false;
        M /= p;
    }
    return true;
}

// One radix-P pass (Stockham, decimation in time).  Ns = product of the radices of the earlier passes; butterfly
// j < M/P of lane `lane` (stride nlanes):
//   v_r = src[j + r M/P] * w_{Ns P}^{-+ r (j mod Ns)},  v = DFT_P(v),  dst[(j - j mod Ns) P + j mod Ns + r Ns] = v_r
// tw[k] = e^{-2 pi i k / M} (w_{Ns P}^{m} = tw[m M / (Ns P)]); the inverse conjugates it.
template <int P, bool INV>
DFB_HD void stockham_pass(const float2 *src, float2 *dst, const float2 *tw, int M, int Ns, int lane, int nlanes) {
    const int q = M / P, tstep = M / (Ns * P);
    for (int j = lane; j < q; j += nlanes) {
        const int jm = j % Ns;
        float2 v[P];
#pragma unroll
        for (int r = 0; r < P; r++) {
            float2 x = src[j + r * q];
            if (r > 0 && jm > 0) {
                float2 w = tw[jm * r * tstep];
                if (INV) w.y = -w.y;
                x = cmul(x, w);
            }
            v[r] = x;
        }
        Dft<P, INV>::run(v);
        const int d = (j - jm) * P + jm;
#pragma unroll
        for (int r = 0; r < P; r++) dst[d + r * Ns] = v[r];
    }
}

template <bool INV>
DFB_HD void fft_any_pass(int P, const float2 *src, float2 *dst, const float2 *tw, int M, int Ns, int lane, int nlanes) {
    switch (P) {
        case 4: stockham_pass<4, INV>(src, dst, tw, M, Ns, lane, nlanes); break;
        case 2: stockham_pass<2, INV>(src, dst, tw, M, Ns, lane, nlanes); break;
        case 3: stockham_pass<3, INV>(src, dst, tw, M, Ns, lane, nlanes); break;
        case 5: stockham_pass<5, INV>(src, dst, tw, M, Ns, lane, nlanes); break;
        default: stockham_pass<7, INV>(src, dst, tw, M, Ns, lane, nlanes); break;
    }
}

}  // namespace dfb
