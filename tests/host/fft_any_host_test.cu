// Host-side emulation of the runtime mixed-radix real FFT in deepfilternet_b200/csrc/dfb_fft.cuh (the transform of
// k_analysis_any / k_apply_synthesis_any): the 32 lanes of every Stockham pass run sequentially on the CPU, followed by
// the real split / merge steps, and the result is checked against a double-precision DFT.
// Usage: fft_any_host_test N [N ...]; prints one line per size, exit code 1 when a size misses 1e-5 * max|X|.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "../../deepfilternet_b200/csrc/dfb_fft.cuh"
using namespace dfb;

// table entries exactly as dfb_state_create builds them
static std::vector<float2> tw_m(int M) {
    std::vector<float2> t(M);
    for (int k = 0; k < M; k++) {
        double a = 2.0 * M_PI * (double)k / (double)M;
        t[k] = make_float2((float)cos(a), (float)-sin(a));
    }
    return t;
}
static std::vector<float2> tw_split(int N) {
    std::vector<float2> t(N / 4 + 1);
    for (int k = 0; k <= N / 4; k++) {
        double a = 2.0 * M_PI * (double)k / (double)N;
        t[k] = make_float2((float)cos(a), (float)-sin(a));
    }
    return t;
}

// the warp loop of the kernels: every pass reads one buffer and writes the other, so running the lanes one after
// another is what the warp does between two __syncwarp()s
template <bool INV>
static float2 *run_passes(int M, float2 *a, float2 *b, const float2 *tw, int *passes) {
    *passes = 0;
    for (int r = M, Ns = 1; r > 1; (*passes)++) {
        const int P = fft_next_radix(r);
        for (int lane = 0; lane < 32; lane++) fft_any_pass<INV>(P, a, b, tw, M, Ns, lane, 32);
        Ns *= P;
        r /= P;
        float2 *t = a; a = b; b = t;
    }
    return a;
}

int main(int argc, char **argv) {
    int bad = 0;
    for (int ai = 1; ai < argc; ai++) {
        const int N = atoi(argv[ai]), M = N / 2, F = M + 1;
        int passes = 0;
        if (N % 2 || !fft_any_supported(M)) { printf("N=%d unsupported\n", N); bad = 1; continue; }
        const std::vector<float2> tw = tw_m(M), tws = tw_split(N);
        std::vector<double> x(N);
        srand(1000 + N);
        for (auto &v : x) v = (float)(rand() / (double)RAND_MAX - 0.5);
        // reference spectrum (double)
        std::vector<double> Xr(F), Xi(F);
        double xmax = 0;
        for (int k = 0; k < F; k++) {
            double ar = 0, ai2 = 0;
            for (int n = 0; n < N; n++) {
                double ang = -2.0 * M_PI * (double)((long)k * n % N) / N;
                ar += x[n] * cos(ang);
                ai2 += x[n] * sin(ang);
            }
            Xr[k] = ar; Xi[k] = ai2;
            xmax = fmax(xmax, hypot(ar, ai2));
        }
        // forward: z[n] = x[2n] + i x[2n+1], M-point FFT, split
        std::vector<float2> A(M), B(M), X(F);
        for (int n = 0; n < M; n++) A[n] = make_float2((float)x[2 * n], (float)x[2 * n + 1]);
        float2 *Z = run_passes<false>(M, A.data(), B.data(), tw.data(), &passes);
        for (int k = 0; k <= M / 2; k++) {
            float2 xk, xnk;
            rfft_split(Z[k], Z[(M - k) % M], tws[k], xk, xnk);
            X[k] = xk;
            if (2 * k != M) X[M - k] = xnk;
        }
        double ef = 0;
        for (int k = 0; k < F; k++) ef = fmax(ef, fmax(fabs(X[k].x - Xr[k]), fabs(X[k].y - Xi[k])));
        // inverse of the reference spectrum: merge, M-point inverse FFT; unnormalised, so the result is N x
        for (int k = 0; k <= M / 2; k++) {
            float2 xk = make_float2((float)Xr[k], (float)Xi[k]), xnk = make_float2((float)Xr[M - k], (float)Xi[M - k]);
            if (k == 0) { xk.y = 0.f; xnk.y = 0.f; }
            float2 zk, znk;
            irfft_merge(xk, xnk, make_float2(tws[k].x, -tws[k].y), zk, znk);
            A[k] = zk;
            if (k > 0 && 2 * k != M) A[M - k] = znk;
        }
        float2 *y = run_passes<true>(M, A.data(), B.data(), tw.data(), &passes);
        double ei = 0;
        for (int n = 0; n < M; n++)
            ei = fmax(ei, fmax(fabs(y[n].x - N * x[2 * n]), fabs(y[n].y - N * x[2 * n + 1])));
        double xs = 0;
        for (int n = 0; n < N; n++) xs = fmax(xs, fabs(N * x[n]));
        const double rf = ef / xmax, ri = ei / xs;
        printf("N=%d passes=%d fwd_rel=%.3e inv_rel=%.3e\n", N, passes, rf, ri);
        if (!(rf <= 1e-5 && ri <= 1e-5)) bad = 1;
    }
    return bad;
}
