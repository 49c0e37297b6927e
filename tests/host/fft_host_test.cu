// Host-side emulation of the warp FFT in deepfilternet_b200/csrc/dfb_fft.cuh: runs the 32 lanes
// sequentially on the CPU and checks against a double-precision DFT.  Built and run by
// tests/test_host_logic.py (no GPU needed).
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "../../deepfilternet_b200/csrc/dfb_fft.cuh"
using namespace dfb;

template <int N, bool INV>
double test_dft() {
    float2 v[N];
    std::vector<double> xr(N), xi(N);
    for (int i = 0; i < N; i++) {
        xr[i] = rand() / (double)RAND_MAX - 0.5; xi[i] = rand() / (double)RAND_MAX - 0.5;
        v[i] = make_float2((float)xr[i], (float)xi[i]);
        xr[i] = v[i].x; xi[i] = v[i].y;
    }
    Dft<N, INV>::run(v);
    double err = 0;
    for (int k = 0; k < N; k++) {
        double ar = 0, ai = 0;
        for (int n = 0; n < N; n++) {
            double ang = (INV ? 2.0 : -2.0) * M_PI * (double)((long)k * n % N) / N;
            ar += xr[n] * cos(ang) - xi[n] * sin(ang);
            ai += xr[n] * sin(ang) + xi[n] * cos(ang);
        }
        err = fmax(err, fmax(fabs(ar - v[k].x), fabs(ai - v[k].y)));
    }
    return err;
}

template <bool INV>
double test_fft480() {
    std::vector<float2> z(480), tile(kTileFloat2), out(480);
    for (auto& c : z) c = make_float2(rand() / (float)RAND_MAX - 0.5f, rand() / (float)RAND_MAX - 0.5f);
    // pass A
    for (int lane = 0; lane < kN2; lane++) {
        float2 a[kN1], tw[kN1];
        for (int n1 = 0; n1 < kN1; n1++) a[n1] = z[24 * n1 + lane];
        for (int k1 = 0; k1 < kN1; k1++) {
            double ang = (INV ? 2.0 : -2.0) * M_PI * (double)(lane * k1) / 480.0;
            tw[k1] = make_float2((float)cos(ang), (float)sin(ang));
        }
        fft480_pass_a<INV>(a, tw, tile.data(), lane);
    }
    // pass B (reads complete before writes: separate loops emulate the warp sync)
    std::vector<std::vector<float2>> regs(kN1, std::vector<float2>(kN2));
    for (int lane = 0; lane < kN1; lane++) {
        float2 b[kN2];
        fft480_pass_b<INV>(b, tile.data(), lane);
        for (int i = 0; i < kN2; i++) regs[lane][i] = b[i];
    }
    for (int lane = 0; lane < kN1; lane++) {
        float2 b[kN2];
        for (int i = 0; i < kN2; i++) b[i] = regs[lane][i];
        fft480_store_natural(b, out.data(), lane);
    }
    double err = 0;
    for (int k = 0; k < 480; k++) {
        double ar = 0, ai = 0;
        for (int n = 0; n < 480; n++) {
            double ang = (INV ? 2.0 : -2.0) * M_PI * (double)((long)k * n % 480) / 480.0;
            ar += z[n].x * cos(ang) - z[n].y * sin(ang);
            ai += z[n].x * sin(ang) + z[n].y * cos(ang);
        }
        err = fmax(err, fmax(fabs(ar - out[k].x), fabs(ai - out[k].y)));
    }
    return err;
}

// full real forward + inverse through split/merge
double test_real_roundtrip(double* fwd_err) {
    const int N = 960;
    std::vector<double> x(N);
    for (auto& v : x) v = rand() / (double)RAND_MAX - 0.5;
    std::vector<float2> z(480), Z(480), X(481);
    for (int n = 0; n < 480; n++) z[n] = make_float2((float)x[2 * n], (float)x[2 * n + 1]);
    for (int n = 0; n < N; n++) x[n] = (n % 2 == 0) ? z[n / 2].x : z[n / 2].y;
    // reference complex DFT in double for Z (the warp passes are tested above)
    for (int k = 0; k < 480; k++) {
        double ar = 0, ai = 0;
        for (int n = 0; n < 480; n++) {
            double ang = -2.0 * M_PI * (double)((long)k * n % 480) / 480.0;
            ar += z[n].x * cos(ang) - z[n].y * sin(ang);
            ai += z[n].x * sin(ang) + z[n].y * cos(ang);
        }
        Z[k] = make_float2((float)ar, (float)ai);
    }
    for (int k = 0; k <= 240; k++) {
        float2 w = make_float2((float)cos(-2 * M_PI * k / 960.0), (float)sin(-2 * M_PI * k / 960.0));
        float2 xk, xnk;
        rfft_split(Z[k], Z[(480 - k) % 480], w, xk, xnk);
        X[k] = xk; X[480 - k] = xnk;
    }
    double e = 0;
    for (int k = 0; k <= 480; k++) {
        double ar = 0, ai = 0;
        for (int n = 0; n < N; n++) {
            double ang = -2.0 * M_PI * (double)((long)k * n % N) / N;
            ar += x[n] * cos(ang); ai += x[n] * sin(ang);
        }
        e = fmax(e, fmax(fabs(ar - X[k].x), fabs(ai - X[k].y)));
    }
    *fwd_err = e;
    // inverse: merge + IDFT480 (double) -> x * N
    std::vector<float2> Zi(480);
    X[0].y = 0; X[480].y = 0;
    for (int k = 0; k <= 240; k++) {
        float2 wc = make_float2((float)cos(2 * M_PI * k / 960.0), (float)sin(2 * M_PI * k / 960.0));
        float2 zk, znk;
        irfft_merge(X[k], X[480 - k], wc, zk, znk);
        Zi[k] = zk;
        if (k > 0) Zi[480 - k] = znk;
    }
    double e2 = 0;
    for (int n = 0; n < 480; n++) {
        double ar = 0, ai = 0;
        for (int k = 0; k < 480; k++) {
            double ang = 2.0 * M_PI * (double)((long)k * n % 480) / 480.0;
            ar += Zi[k].x * cos(ang) - Zi[k].y * sin(ang);
            ai += Zi[k].x * sin(ang) + Zi[k].y * cos(ang);
        }
        e2 = fmax(e2, fmax(fabs(ar / N - x[2 * n]), fabs(ai / N - x[2 * n + 1])));
    }
    return e2;
}

int main() {
    srand(7);
    int bad = 0;
#define T(N) { double a = test_dft<N,false>(), b = test_dft<N,true>(); printf("dft%-3d fwd %.3e inv %.3e\n", N, a, b); if (a > 2e-6*N || b > 2e-6*N) bad++; }
    T(2) T(3) T(4) T(5) T(6) T(8) T(10) T(12) T(15) T(16) T(20) T(24) T(30) T(32)
    double f = test_fft480<false>(), i = test_fft480<true>();
    printf("fft480 fwd %.3e inv %.3e\n", f, i);
    if (f > 2e-5 || i > 2e-5) bad++;
    double fe, re = test_real_roundtrip(&fe);
    printf("rfft split err %.3e  irfft roundtrip err %.3e\n", fe, re);
    if (fe > 5e-5 || re > 1e-6) bad++;
    printf(bad ? "FAIL\n" : "OK\n");
    return bad;
}
