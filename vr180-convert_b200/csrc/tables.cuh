// tables.cuh -- host construction of OpenCV's INTER_CUBIC / INTER_LANCZOS4 weight tables (cv::initInterTab2D in
// imgproc/imgwarp.cpp; third-party to the reference, restated in oracle/remap_np.py, oracle/remap_float_np.py and
// SURVEY.md Appendix B.3).  8-bit images: int16 [ay*32+ax][ky][kx], every K*K block sums to exactly 32768.  16-bit
// images: the float products before that conversion.
#pragma once
#include <cfloat>
#include <cmath>
#include <cstdint>
#include <vector>

namespace vr180 {

// All arithmetic below is float32 with one rounding per operation, as the C++ original compiled for SSE2.
// `volatile` stores keep the host compiler from contracting or widening.
inline void coef_cubic(float t, float* c) {
    const float A = -0.75f;
    volatile float a0 = t + 1.0f;
    volatile float p0 = A * a0;
    p0 = p0 - 5.0f * A;
    p0 = p0 * a0;
    p0 = p0 + 8.0f * A;
    p0 = p0 * a0;
    p0 = p0 - 4.0f * A;
    c[0] = p0;
    volatile float p1 = (A + 2.0f) * t;
    p1 = p1 - (A + 3.0f);
    p1 = p1 * t;
    p1 = p1 * t;
    p1 = p1 + 1.0f;
    c[1] = p1;
    volatile float u = 1.0f - t;
    volatile float p2 = (A + 2.0f) * u;
    p2 = p2 - (A + 3.0f);
    p2 = p2 * u;
    p2 = p2 * u;
    p2 = p2 + 1.0f;
    c[2] = p2;
    volatile float p3 = 1.0f - c[0];
    p3 = p3 - c[1];
    p3 = p3 - c[2];
    c[3] = p3;
}

inline void coef_lanczos4(float t, float* c) {
    if (t < FLT_EPSILON) {
        for (int i = 0; i < 8; ++i) c[i] = 0.0f;
        c[3] = 1.0f;
        return;
    }
    static const double s45 = 0.70710678118654752440084436210485;
    static const double cs[8][2] = {{1, 0}, {-s45, -s45}, {0, 1}, {s45, -s45}, {-1, 0}, {s45, s45}, {0, -1}, {-s45, s45}};
    const double x = (double)t;
    const double y0 = -(x + 3) * M_PI * 0.25, s0 = std::sin(y0), c0 = std::cos(y0);
    volatile float sum = 0.0f;
    for (int i = 0; i < 8; ++i) {
        const double y = -(x + 3 - i) * M_PI * 0.25;
        c[i] = (float)((cs[i][0] * s0 + cs[i][1] * c0) / (y * y));
        sum = sum + c[i];
    }
    volatile float inv = 1.0f / sum;
    for (int i = 0; i < 8; ++i) {
        volatile float v = c[i] * inv;
        c[i] = v;
    }
}

// 1-D coefficients of the 32 fractional positions t = i * (1/32) (cv::initInterTab1D)
inline void one_d_table(int K, float one[32][8]) {
    for (int i = 0; i < 32; ++i) {
        volatile float t = (float)i * (1.0f / 32.0f);
        if (K == 4) coef_cubic(t, one[i]);
        else coef_lanczos4(t, one[i]);
    }
}

// The float table of the non-8-bit depths: w[ay*32+ax][ky][kx] = float(one[ay][ky] * one[ax][kx]), rounded once and
// without the sum fix-up of the int16 table (initInterTab2D with fixpt = false).
inline std::vector<float> build_float_table(int K) {
    std::vector<float> tab((size_t)1024 * K * K);
    float one[32][8];
    one_d_table(K, one);
    for (int ay = 0; ay < 32; ++ay)
        for (int ax = 0; ax < 32; ++ax)
            for (int ky = 0; ky < K; ++ky)
                for (int kx = 0; kx < K; ++kx) {
                    volatile float v = one[ay][ky] * one[ax][kx];
                    tab[((size_t)(ay * 32 + ax) * K + ky) * K + kx] = v;
                }
    return tab;
}

inline std::vector<int16_t> build_weight_table(int K) {
    std::vector<int16_t> tab((size_t)1024 * K * K);
    float one[32][8];
    one_d_table(K, one);
    const int k2 = K / 2;
    for (int ay = 0; ay < 32; ++ay)
        for (int ax = 0; ax < 32; ++ax) {
            int16_t* it = &tab[(size_t)(ay * 32 + ax) * K * K];
            int isum = 0;
            for (int ky = 0; ky < K; ++ky)
                for (int kx = 0; kx < K; ++kx) {
                    volatile float v = one[ay][ky] * one[ax][kx];
                    volatile float sc = v * 32768.0f;
                    long r = std::lrintf(sc);  // round-half-even under the default rounding mode
                    if (r > 32767) r = 32767;
                    if (r < -32768) r = -32768;
                    it[ky * K + kx] = (int16_t)r;
                    isum += (int)r;
                }
            const int diff = isum - 32768;
            if (diff != 0) {
                int mk1 = k2, mk2 = k2, Mk1 = k2, Mk2 = k2;
                for (int k1 = k2; k1 < k2 + 2; ++k1)
                    for (int kk = k2; kk < k2 + 2; ++kk) {
                        if (it[k1 * K + kk] < it[mk1 * K + mk2]) { mk1 = k1; mk2 = kk; }
                        else if (it[k1 * K + kk] > it[Mk1 * K + Mk2]) { Mk1 = k1; Mk2 = kk; }
                    }
                if (diff < 0) it[Mk1 * K + Mk2] = (int16_t)(it[Mk1 * K + Mk2] - diff);
                else it[mk1 * K + mk2] = (int16_t)(it[mk1 * K + mk2] - diff);
            }
        }
    return tab;
}

}  // namespace vr180
