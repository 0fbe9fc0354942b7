// sampler.cuh -- OpenCV-exact coordinate quantisation and uint8 / uint16 gather (device side).
//
// Replaces the inside of cv::remap as called at /root/reference/src/vr180_convert/remapper.py:388-398.
// OpenCV is a third-party dependency of the reference (opencv-python 4.10.0.82 pinned, poetry.lock:1014-1015);
// the arithmetic reproduced here is its published fixed-point scheme (imgproc/imgwarp.cpp, INTER_BITS = 5,
// INTER_REMAP_COEF_BITS = 15), restated and verified bit-exact against the installed cv2 in oracle/remap_np.py.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/vr180_b200.h"

namespace vr180 {

constexpr int kInterBits = 5;
constexpr int kInterTab = 32;

// cvRound(v) on x86 (cvtps2dq): round-half-even; NaN, +-inf and |v| >= 2^31 give INT_MIN.
__device__ __forceinline__ int cv_round(float v) {
    return (fabsf(v) < 2147483648.0f) ? __float2int_rn(v) : (int)0x80000000;
}
// sx = cvRound(map * 32) -- float32 multiply first, exactly like the reference's float32 maps going through cv::remap
__device__ __forceinline__ int quantise(float m) { return cv_round(__fmul_rn(m, 32.0f)); }
__device__ __forceinline__ int sat16(int v) { return max(-32768, min(32767, v)); }

struct Src {
    const uint8_t* __restrict__ p;  // frame base
    int rows, cols;
    long long pitch;
};

// cv::borderInterpolate for REPLICATE / REFLECT / WRAP / REFLECT_101 (any integer p; n >= 1)
__device__ __forceinline__ int border_index(int p, int n, int mode) {
    if ((unsigned)p < (unsigned)n) return p;
    if (mode == VR180_BORDER_REPLICATE) return p < 0 ? 0 : n - 1;
    if (mode == VR180_BORDER_WRAP) {
        int q = p % n;
        return q < 0 ? q + n : q;
    }
    if (n == 1) return 0;
    const int delta = (mode == VR180_BORDER_REFLECT_101) ? 1 : 0;
    const int period = 2 * n - 2 * delta;
    int q = p % period;
    if (q < 0) q += period;
    return q < n ? q : period - 1 + delta - q;
}

template <int C>
struct Px {
    int v[C];
};

// One tap with border handling.  `constant` border: outside taps contribute border_value (OpenCV blends partially
// outside footprints with the border colour); other modes remap the index.
template <int C>
__device__ __forceinline__ void fetch_tap(const Src& s, int x, int y, int border_mode, const uint8_t* bv, int* out) {
    if (border_mode == VR180_BORDER_CONSTANT) {
        if ((unsigned)x < (unsigned)s.cols && (unsigned)y < (unsigned)s.rows) {
            const uint8_t* q = s.p + (long long)y * s.pitch + (long long)x * C;
#pragma unroll
            for (int c = 0; c < C; ++c) out[c] = __ldg(q + c);
        } else {
#pragma unroll
            for (int c = 0; c < C; ++c) out[c] = bv[c];
        }
    } else {
        const int xx = border_index(x, s.cols, border_mode);
        const int yy = border_index(y, s.rows, border_mode);
        const uint8_t* q = s.p + (long long)yy * s.pitch + (long long)xx * C;
#pragma unroll
        for (int c = 0; c < C; ++c) out[c] = __ldg(q + c);
    }
}

// INTER_NEAREST: ix = saturate_int16(cvRound(x)), out = src[iy, ix] or border.
template <int C>
__device__ __forceinline__ void sample_nearest(const Src& s, float mx, float my, int border_mode, const uint8_t* bv,
                                               int* out) {
    const int ix = sat16(cv_round(mx));
    const int iy = sat16(cv_round(my));
    fetch_tap<C>(s, ix, iy, border_mode, bv, out);
}

// INTER_LINEAR on fixed-point coordinates: weights (32-ax)(32-ay) .. ax*ay (sum 1024), (acc + 512) >> 10.
// Identical to OpenCV's 15-bit table form for uint8 (oracle/remap_np.py, SURVEY.md B.2).
template <int C>
__device__ __forceinline__ void sample_linear(const Src& s, int sx, int sy, int border_mode, const uint8_t* bv, int* out) {
    const int ix = sat16(sx >> kInterBits), iy = sat16(sy >> kInterBits);
    const int ax = sx & 31, ay = sy & 31;
    const int w00 = (32 - ax) * (32 - ay), w01 = ax * (32 - ay), w10 = (32 - ax) * ay, w11 = ax * ay;
    if ((unsigned)ix < (unsigned)(s.cols - 1) && (unsigned)iy < (unsigned)(s.rows - 1)) {
        const uint8_t* q0 = s.p + (long long)iy * s.pitch + (long long)ix * C;
        const uint8_t* q1 = q0 + s.pitch;
#pragma unroll
        for (int c = 0; c < C; ++c) {
            const int acc = w00 * __ldg(q0 + c) + w01 * __ldg(q0 + C + c) + w10 * __ldg(q1 + c) + w11 * __ldg(q1 + C + c);
            out[c] = (acc + 512) >> 10;
        }
        return;
    }
    if (border_mode == VR180_BORDER_CONSTANT &&
        (ix >= s.cols || ix + 1 < 0 || iy >= s.rows || iy + 1 < 0)) {
#pragma unroll
        for (int c = 0; c < C; ++c) out[c] = bv[c];
        return;
    }
    int t00[C], t01[C], t10[C], t11[C];
    fetch_tap<C>(s, ix, iy, border_mode, bv, t00);
    fetch_tap<C>(s, ix + 1, iy, border_mode, bv, t01);
    fetch_tap<C>(s, ix, iy + 1, border_mode, bv, t10);
    fetch_tap<C>(s, ix + 1, iy + 1, border_mode, bv, t11);
#pragma unroll
    for (int c = 0; c < C; ++c) out[c] = (w00 * t00[c] + w01 * t01[c] + w10 * t10[c] + w11 * t11[c] + 512) >> 10;
}

// s16 x u8 two-way dot products (weights are OpenCV's signed int16 table entries, pixels unsigned bytes)
__device__ __forceinline__ int dp2a_lo_s16u8(uint32_t w, uint32_t px, int acc) {  // w.lo * px.b0 + w.hi * px.b1
    int d;
    asm("dp2a.lo.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(w), "r"(px), "r"(acc));
    return d;
}
__device__ __forceinline__ int dp2a_hi_s16u8(uint32_t w, uint32_t px, int acc) {  // w.lo * px.b2 + w.hi * px.b3
    int d;
    asm("dp2a.hi.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(w), "r"(px), "r"(acc));
    return d;
}

// Interior K x K footprint of a 3-channel image whose rows are word-aligned: every tap row is K * 3 contiguous
// bytes, fetched as aligned 32-bit words (K * 3 / 4 + 1 loads instead of K * 3 byte loads), byte-aligned with funnel
// shifts, regrouped per channel with PRMT and accumulated with dp2a against the row's int16 weights (one 8- or
// 16-byte load instead of K 2-byte loads).  The caller guarantees 3 readable bytes past the last tap of a row.
template <int K>
__device__ __forceinline__ void sample_tab3_words(const uint8_t* __restrict__ q, long long pitch,
                                                  const short* __restrict__ w, int* out) {
    constexpr int NW = K * 3 / 4;  // payload words per tap row: 3 (cubic) or 6 (Lanczos4)
    const int sh = (int)((uintptr_t)q & 3) * 8;
    const uint8_t* r = q - ((uintptr_t)q & 3);
    int acc0 = 16384, acc1 = 16384, acc2 = 16384;  // + 1 << 14 before the >> 15
#pragma unroll
    for (int ky = 0; ky < K; ++ky, r += pitch) {
        const uint32_t* rw = reinterpret_cast<const uint32_t*>(r);
        uint32_t x[NW + 1], A[NW], wv[K / 2];
#pragma unroll
        for (int i = 0; i <= NW; ++i) x[i] = __ldg(rw + i);
#pragma unroll
        for (int i = 0; i < NW; ++i) A[i] = __funnelshift_r(x[i], x[i + 1], sh);
        if (K == 4) {
            const uint2 t = __ldg(reinterpret_cast<const uint2*>(w + ky * K));
            wv[0] = t.x; wv[1] = t.y;
        } else {
            const uint4 t = __ldg(reinterpret_cast<const uint4*>(w + ky * K));
            wv[0] = t.x; wv[1] = t.y; wv[K / 2 - 2] = t.z; wv[K / 2 - 1] = t.w;
        }
#pragma unroll
        for (int g = 0; g < K / 4; ++g) {  // taps 4 g .. 4 g + 3 = bytes of A[3 g .. 3 g + 2]
            const uint32_t A0 = A[3 * g], A1 = A[3 * g + 1], A2 = A[3 * g + 2];
            const uint32_t q0 = __byte_perm(__byte_perm(A0, A1, 0x0630), A2, 0x5210);  // [t0c0 t1c0 t2c0 t3c0]
            const uint32_t q1 = __byte_perm(__byte_perm(A0, A1, 0x0741), A2, 0x6210);  // [t0c1 t1c1 t2c1 t3c1]
            const uint32_t q2 = __byte_perm(__byte_perm(A0, A1, 0x0052), A2, 0x7410);  // [t0c2 t1c2 t2c2 t3c2]
            const uint32_t w01 = wv[2 * g], w23 = wv[2 * g + 1];
            acc0 = dp2a_hi_s16u8(w23, q0, dp2a_lo_s16u8(w01, q0, acc0));
            acc1 = dp2a_hi_s16u8(w23, q1, dp2a_lo_s16u8(w01, q1, acc1));
            acc2 = dp2a_hi_s16u8(w23, q2, dp2a_lo_s16u8(w01, q2, acc2));
        }
    }
    out[0] = max(0, min(255, acc0 >> 15));
    out[1] = max(0, min(255, acc1 >> 15));
    out[2] = max(0, min(255, acc2 >> 15));
}

// INTER_CUBIC (K = 4) / INTER_LANCZOS4 (K = 8): K x K taps from ix-(K/2-1), int16 weights itab[ay*32+ax][ky][kx]
// summing to 32768, out = clip((acc + 16384) >> 15).
template <int C, int K>
__device__ __forceinline__ void sample_tab(const Src& s, int sx, int sy, const short* __restrict__ tab, int border_mode,
                                           const uint8_t* bv, int* out) {
    const int ix = sat16(sx >> kInterBits) - (K / 2 - 1), iy = sat16(sy >> kInterBits) - (K / 2 - 1);
    const short* w = tab + (size_t)(((sy & 31) << 5) | (sx & 31)) * (K * K);
    int acc[C];
#pragma unroll
    for (int c = 0; c < C; ++c) acc[c] = 0;
    if (C == 3 && (unsigned)ix < (unsigned)max(s.cols - (K + 1), 0) && (unsigned)iy < (unsigned)max(s.rows - (K - 1), 0) &&
        (((uintptr_t)s.p | (uintptr_t)s.pitch) & 3) == 0) {  // word path: needs 3 spare bytes after the last tap of a row
        sample_tab3_words<K>(s.p + (long long)iy * s.pitch + (long long)ix * 3, s.pitch, w, out);
        return;
    }
    if ((unsigned)ix < (unsigned)max(s.cols - (K - 1), 0) && (unsigned)iy < (unsigned)max(s.rows - (K - 1), 0)) {
        const uint8_t* q = s.p + (long long)iy * s.pitch + (long long)ix * C;
#pragma unroll
        for (int ky = 0; ky < K; ++ky, q += s.pitch) {
#pragma unroll
            for (int kx = 0; kx < K; ++kx) {
                const int wv = w[ky * K + kx];
#pragma unroll
                for (int c = 0; c < C; ++c) acc[c] += wv * __ldg(q + kx * C + c);
            }
        }
    } else if (border_mode == VR180_BORDER_CONSTANT &&
               (ix >= s.cols || ix + K <= 0 || iy >= s.rows || iy + K <= 0)) {
#pragma unroll
        for (int c = 0; c < C; ++c) out[c] = bv[c];
        return;
    } else {
        for (int ky = 0; ky < K; ++ky) {
            for (int kx = 0; kx < K; ++kx) {
                int t[C];
                fetch_tap<C>(s, ix + kx, iy + ky, border_mode, bv, t);
                const int wv = w[ky * K + kx];
#pragma unroll
                for (int c = 0; c < C; ++c) acc[c] += wv * t[c];
            }
        }
    }
#pragma unroll
    for (int c = 0; c < C; ++c) out[c] = max(0, min(255, (acc[c] + 16384) >> 15));
}

// ---------------------------------------------------------------------------------------------------------
// 16-bit images: cv::remap's float-weight arithmetic for non-8-bit depths (remapBilinear / remapBicubic /
// remapLanczos4, restated in oracle/remap_float_np.py).  Src.p / pitch stay in bytes; elements are uint16.  Every
// product and sum is one float32 operation (__fmul_rn / __fadd_rn: no contraction into FMA), in OpenCV's order, and
// the result is saturate(cvRound(s)).  `cval` is the border colour as float (a uint16 converts exactly).
// ---------------------------------------------------------------------------------------------------------
template <int C>
__device__ __forceinline__ const uint16_t* px16(const Src& s, int x, int y) {
    return reinterpret_cast<const uint16_t*>(s.p + (long long)y * s.pitch) + (long long)x * C;
}
__device__ __forceinline__ int sat_u16(float v) { return max(0, min(65535, __float2int_rn(v))); }

template <int C>
__device__ __forceinline__ void sample16_nearest(const Src& s, float mx, float my, int border_mode, const float* cval,
                                                 int* out) {
    const int ix = sat16(cv_round(mx)), iy = sat16(cv_round(my));
    if (border_mode == VR180_BORDER_CONSTANT && !((unsigned)ix < (unsigned)s.cols && (unsigned)iy < (unsigned)s.rows)) {
#pragma unroll
        for (int c = 0; c < C; ++c) out[c] = (int)cval[c];
        return;
    }
    const uint16_t* q = px16<C>(s, border_index(ix, s.cols, border_mode), border_index(iy, s.rows, border_mode));
#pragma unroll
    for (int c = 0; c < C; ++c) out[c] = __ldg(q + c);
}

// INTER_NEAREST on the integer coordinate (ix, iy) = (sat16(cvRound(x)), sat16(cvRound(y))): the pixel or the border.
template <int C>
__device__ __forceinline__ void nearest16(const Src& s, int ix, int iy, int border_mode, const float* cval, int* out) {
    if (border_mode == VR180_BORDER_CONSTANT && !((unsigned)ix < (unsigned)s.cols && (unsigned)iy < (unsigned)s.rows)) {
#pragma unroll
        for (int c = 0; c < C; ++c) out[c] = (int)cval[c];
        return;
    }
    const uint16_t* q = px16<C>(s, border_index(ix, s.cols, border_mode), border_index(iy, s.rows, border_mode));
#pragma unroll
    for (int c = 0; c < C; ++c) out[c] = __ldg(q + c);
}

// One bilinear tap as float: the pixel, or under BORDER_CONSTANT the border colour outside the source.
template <int C>
__device__ __forceinline__ void tap16(const Src& s, int x, int y, int border_mode, const float* cval, float* v) {
    if (border_mode == VR180_BORDER_CONSTANT && !((unsigned)x < (unsigned)s.cols && (unsigned)y < (unsigned)s.rows)) {
#pragma unroll
        for (int c = 0; c < C; ++c) v[c] = cval[c];
        return;
    }
    const uint16_t* q = px16<C>(s, border_index(x, s.cols, border_mode), border_index(y, s.rows, border_mode));
#pragma unroll
    for (int c = 0; c < C; ++c) v[c] = (float)__ldg(q + c);
}

// INTER_LINEAR: w = float((1 - ty or ty) * (1 - tx or tx)) = (32-ay or ay)(32-ax or ax) / 1024 exactly;
// s = ((v00 w00 + v01 w01) + v10 w10) + v11 w11.  A footprint entirely outside under BORDER_CONSTANT is cval itself.
template <int C>
__device__ __forceinline__ void sample16_linear(const Src& s, int sx, int sy, int border_mode, const float* cval,
                                                int* out) {
    const int ix = sat16(sx >> kInterBits), iy = sat16(sy >> kInterBits);
    const int ax = sx & 31, ay = sy & 31;
    const float w00 = (float)((32 - ax) * (32 - ay)) * (1.0f / 1024.0f), w01 = (float)(ax * (32 - ay)) * (1.0f / 1024.0f);
    const float w10 = (float)((32 - ax) * ay) * (1.0f / 1024.0f), w11 = (float)(ax * ay) * (1.0f / 1024.0f);
    if (border_mode == VR180_BORDER_CONSTANT && (ix >= s.cols || ix + 1 < 0 || iy >= s.rows || iy + 1 < 0)) {
#pragma unroll
        for (int c = 0; c < C; ++c) out[c] = (int)cval[c];
        return;
    }
    float v00[C], v01[C], v10[C], v11[C];
    if ((unsigned)ix < (unsigned)(s.cols - 1) && (unsigned)iy < (unsigned)(s.rows - 1)) {
        const uint16_t* q0 = px16<C>(s, ix, iy);
        const uint16_t* q1 = reinterpret_cast<const uint16_t*>(reinterpret_cast<const uint8_t*>(q0) + s.pitch);
#pragma unroll
        for (int c = 0; c < C; ++c) {
            v00[c] = __ldg(q0 + c);
            v01[c] = __ldg(q0 + C + c);
            v10[c] = __ldg(q1 + c);
            v11[c] = __ldg(q1 + C + c);
        }
    } else {
        tap16<C>(s, ix, iy, border_mode, cval, v00);
        tap16<C>(s, ix + 1, iy, border_mode, cval, v01);
        tap16<C>(s, ix, iy + 1, border_mode, cval, v10);
        tap16<C>(s, ix + 1, iy + 1, border_mode, cval, v11);
    }
#pragma unroll
    for (int c = 0; c < C; ++c) {
        float acc = __fadd_rn(__fmul_rn(v00[c], w00), __fmul_rn(v01[c], w01));
        acc = __fadd_rn(acc, __fmul_rn(v10[c], w10));
        acc = __fadd_rn(acc, __fmul_rn(v11[c], w11));
        out[c] = sat_u16(acc);
    }
}

// INTER_CUBIC (K = 4) / INTER_LANCZOS4 (K = 8) with the float table ftab[ay*32+ax][ky][kx].
//   interior (every tap inside): each row summed left to right, then the rows left to right;
//   elsewhere, in EVERY border mode: s = cval, then s += (S - cval) * w for each valid tap in row-major order (under
//   BORDER_CONSTANT a tap outside the source is not valid; other modes remap its index) -- so the border colour
//   reaches results under REPLICATE / REFLECT / WRAP / REFLECT_101 too, as in OpenCV.
template <int C, int K>
__device__ __forceinline__ void sample16_tab(const Src& s, int sx, int sy, const float* __restrict__ ftab, int border_mode,
                                             const float* cval, int* out) {
    const int ix = sat16(sx >> kInterBits) - (K / 2 - 1), iy = sat16(sy >> kInterBits) - (K / 2 - 1);
    const float* w = ftab + (size_t)(((sy & 31) << 5) | (sx & 31)) * (K * K);
    float acc[C];
    if ((unsigned)ix < (unsigned)max(s.cols - (K - 1), 0) && (unsigned)iy < (unsigned)max(s.rows - (K - 1), 0)) {
        const uint16_t* q = px16<C>(s, ix, iy);
#pragma unroll
        for (int ky = 0; ky < K; ++ky) {
            float r[C];
#pragma unroll
            for (int kx = 0; kx < K; ++kx) {
                const float wv = __ldg(w + ky * K + kx);
#pragma unroll
                for (int c = 0; c < C; ++c) {
                    const float p = __fmul_rn((float)__ldg(q + kx * C + c), wv);
                    r[c] = kx ? __fadd_rn(r[c], p) : p;
                }
            }
#pragma unroll
            for (int c = 0; c < C; ++c) acc[c] = ky ? __fadd_rn(acc[c], r[c]) : r[c];
            q = reinterpret_cast<const uint16_t*>(reinterpret_cast<const uint8_t*>(q) + s.pitch);
        }
    } else {
#pragma unroll
        for (int c = 0; c < C; ++c) acc[c] = cval[c];
        for (int ky = 0; ky < K; ++ky) {
            const int y = iy + ky;
            if (border_mode == VR180_BORDER_CONSTANT && (unsigned)y >= (unsigned)s.rows) continue;
            const int yy = border_index(y, s.rows, border_mode);
            for (int kx = 0; kx < K; ++kx) {
                const int x = ix + kx;
                if (border_mode == VR180_BORDER_CONSTANT && (unsigned)x >= (unsigned)s.cols) continue;
                const uint16_t* q = px16<C>(s, border_index(x, s.cols, border_mode), yy);
                const float wv = __ldg(w + ky * K + kx);
#pragma unroll
                for (int c = 0; c < C; ++c)
                    acc[c] = __fadd_rn(acc[c], __fmul_rn(__fsub_rn((float)__ldg(q + c), cval[c]), wv));
            }
        }
    }
#pragma unroll
    for (int c = 0; c < C; ++c) out[c] = sat_u16(acc[c]);
}

}  // namespace vr180
