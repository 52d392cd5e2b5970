// Device-side building blocks shared by the compositing kernels.
//
// Coordinate recipe (bit-exact with OpenCV's WarpPerspectiveInvoker, SURVEY.md section 8 a1):
//   (xl, yl) = pixel in the layer's own canvas frame;  xb = xl & ~63, x1 = xl & 63
//   X0 = (Mi0*xb + Mi1*yl) + Mi2  (likewise Y0, W0)          -- float64, round-to-nearest, NO fma
//   W  = W0 + Mi6*x1 ; W = W ? 32/W : 0
//   X  = rint(clamp((X0 + Mi0*x1) * W))   Y likewise          -- 1/32-px fixed point
// The float64 operations use the __d*_rn intrinsics, which the compiler never contracts.
#pragma once

#include "mcs_common.h"

struct RowBlock {  // X0, Y0, W0 of one (layer, row, 64-column block)
    double X0, Y0, W0;
};

__device__ __forceinline__ RowBlock row_block(const double* __restrict__ mi, int xb, int yl) {
    const double xbd = (double)xb, yd = (double)yl;
    RowBlock r;
    r.X0 = __dadd_rn(__dadd_rn(__dmul_rn(mi[0], xbd), __dmul_rn(mi[1], yd)), mi[2]);
    r.Y0 = __dadd_rn(__dadd_rn(__dmul_rn(mi[3], xbd), __dmul_rn(mi[4], yd)), mi[5]);
    r.W0 = __dadd_rn(__dadd_rn(__dmul_rn(mi[6], xbd), __dmul_rn(mi[7], yd)), mi[8]);
    return r;
}

// 1/32-px source coordinates of column x1 (0..63) of a row block; m0/m3/m6 = Mi[0], Mi[3], Mi[6].
__device__ __forceinline__ void fixed_coords(double m0, double m3, double m6, const RowBlock& rb,
                                             int x1, int& X, int& Y) {
    const double x1d = (double)x1;
    double W = __dadd_rn(rb.W0, __dmul_rn(m6, x1d));
    const bool wz = (W == 0.0);
    W = __ddiv_rn(32.0, W);
    const double fX = __dmul_rn(__dadd_rn(rb.X0, __dmul_rn(m0, x1d)), W);
    const double fY = __dmul_rn(__dadd_rn(rb.Y0, __dmul_rn(m3, x1d)), W);
    // cvt.rni.s32.f64 saturates to [INT_MIN, INT_MAX] exactly like the reference's clamp + cvRound
    X = wz ? 0 : __double2int_rn(fX);
    Y = wz ? 0 : __double2int_rn(fY);
}

// saturate_cast<short> of the integer part of a 1/32-px coordinate
__device__ __forceinline__ int sat16(int v) { return max(-32768, min(32767, v)); }

// Fixed-point bilinear sample of one uint8 weight map (w x h, no pitch) at (X, Y), 1/32 px; taps outside the map read 0,
// a missing map reads 255 inside.
__device__ __forceinline__ int weight_sample(const uint8_t* __restrict__ m, int w, int h, int X, int Y) {
    const int sx = sat16(X >> 5), sy = sat16(Y >> 5), ax = X & 31, ay = Y & 31;
    const bool x0in = (unsigned)sx < (unsigned)w, x1in = (unsigned)(sx + 1) < (unsigned)w;
    const bool y0in = (unsigned)sy < (unsigned)h, y1in = (unsigned)(sy + 1) < (unsigned)h;
    const uint8_t* r0 = m + (long long)sy * w + sx;
    int p00 = 0, p01 = 0, p10 = 0, p11 = 0;
    if (y0in && x0in) p00 = m ? __ldg(r0) : 255;
    if (y0in && x1in) p01 = m ? __ldg(r0 + 1) : 255;
    if (y1in && x0in) p10 = m ? __ldg(r0 + w) : 255;
    if (y1in && x1in) p11 = m ? __ldg(r0 + w + 1) : 255;
    return ((32 - ay) * (32 - ax) * 32 * p00 + (32 - ay) * ax * 32 * p01 + ay * (32 - ax) * 32 * p10 +
            ay * ax * 32 * p11 + 16384) >> 15;
}

// Some of the four bilinear taps at 1/32-px (X, Y) lies inside the layer's source (otherwise the
// sample is BORDER_CONSTANT 0 and the layer does not touch the pixel).
__device__ __forceinline__ bool some_tap_inside(const McsLayer& g, int X, int Y) {
    const int sx = sat16(X >> 5), sy = sat16(Y >> 5);
    return ((unsigned)sx < (unsigned)g.src_w || (unsigned)(sx + 1) < (unsigned)g.src_w) &&
           ((unsigned)sy < (unsigned)g.src_h || (unsigned)(sy + 1) < (unsigned)g.src_h);
}

// 1/32-px source coordinates of pixel (xl, yl) of a layer's own canvas frame: the homography
// recipe above for WARP layers, the plan's fixed-point map (cv2.remap with CV_16SC2 + CV_16UC1
// maps: X = 32 * map_x + fx, Y = 32 * map_y + fy) for REMAP layers.
__device__ __forceinline__ void layer_coords(const McsLayer& L, int xl, int yl, int& X, int& Y) {
    if (L.kind == MCS_LAYER_REMAP) {
        if ((unsigned)xl < (unsigned)L.map_w && (unsigned)yl < (unsigned)L.map_h) {
            const int2 m = __ldg(L.map + (size_t)yl * L.map_w + xl);
            X = m.x;
            Y = m.y;
        } else {
            X = Y = -64 * 32;   // outside the map: no tap inside any source
        }
        return;
    }
    const RowBlock rb = row_block(L.mi, xl & ~63, yl);
    fixed_coords(L.mi[0], L.mi[3], L.mi[6], rb, xl & 63, X, Y);
}
