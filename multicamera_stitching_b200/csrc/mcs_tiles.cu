// Plan-time tiling for the tiled compositing kernel.
//
// The panorama is cut into work items ("tiles"), each owned by exactly one layer: layer k owns
// rect_k minus rect_{k-1} (rectangles are nested, innermost first).  Tiles live on one 128 x 16
// cell grid anchored at panorama column 0 (a cell row is then a whole number of 32-byte sectors
// of a 32-byte aligned panorama row).  One-off kernels evaluate OpenCV's exact fixed-point
// coordinates of every pixel of every WARP tile: first the bounding box of the source pixels a
// tile touches - the host turns that into the TMA box origin of the tile and the per-layer box
// size - then one 32-bit sampling descriptor per pixel relative to that box.  The table is sorted
// by class and carries a per-frame cost estimate for the launch-time work split.
#include "mcs_device.cuh"

#include <algorithm>
#include <vector>
#include <limits.h>
#include <stdlib.h>
#include <string.h>

struct TileBounds {
    int min_sx, max_sx, min_sy, max_sy;
    int touched;
    int clamped;   // some tap coordinate had to be clamped (lies 2+ pixels outside the source)
    int pad[2];
};

// One warp per tile.  sx / sy are clamped to [-2, src_w] / [-2, src_h]: at the clamp values both
// taps of that axis are outside the source, so they read zero-filled box bytes, exactly what
// BORDER_CONSTANT(0) returns.
__global__ void __launch_bounds__(256)
mcs_tile_bounds_kernel(const McsTile* __restrict__ tiles, const McsLayer* __restrict__ layers, int n_tiles,
                       TileBounds* __restrict__ out) {
    const int t = blockIdx.x * 8 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (t >= n_tiles) return;
    const McsTile tile = tiles[t];
    int mnx = INT_MAX, mxx = INT_MIN, mny = INT_MAX, mxy = INT_MIN, touched = 0, clamped = 0;
    if (tile.layer >= 0 && tile.cls == MCS_TILE_WARP) {
        const McsLayer& L = layers[tile.layer];
        const int w = tile.c1 - tile.c0;
        const int n = w * tile.h;
        for (int i = lane; i < n; i += 32) {
            const int r = i / w, c = tile.c0 + (i - r * w);
            const int xl = tile.cx0 + c - L.ox, yl = tile.y0 + r - L.oy;
            int X, Y;
            layer_coords(L, xl, yl, X, Y);
            const int rsx = sat16(X >> 5), rsy = sat16(Y >> 5);
            const bool in = ((unsigned)rsx < (unsigned)L.src_w || (unsigned)(rsx + 1) < (unsigned)L.src_w) &&
                            ((unsigned)rsy < (unsigned)L.src_h || (unsigned)(rsy + 1) < (unsigned)L.src_h);
            touched |= in ? 1 : 0;
            const int sx = max(-2, min(L.src_w, rsx)), sy = max(-2, min(L.src_h, rsy));
            clamped |= (sx != (X >> 5) || sy != (Y >> 5)) ? 1 : 0;
            mnx = min(mnx, sx); mxx = max(mxx, sx);
            mny = min(mny, sy); mxy = max(mxy, sy);
        }
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        mnx = min(mnx, __shfl_xor_sync(0xffffffffu, mnx, off));
        mxx = max(mxx, __shfl_xor_sync(0xffffffffu, mxx, off));
        mny = min(mny, __shfl_xor_sync(0xffffffffu, mny, off));
        mxy = max(mxy, __shfl_xor_sync(0xffffffffu, mxy, off));
        touched |= __shfl_xor_sync(0xffffffffu, touched, off);
        clamped |= __shfl_xor_sync(0xffffffffu, clamped, off);
    }
    if (lane == 0) {
        TileBounds b;
        b.min_sx = mnx; b.max_sx = mxx; b.min_sy = mny; b.max_sy = mxy; b.touched = touched;
        b.clamped = clamped;
        b.pad[0] = b.pad[1] = 0;
        out[t] = b;
    }
}

// One CTA of 256 threads per WARP tile: the frame-invariant sampling descriptor of each of its
// 128 x 16 pixel slots, in the order the tiled kernel's threads read them ([j][warp][lane] with
// row = warp + 8 * (j >> 2), column = lane + 32 * (j & 3)):
//   bits 0..15   byte offset of tap (sx, sy) inside the tile's staged box
//   bits 16..20  ax,  bits 21..25  ay   (1/32-px fractions)
// sx / sy are clamped to [-2, src_w] / [-2, src_h] like in the bounds pass: at the clamp values
// both taps of that axis read the zero fill of the box.  Slots the tile does not own get 0.
__global__ void __launch_bounds__(32 * MCS_TILED_WARPS)
mcs_tile_desc_kernel(const McsTile* __restrict__ tiles, const McsLayer* __restrict__ layers, int channels,
                     uint32_t* __restrict__ desc) {
    const int t = blockIdx.x;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const McsTile tile = tiles[t];
    const McsLayer& L = layers[tile.layer];
    const int sp = L.bw4 * 4;
    for (int j = 0; j < 8; ++j) {
        const int row = warp + MCS_TILED_WARPS * (j >> 2), col = lane + 32 * (j & 3);
        uint32_t w = 0;
        if (col >= tile.c0 && col < tile.c1 && row < tile.h) {
            const int xl = tile.cx0 + col - L.ox, yl = tile.y0 + row - L.oy;
            int X, Y;
            layer_coords(L, xl, yl, X, Y);
            const int sx = max(-2, min(L.src_w, sat16(X >> 5))), sy = max(-2, min(L.src_h, sat16(Y >> 5)));
            const int b = (sy - tile.by) * sp + sx * channels - 4 * tile.bx;
            w = (uint32_t)b | ((uint32_t)(X & 31) << 16) | ((uint32_t)(Y & 31) << 21);
        }
        desc[(size_t)t * (MCS_CELL_W * MCS_CELL_H) + (j * MCS_TILED_WARPS + warp) * 32 + lane] = w;
    }
}

// Group descriptors of a WARP tile (C == 3): thread (warp, lane) describes, for each of its two cell
// rows (slot 0: row warp, slot 1: row warp + 8), the GROUP of four adjacent pixels at cell columns
// 4 lane .. 4 lane + 3.  At near-unit scale those pixels sample adjacent source pixels of one source
// row pair, so one window of five words per source row serves all four of them.  The template: pixel
// j's taps start 3 j bytes after those of the group's anchor (bA = box byte offset of the first owned
// pixel's tap, minus 3 bytes per preceding column).  A group record is
//   x = bA | ax0 << 16 | ay0 << 21,   y = ax1 | ay1 << 5 | ax2 << 10 | ay2 << 15 | ax3 << 20 | ay3 << 25
// Owned pixels that do not fit the template (the source column or row slips inside the group) go to
// the warp's GENERAL list, one entry per pixel: x = the per-pixel descriptor of mcs_tile_desc_kernel,
// y = slot << 7 | cell column (0xffffffff = unused entry).  The list is stored pass-major
// ([pass][warp][lane]) so that lane l of the warp resamples entries l, 32 + l, ...
// `counts` (analysis, may be nullptr) receives the list length of each warp, saturated at 255; records
// are written when `rec` is not nullptr (entries beyond passes * 32 are dropped: the host only marks
// a tile FAST when every warp's list fits).
__global__ void __launch_bounds__(256)
mcs_tile_fast_kernel(const McsTile* __restrict__ tiles, const McsLayer* __restrict__ layers, int n_tiles,
                     uint8_t* __restrict__ rec, int stride, int passes, uint8_t* __restrict__ counts) {
    const int t = blockIdx.x;
    if (t >= n_tiles) return;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const McsTile tile = tiles[t];
    const McsLayer& L = layers[tile.layer];
    const int sp = L.bw4 * 4;
    uint2 grp[2];
    uint2 gen[8];
    int n_gen = 0;
#pragma unroll
    for (int slot = 0; slot < 2; ++slot) {
        const int row = warp + 8 * slot;
        int b[4], ax[4], ay[4];
        bool own[4];
        int j0 = 4;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int col = 4 * lane + j;
            own[j] = col >= tile.c0 && col < tile.c1 && row < tile.h;
            b[j] = ax[j] = ay[j] = 0;
            if (own[j]) {
                const int xl = tile.cx0 + col - L.ox, yl = tile.y0 + row - L.oy;
                int X, Y;
                layer_coords(L, xl, yl, X, Y);
                const int sx = max(-2, min(L.src_w, sat16(X >> 5))), sy = max(-2, min(L.src_h, sat16(Y >> 5)));
                b[j] = (sy - tile.by) * sp + sx * 3 - 4 * tile.bx;
                ax[j] = X & 31;
                ay[j] = Y & 31;
                if (j0 == 4) j0 = j;
            }
        }
        int bA = j0 < 4 ? b[j0] - 3 * j0 : 0;
        const bool anchored = bA >= 0;   // an anchor left of the box start is not addressable
        if (!anchored) bA = 0;
        uint32_t fx = (uint32_t)bA, fy = 0;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const bool fit = own[j] && anchored && b[j] == bA + 3 * j;
            if (fit) {
                if (j == 0) fx |= ((uint32_t)ax[0] << 16) | ((uint32_t)ay[0] << 21);
                else fy |= (((uint32_t)ax[j]) | ((uint32_t)ay[j] << 5)) << (10 * (j - 1));
            } else if (own[j]) {
                gen[n_gen++] = make_uint2((uint32_t)b[j] | ((uint32_t)ax[j] << 16) | ((uint32_t)ay[j] << 21),
                                          (uint32_t)(slot << 7) | (uint32_t)(4 * lane + j));
            }
        }
        grp[slot] = make_uint2(fx, fy);
    }
    // position of this lane's entries in the warp's list
    int incl = n_gen;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, off);
        if (lane >= off) incl += v;
    }
    const int total = __shfl_sync(0xffffffffu, incl, 31);
    const int first = incl - n_gen;
    if (counts && lane == 0) counts[(size_t)t * 8 + warp] = (uint8_t)min(total, 255);
    if (!rec) return;
    uint8_t* r = rec + (size_t)t * stride;
    if (threadIdx.x < 8) reinterpret_cast<int*>(r)[threadIdx.x] = reinterpret_cast<const int*>(&tiles[t])[threadIdx.x];
    if (lane == 0) r[32 + warp] = (uint8_t)min(total, 255);
    uint2* g = reinterpret_cast<uint2*>(r + MCS_FAST_HEADER_BYTES);
    g[(0 * 8 + warp) * 32 + lane] = grp[0];
    g[(1 * 8 + warp) * 32 + lane] = grp[1];
    uint2* lst = reinterpret_cast<uint2*>(r + MCS_FAST_HEADER_BYTES + MCS_FAST_GROUP_BYTES);
    for (int p = 0; p < passes; ++p) lst[(p * 8 + warp) * 32 + lane] = make_uint2(0u, 0xffffffffu);
    __syncwarp();
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int e = first + i;
        if (i < n_gen && e < passes * 32) lst[((e >> 5) * 8 + warp) * 32 + (e & 31)] = gen[i];
    }
}


// ---- feather mode: seam bands ------------------------------------------------------------------
// Specification: oracle/feather_model.py.  At stage k the running canvas (layers 0 .. k-1) is pasted over the
// warp of layer k; inside the pasted rectangle (that of layer k-1) the two are blended where the weight
// a = weight of the canvas so far is below F = 2^feather_log2 and layer k's warp touches its source:
//   value = (a * value + (F - a) * sample_k + F/2) >> feather_log2
// a comes from the stage's weight map when one was given, else from the distance ramp min(F, 1 + distance to the
// nearest edge of the pasted rectangle).
struct BandMaps {
    const uint8_t* wmap[MCS_MAX_LAYERS];
};

__device__ __forceinline__ int band_weight(const McsLayer* __restrict__ layers, const BandMaps& maps, int k, int x,
                                           int y, int F) {
    const McsLayer& in = layers[k - 1];   // the rectangle pasted at stage k
    if (maps.wmap[k]) return min(F, (int)__ldg(maps.wmap[k] + (size_t)(y - in.py0) * (in.px1 - in.px0) + (x - in.px0)));
    return min(F, min(min(x - in.px0, in.px1 - 1 - x), min(y - in.py0, in.py1 - 1 - y)) + 1);
}

// One warp per (tile, outer layer k): bounding box of the source pixels of layer k that the tile's blended
// pixels sample (as mcs_tile_bounds_kernel); touched = the tile has such pixels.
__global__ void __launch_bounds__(256)
mcs_band_bounds_kernel(const McsTile* __restrict__ tiles, const McsLayer* __restrict__ layers, int n_tiles,
                       int n_layers, int F, const __grid_constant__ BandMaps maps, TileBounds* __restrict__ out) {
    const int job = blockIdx.x * 8 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (job >= n_tiles * n_layers) return;
    const int t = job / n_layers, k = job - t * n_layers;
    const McsTile tile = tiles[t];
    int mnx = INT_MAX, mxx = INT_MIN, mny = INT_MAX, mxy = INT_MIN, touched = 0;
    bool live = tile.layer >= 0 && k > tile.layer;
    if (live && !maps.wmap[k]) {   // ramp: the tile must come within F - 1 pixels of an edge of the pasted rectangle
        const McsLayer& in = layers[k - 1];
        const int x0 = tile.cx0 + tile.c0, x1 = tile.cx0 + tile.c1, y0 = tile.y0, y1 = tile.y0 + tile.h;
        live = x0 < in.px0 + F - 1 || x1 > in.px1 - (F - 1) || y0 < in.py0 + F - 1 || y1 > in.py1 - (F - 1);
    }
    if (live) {
        const McsLayer& L = layers[k];
        const int w = tile.c1 - tile.c0;
        const int n = w * tile.h;
        for (int i = lane; i < n; i += 32) {
            const int r = i / w, c = tile.c0 + (i - r * w);
            const int x = tile.cx0 + c, y = tile.y0 + r;
            if (band_weight(layers, maps, k, x, y, F) >= F) continue;
            int X, Y;
            layer_coords(L, x - L.ox, y - L.oy, X, Y);
            const int rsx = sat16(X >> 5), rsy = sat16(Y >> 5);
            const bool in = ((unsigned)rsx < (unsigned)L.src_w || (unsigned)(rsx + 1) < (unsigned)L.src_w) &&
                            ((unsigned)rsy < (unsigned)L.src_h || (unsigned)(rsy + 1) < (unsigned)L.src_h);
            if (!in) continue;
            touched = 1;
            const int sx = max(-2, min(L.src_w, rsx)), sy = max(-2, min(L.src_h, rsy));
            mnx = min(mnx, sx); mxx = max(mxx, sx);
            mny = min(mny, sy); mxy = max(mxy, sy);
        }
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        mnx = min(mnx, __shfl_xor_sync(0xffffffffu, mnx, off));
        mxx = max(mxx, __shfl_xor_sync(0xffffffffu, mxx, off));
        mny = min(mny, __shfl_xor_sync(0xffffffffu, mny, off));
        mxy = max(mxy, __shfl_xor_sync(0xffffffffu, mxy, off));
        touched |= __shfl_xor_sync(0xffffffffu, touched, off);
    }
    if (lane == 0) {
        TileBounds b;
        b.min_sx = mnx; b.max_sx = mxx; b.min_sy = mny; b.max_sy = mxy; b.touched = touched;
        b.clamped = 0;
        b.pad[0] = b.pad[1] = 0;
        out[job] = b;
    }
}

// One CTA per (BAND tile, overlay slot): the overlay descriptors of the tile's 128 x 16 pixel slots in the
// order of mcs_tile_desc_kernel:  per-pixel descriptor of the outer layer (offset inside ITS staged box, ax,
// ay) | (a + 1) << 26, or 0 where the pixel does not blend with that layer.
__global__ void __launch_bounds__(32 * MCS_TILED_WARPS)
mcs_band_desc_kernel(const McsTile* __restrict__ tiles, const McsLayer* __restrict__ layers, int channels, int F,
                     const __grid_constant__ BandMaps maps, const int4* __restrict__ band_issue,
                     uint32_t* __restrict__ desc) {
    const int t = blockIdx.x / MCS_BAND_MAX_OVERLAYS, o = blockIdx.x - t * MCS_BAND_MAX_OVERLAYS;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const McsTile tile = tiles[t];
    const int4 rec = band_issue[t * (1 + MCS_BAND_MAX_OVERLAYS) + 1 + o];
    const int k = rec.x;
    for (int j = 0; j < 8; ++j) {
        const int row = warp + MCS_TILED_WARPS * (j >> 2), col = lane + 32 * (j & 3);
        uint32_t w = 0;
        if (k >= 0 && col >= tile.c0 && col < tile.c1 && row < tile.h) {
            const McsLayer& L = layers[k];
            const int x = tile.cx0 + col, y = tile.y0 + row;
            const int a = band_weight(layers, maps, k, x, y, F);
            if (a < F) {
                int X, Y;
                layer_coords(L, x - L.ox, y - L.oy, X, Y);
                const int rsx = sat16(X >> 5), rsy = sat16(Y >> 5);
                const bool in = ((unsigned)rsx < (unsigned)L.src_w || (unsigned)(rsx + 1) < (unsigned)L.src_w) &&
                                ((unsigned)rsy < (unsigned)L.src_h || (unsigned)(rsy + 1) < (unsigned)L.src_h);
                if (in) {
                    const int sx = max(-2, min(L.src_w, rsx)), sy = max(-2, min(L.src_h, rsy));
                    const int b = (sy - rec.z) * (L.bw4 * 4) + sx * channels - 4 * rec.y;
                    w = (uint32_t)b | ((uint32_t)(X & 31) << 16) | ((uint32_t)(Y & 31) << 21) | ((uint32_t)(a + 1) << 26);
                }
            }
        }
        desc[((size_t)t * MCS_BAND_MAX_OVERLAYS + o) * (MCS_CELL_W * MCS_CELL_H) + (j * MCS_TILED_WARPS + warp) * 32 + lane] = w;
    }
}

// ---------------------------------------------------------------------------------------------
namespace {

struct Rect { int x0, y0, x1, y1; };

inline bool empty(const Rect& r) { return r.x1 <= r.x0 || r.y1 <= r.y0; }

inline int floor_div(int a, int b) { return (a >= 0) ? a / b : -((-a + b - 1) / b); }

// tiles of `piece` on the grid whose cell columns start at ox + 128*i (the kernel takes any ox;
// the plan anchors every layer at panorama column 0, see mcs_plan_build_tiles)
void tile_piece(std::vector<McsTile>& out, const Rect& piece, int layer, int cls, int ox) {
    if (empty(piece)) return;
    const int i0 = floor_div(piece.x0 - ox, MCS_CELL_W), i1 = floor_div(piece.x1 - 1 - ox, MCS_CELL_W);
    for (int y = piece.y0; y < piece.y1; y += MCS_CELL_H) {
        for (int i = i0; i <= i1; ++i) {
            McsTile t;
            memset(&t, 0, sizeof(t));
            t.cx0 = ox + i * MCS_CELL_W;
            t.y0 = y;
            t.c0 = (short)(std::max(piece.x0, t.cx0) - t.cx0);
            t.c1 = (short)(std::min(piece.x1, t.cx0 + MCS_CELL_W) - t.cx0);
            t.h = (short)std::min(MCS_CELL_H, piece.y1 - y);
            t.layer = (short)layer;
            t.cls = (short)cls;
            out.push_back(t);
        }
    }
}

// outer minus inner (inner inside outer) as up to four rectangles
void ring_pieces(const Rect& outer, const Rect& inner, Rect (&p)[4], int& n) {
    n = 0;
    if (empty(outer)) return;
    if (empty(inner)) { p[n++] = outer; return; }
    p[n++] = Rect{outer.x0, outer.y0, outer.x1, inner.y0};   // top band
    p[n++] = Rect{outer.x0, inner.y1, outer.x1, outer.y1};   // bottom band
    p[n++] = Rect{outer.x0, inner.y0, inner.x0, inner.y1};   // left strip
    p[n++] = Rect{inner.x1, inner.y0, outer.x1, inner.y1};   // right strip
}

void why(mcs_plan* plan, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(plan->tiled_why, sizeof(plan->tiled_why), fmt, ap);
    va_end(ap);
}

}  // namespace

void mcs_plan_free_tiles(mcs_plan* plan) {
    if (plan->d_tiles) cudaFree(plan->d_tiles);
    if (plan->d_layers) cudaFree(plan->d_layers);
    if (plan->d_issue) cudaFree(plan->d_issue);
    plan->d_issue = nullptr;
    if (plan->d_work) cudaFree(plan->d_work);
    if (plan->d_desc) cudaFree(plan->d_desc);
    if (plan->d_fast) cudaFree(plan->d_fast);
    if (plan->d_band_issue) cudaFree(plan->d_band_issue);
    if (plan->d_band_desc) cudaFree(plan->d_band_desc);
    plan->d_desc = nullptr;
    plan->d_fast = nullptr;
    plan->d_band_issue = nullptr;
    plan->d_band_desc = nullptr;
    plan->band_fused = 0;
    plan->n_band = 0;
    plan->band_max_ov = 0;
    for (int k = 0; k < MCS_MAX_LAYERS; ++k) {
        free(plan->h_row_span[k]);
        plan->h_row_span[k] = nullptr;
    }
    plan->src_win_valid = 0;
    plan->d_tiles = nullptr;
    plan->d_layers = nullptr;
    plan->d_work = nullptr;
    plan->tiled_ok = 0;
}

// Estimated cost of one frame of a tile, in consumer-warp instructions of the tiled kernel: the
// slowest warp sets the pace of a cell (all warps share the staged box).
static int tile_cost(const McsTile& t, int fast_passes) {
    if (t.cls == MCS_TILE_ZERO) return 40;
    if (t.cls == MCS_TILE_COPY) return 90;
    if (t.cls == MCS_TILE_FAST) return 70 + 72 * (t.h > MCS_TILED_WARPS ? 2 : 1) + 36 * fast_passes;
    int groups = 0;
    for (int g = 0; g < 4; ++g)
        if (32 * g < t.c1 && 32 * g + 32 > t.c0) ++groups;
    const int px = groups * (t.h > MCS_TILED_WARPS ? 2 : 1);     // pixels per thread of the busiest warp
    if (t.cls == MCS_TILE_BAND) return 63 + 26 * px + 60 * fast_passes;   // fast_passes = overlays here
    return 63 + 26 * px;
}

void mcs_plan_build_tiles(mcs_plan* plan) {
    plan->tiled_ok = 0;
    plan->rows_need_pad = 0;
    plan->src_win_valid = 0;
    plan->tiled_why[0] = 0;
    const int C = plan->channels;
    if (plan->out_w == 0 || plan->out_h == 0) { why(plan, "empty panorama"); return; }

    // rectangles must be nested (innermost first) for the ring decomposition
    Rect inner{0, 0, 0, 0};
    for (int k = 0; k < plan->n_layers; ++k) {
        const McsLayer& L = plan->layers[k];
        Rect r{L.rx0, L.ry0, L.rx1, L.ry1};
        if (!empty(inner) && (empty(r) || r.x0 > inner.x0 || r.y0 > inner.y0 || r.x1 < inner.x1 || r.y1 < inner.y1)) {
            why(plan, "layer rectangles are not nested (layer %d)", k);
            return;
        }
        // TMA addresses a source row as 4-byte words: a row of another length is served only when
        // the caller promises zero bytes up to the next multiple of 4 (mcs_plan_promise_padded_rows)
        if ((L.src_w * C) % 4 != 0) plan->rows_need_pad = 1;
        if (!empty(r)) inner = r;
    }

    std::vector<McsTile> tiles;
    inner = Rect{0, 0, 0, 0};
    for (int k = 0; k < plan->n_layers; ++k) {
        const McsLayer& L = plan->layers[k];
        Rect r{L.rx0, L.ry0, L.rx1, L.ry1};
        if (empty(r)) continue;
        Rect pieces[4];
        int n;
        ring_pieces(r, inner, pieces, n);
        for (int i = 0; i < n; ++i)
            tile_piece(tiles, pieces[i], k, L.kind == MCS_LAYER_COPY ? MCS_TILE_COPY : MCS_TILE_WARP, 0);
        inner = r;
    }
    {   // background: the panorama outside the outermost rectangle
        Rect pieces[4];
        int n;
        ring_pieces(Rect{0, 0, plan->out_w, plan->out_h}, inner, pieces, n);
        for (int i = 0; i < n; ++i) tile_piece(tiles, pieces[i], -1, MCS_TILE_ZERO, 0);
    }
    const int n_tiles = (int)tiles.size();
    if (n_tiles == 0) { why(plan, "no tiles"); return; }

    McsTile* d_tiles = nullptr;
    McsLayer* d_layers = nullptr;
    TileBounds* d_bounds = nullptr;
    std::vector<TileBounds> bounds(n_tiles);
    cudaError_t e = cudaMalloc(&d_tiles, sizeof(McsTile) * n_tiles);
    if (e == cudaSuccess) e = cudaMalloc(&d_layers, sizeof(McsLayer) * MCS_MAX_LAYERS);
    if (e == cudaSuccess) e = cudaMalloc(&d_bounds, sizeof(TileBounds) * n_tiles);
    if (e == cudaSuccess) e = cudaMemcpy(d_tiles, tiles.data(), sizeof(McsTile) * n_tiles, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(d_layers, plan->layers, sizeof(McsLayer) * MCS_MAX_LAYERS, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) {
        mcs_tile_bounds_kernel<<<(n_tiles + 7) / 8, 256>>>(d_tiles, d_layers, n_tiles, d_bounds);
        mcs_count_launch(1);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpy(bounds.data(), d_bounds, sizeof(TileBounds) * n_tiles, cudaMemcpyDeviceToHost);
    if (d_bounds) cudaFree(d_bounds);
    if (e != cudaSuccess) {
        why(plan, "tile analysis failed: %s", cudaGetErrorString(e));
        if (d_tiles) cudaFree(d_tiles);
        if (d_layers) cudaFree(d_layers);
        return;
    }

    // feather mode: which tiles blend with which outer layers (at most MCS_BAND_MAX_OVERLAYS per tile, else
    // the plan keeps the two-pass band path of mcs_stitch.cu)
    struct BandInfo {
        int n;
        int zero_base;   // the owner contributes nothing (untouched): no box of it is staged
        int layer[MCS_BAND_MAX_OVERLAYS], bx[MCS_BAND_MAX_OVERLAYS], by[MCS_BAND_MAX_OVERLAYS];
        TileBounds b[MCS_BAND_MAX_OVERLAYS];
    };
    std::vector<BandInfo> binfo(n_tiles);
    memset(binfo.data(), 0, sizeof(BandInfo) * n_tiles);
    const int F = 1 << plan->feather_log2;
    BandMaps maps;
    for (int k = 0; k < MCS_MAX_LAYERS; ++k) maps.wmap[k] = plan->d_wmap[k];
    bool fused = false;
    {
        const char* env = getenv("MCS_TILED_BAND");   // "0": keep the two-pass band path (tests)
        const bool want = (plan->feather_log2 > 0 || plan->blend_custom) && plan->feather_log2 <= MCS_BAND_MAX_LOG2 && plan->n_layers > 1 &&
                          !(env && atoi(env) == 0);
        if (want) {
            const size_t n_jobs = (size_t)n_tiles * plan->n_layers;
            std::vector<TileBounds> bb(n_jobs);
            TileBounds* d_bb = nullptr;
            e = cudaMalloc(&d_bb, sizeof(TileBounds) * n_jobs);
            if (e == cudaSuccess) {
                mcs_band_bounds_kernel<<<(unsigned)((n_jobs + 7) / 8), 256>>>(d_tiles, d_layers, n_tiles, plan->n_layers, F,
                                                                              maps, d_bb);
                mcs_count_launch(1);
                e = cudaGetLastError();
            }
            if (e == cudaSuccess) e = cudaMemcpy(bb.data(), d_bb, sizeof(TileBounds) * n_jobs, cudaMemcpyDeviceToHost);
            if (d_bb) cudaFree(d_bb);
            fused = e == cudaSuccess;
            for (int i = 0; fused && i < n_tiles; ++i)
                for (int k = 1; fused && k < plan->n_layers; ++k) {
                    const TileBounds& b = bb[(size_t)i * plan->n_layers + k];
                    if (!b.touched) continue;
                    if (binfo[i].n == MCS_BAND_MAX_OVERLAYS) { fused = false; break; }
                    binfo[i].layer[binfo[i].n] = k;
                    binfo[i].b[binfo[i].n] = b;
                    ++binfo[i].n;
                }
            if (!fused) memset(binfo.data(), 0, sizeof(BandInfo) * n_tiles);
            e = cudaSuccess;   // a failed analysis only costs the fused form
        }
    }

    // classify, place the boxes, size them per layer
    int bw4[MCS_MAX_LAYERS], bh[MCS_MAX_LAYERS];
    int win[MCS_MAX_LAYERS][4];   // source pixels the owned tiles of a layer read: x0, y0, x1, y1
    for (int k = 0; k < MCS_MAX_LAYERS; ++k) {
        bw4[k] = bh[k] = 0;
        win[k][0] = win[k][1] = INT_MAX;
        win[k][2] = win[k][3] = INT_MIN;
    }
    std::vector<int> span[MCS_MAX_LAYERS];   // per source row {x0, x1}
    for (int k = 0; k < plan->n_layers; ++k) {
        span[k].resize(2 * (size_t)plan->layers[k].src_h);
        for (int r = 0; r < plan->layers[k].src_h; ++r) { span[k][2 * r] = INT_MAX; span[k][2 * r + 1] = INT_MIN; }
    }
    auto grow = [&](int k, int x0, int y0, int x1, int y1) {
        win[k][0] = std::min(win[k][0], x0); win[k][1] = std::min(win[k][1], y0);
        win[k][2] = std::max(win[k][2], x1); win[k][3] = std::max(win[k][3], y1);
        for (int r = std::max(0, y0); r < y1 && r < plan->layers[k].src_h; ++r) {
            span[k][2 * r] = std::min(span[k][2 * r], x0);
            span[k][2 * r + 1] = std::max(span[k][2 * r + 1], x1);
        }
    };
    for (int i = 0; i < n_tiles; ++i) {
        McsTile& t = tiles[i];
        if (t.layer < 0) continue;
        const McsLayer& L = plan->layers[t.layer];
        int need_w = 0, need_h = 0;
        const bool is_band = binfo[i].n > 0;
        if (is_band) {
            // a BAND tile resamples its owner through per-pixel descriptors (a COPY owner too: taps with
            // ax = ay = 0) and stages one more box per outer layer it blends with
            TileBounds b = bounds[i];
            if (t.cls == MCS_TILE_COPY) {
                b.min_sx = t.cx0 + t.c0 - L.ox; b.max_sx = t.cx0 + t.c1 - 1 - L.ox;
                b.min_sy = t.y0 - L.oy;         b.max_sy = t.y0 + t.h - 1 - L.oy;
                b.touched = 1;
            }
            t.cls = MCS_TILE_BAND;
            if (b.touched) {
                t.bx = 4 * floor_div(b.min_sx * C, 16);
                t.by = b.min_sy;
                need_w = ((b.max_sx + 2) * C + 3) / 4 - t.bx + 1;
                need_h = b.max_sy + 2 - b.min_sy;
                grow(t.layer, std::max(0, b.min_sx), std::max(0, b.min_sy), std::min(L.src_w, b.max_sx + 2),
                     std::min(L.src_h, b.max_sy + 2));
            } else {
                // the owner's warp touches nothing here (background inside its rectangle): the value so far is 0,
                // the kernel stages no box of the owner and starts from zeros
                binfo[i].zero_base = 1;
                t.bx = t.by = 0;
            }
            for (int o = 0; o < binfo[i].n; ++o) {
                const int k = binfo[i].layer[o];
                const McsLayer& K = plan->layers[k];
                const TileBounds& ob = binfo[i].b[o];
                binfo[i].bx[o] = 4 * floor_div(ob.min_sx * C, 16);
                binfo[i].by[o] = ob.min_sy;
                bw4[k] = std::max(bw4[k], ((ob.max_sx + 2) * C + 3) / 4 - binfo[i].bx[o] + 1);
                bh[k] = std::max(bh[k], ob.max_sy + 2 - ob.min_sy);
                grow(k, std::max(0, ob.min_sx), std::max(0, ob.min_sy), std::min(K.src_w, ob.max_sx + 2),
                     std::min(K.src_h, ob.max_sy + 2));
            }
        } else if (t.cls == MCS_TILE_COPY) {
            const int first_byte = (t.cx0 + t.c0 - L.ox) * C, end_byte = (t.cx0 + t.c1 - L.ox) * C;
            t.bx = 4 * floor_div(first_byte, 16);   // TMA: the box must start on a 16-byte boundary
            t.by = t.y0 - L.oy;
            need_w = (end_byte + 3) / 4 - t.bx + 1;   // +1: the realigning write-out reads one word ahead
            need_h = t.h;
            grow(t.layer, t.cx0 + t.c0 - L.ox, t.y0 - L.oy, t.cx0 + t.c1 - L.ox, t.y0 - L.oy + t.h);
        } else if (!bounds[i].touched) {
            t.cls = MCS_TILE_ZERO;
            continue;
        } else {
            const TileBounds& b = bounds[i];
            t.bx = 4 * floor_div(b.min_sx * C, 16);   // TMA: the box must start on a 16-byte boundary
            t.by = b.min_sy;
            need_w = ((b.max_sx + 2) * C + 3) / 4 - t.bx + 1;   // taps sx, sx+1 and one spare word
            need_h = b.max_sy + 2 - b.min_sy;
            grow(t.layer, std::max(0, b.min_sx), std::max(0, b.min_sy), std::min(L.src_w, b.max_sx + 2),
                 std::min(L.src_h, b.max_sy + 2));
        }
        bw4[t.layer] = std::max(bw4[t.layer], need_w);
        bh[t.layer] = std::max(bh[t.layer], need_h);
    }
    int box_bytes = 0;
    for (int k = 0; k < plan->n_layers; ++k) {
        if (bw4[k] == 0) { bw4[k] = 4; bh[k] = 1; }   // layer owns nothing that needs staging
        // box pitch a multiple of 128 bytes (32 banks): when the lanes of a warp straddle two
        // source rows their words still fall into disjoint shared-memory banks
        {
            const char* env = getenv("MCS_TILED_PITCH_WORDS");   // tests: box pitch granularity
            const int g = env && atoi(env) >= 4 ? atoi(env) : 32;
            bw4[k] = (bw4[k] + g - 1) / g * g;
        }
        if (bw4[k] > 256 || bh[k] > 256 || bw4[k] * 4 * bh[k] > MCS_BOX_BYTES_MAX) {
            why(plan, "layer %d needs a %d x %d byte source box per tile (limit 1024 x 256, %d bytes)", k,
                bw4[k] * 4, bh[k], MCS_BOX_BYTES_MAX);
            cudaFree(d_tiles);
            cudaFree(d_layers);
            return;
        }
        plan->layers[k].bw4 = bw4[k];
        plan->layers[k].bh = bh[k];
        box_bytes = std::max(box_bytes, bw4[k] * 4 * bh[k]);
    }
    for (int i = 0; i < n_tiles; ++i) tiles[i].reserved = i;   // the tile's index in `binfo` through the sorts below
    // Work split: tiles grouped by class (each class keeps its layer / row / column order, so a
    // CTA's range covers neighbouring cells), costs prefix-summed for the launch-time cut.
    // Inside a class the tiles run cell row by cell row over the whole panorama width, each row left to right.
    auto by_class = [](const McsTile& a, const McsTile& b) {
        if (a.cls != b.cls) return a.cls > b.cls;
        if (a.y0 / MCS_CELL_H != b.y0 / MCS_CELL_H) return a.y0 / MCS_CELL_H < b.y0 / MCS_CELL_H;
        return a.cx0 < b.cx0;
    };
    std::stable_sort(tiles.begin(), tiles.end(), by_class);
    unsigned* d_work = nullptr;
    e = cudaMemcpy(d_tiles, tiles.data(), sizeof(McsTile) * n_tiles, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(d_layers, plan->layers, sizeof(McsLayer) * MCS_MAX_LAYERS, cudaMemcpyHostToDevice);

    // FAST class (C == 3): WARP tiles whose pixels fit the four-pixel group template but for a short
    // per-warp list.  Analysis pass first (list lengths only), then the records once the table has
    // its final order.
    int first_warp = 0;   // BAND tiles come first
    while (first_warp < n_tiles && tiles[first_warp].cls == MCS_TILE_BAND) ++first_warp;
    int n_warp_tiles = 0;
    while (first_warp + n_warp_tiles < n_tiles && tiles[first_warp + n_warp_tiles].cls == MCS_TILE_WARP) ++n_warp_tiles;
    std::vector<uint8_t> tile_passes(n_tiles, 0);
    int fast_passes = 0, n_fast = 0;
    {
        const char* env = getenv("MCS_TILED_FAST");   // tests: 0 = per-pixel descriptors only
        const bool want = !(env && atoi(env) == 0) && C == 3;
        if (want && e == cudaSuccess && n_warp_tiles > 0) {
            uint8_t* d_counts = nullptr;
            std::vector<uint8_t> counts(8 * (size_t)n_warp_tiles);
            e = cudaMalloc(&d_counts, counts.size());
            if (e == cudaSuccess) {
                mcs_tile_fast_kernel<<<n_warp_tiles, 256>>>(d_tiles + first_warp, d_layers, n_warp_tiles, nullptr, 0, 0, d_counts);
                mcs_count_launch(1);
                e = cudaGetLastError();
            }
            if (e == cudaSuccess) e = cudaMemcpy(counts.data(), d_counts, counts.size(), cudaMemcpyDeviceToHost);
            if (d_counts) cudaFree(d_counts);
            if (e == cudaSuccess) {
                // A general pass costs about as much as one of the eight per-pixel slots it is meant to save
                // (and more shared-memory wavefronts: its lanes hit random banks).  Measured on config 2, whose
                // cameras step 0.93 - 1.13 source pixels per output pixel: with up to 64 pixels per warp off the
                // template (two passes, 86 % of the tiles) 0.877 ms per 64 panoramas against 0.833 ms for the
                // per-pixel path, with up to 32 (one pass, 20 % of the tiles) 0.837 against 0.821.  The group path
                // is therefore kept for tiles that are really at unit scale: at most 12 pixels per warp (5 %) off.
                const char* env_max = getenv("MCS_TILED_FAST_MAX");   // tests
                int limit = env_max ? atoi(env_max) : 12;
                limit = std::max(0, std::min(limit, 32 * MCS_FAST_MAX_PASSES));
                for (int i = 0; i < n_warp_tiles; ++i) {
                    int mx = 0;
                    for (int w = 0; w < 8; ++w) mx = std::max(mx, (int)counts[8 * (size_t)i + w]);
                    if (mx > limit) continue;
                    tiles[first_warp + i].cls = MCS_TILE_FAST;
                    tiles[first_warp + i].flags = (short)((mx + 31) / 32);   // carried through the sort, then replaced by the cost
                    ++n_fast;
                }
                if (n_fast > 0) {
                    std::stable_sort(tiles.begin(), tiles.end(), by_class);
                    for (int i = first_warp; i < first_warp + n_fast; ++i) {
                        tile_passes[i] = (uint8_t)tiles[i].flags;
                        fast_passes = std::max(fast_passes, (int)tiles[i].flags);
                    }
                }
            }
        }
    }
    // the sorts are done: band records in table order, then the staged bytes of every tile (mbarrier transaction count)
    const int n_band = first_warp;
    std::vector<int4> band_issue((size_t)n_band * (1 + MCS_BAND_MAX_OVERLAYS));
    for (int i = 0; i < n_tiles; ++i) {
        McsTile& t = tiles[i];
        const BandInfo bi = binfo[t.reserved];
        t.reserved = t.layer >= 0 ? bw4[t.layer] * 4 * bh[t.layer] : 0;
        if (i < n_band) {
            tile_passes[i] = (uint8_t)bi.n;
            t.reserved |= (bi.n << 24) | (bi.zero_base << 28);   // the tile record and the issue record carry the number of overlays
                                                                 // and the zero-base flag
            int4* r = &band_issue[(size_t)i * (1 + MCS_BAND_MAX_OVERLAYS)];
            r[0] = make_int4(t.layer, t.bx, t.by, t.reserved);
            for (int o = 0; o < MCS_BAND_MAX_OVERLAYS; ++o)
                r[1 + o] = o < bi.n ? make_int4(bi.layer[o], bi.bx[o], bi.by[o], bw4[bi.layer[o]] * 4 * bh[bi.layer[o]])
                                    : make_int4(-1, 0, 0, 0);
        }
    }
    for (int i = 0; i < n_tiles; ++i) tiles[i].flags = (short)tile_cost(tiles[i], tile_passes[i]);
    for (int c = 0; c <= MCS_N_CLASSES; ++c) plan->class_first[c] = n_tiles;
    plan->class_first[0] = 0;
    for (int i = n_tiles - 1; i >= 0; --i) {   // segment s holds class MCS_N_CLASSES - 1 - s
        for (int sgm = 1; sgm < MCS_N_CLASSES; ++sgm)
            if (tiles[i].cls <= MCS_N_CLASSES - 1 - sgm) plan->class_first[sgm] = i;
    }
    int4* d_issue = nullptr;
    {
        std::vector<int4> issue(n_tiles);
        for (int i = 0; i < n_tiles; ++i) issue[i] = make_int4(tiles[i].layer, tiles[i].bx, tiles[i].by, tiles[i].reserved);
        if (e == cudaSuccess) e = cudaMalloc(&d_issue, sizeof(int4) * n_tiles);
        if (e == cudaSuccess) e = cudaMemcpy(d_issue, issue.data(), sizeof(int4) * n_tiles, cudaMemcpyHostToDevice);
    }
    if (e == cudaSuccess) e = cudaMalloc(&d_work, 2 * sizeof(unsigned));
    if (e == cudaSuccess) e = cudaMemset(d_work, 0, 2 * sizeof(unsigned));
    if (e == cudaSuccess) e = cudaMemcpy(d_tiles, tiles.data(), sizeof(McsTile) * n_tiles, cudaMemcpyHostToDevice);
    // per-pixel descriptors of the FAST and WARP tiles (they come first in the sorted table); the FAST
    // tiles keep theirs for launches whose output alignment rules the group path out
    uint32_t* d_desc = nullptr;
    uint8_t* d_fast = nullptr;
    const int fast_stride = MCS_FAST_HEADER_BYTES + MCS_FAST_GROUP_BYTES + fast_passes * MCS_FAST_PASS_BYTES;
    n_warp_tiles = plan->class_first[MCS_SEG(MCS_TILE_COPY)];   // BAND, FAST and WARP tiles
    int4* d_band_issue = nullptr;
    uint32_t* d_band_desc = nullptr;
    if (e == cudaSuccess && n_band > 0) {
        e = cudaMalloc(&d_band_issue, sizeof(int4) * band_issue.size());
        if (e == cudaSuccess)
            e = cudaMemcpy(d_band_issue, band_issue.data(), sizeof(int4) * band_issue.size(), cudaMemcpyHostToDevice);
        if (e == cudaSuccess)
            e = cudaMalloc(&d_band_desc, sizeof(uint32_t) * MCS_CELL_W * MCS_CELL_H * MCS_BAND_MAX_OVERLAYS * (size_t)n_band);
        if (e == cudaSuccess) {
            mcs_band_desc_kernel<<<n_band * MCS_BAND_MAX_OVERLAYS, 32 * MCS_TILED_WARPS>>>(d_tiles, d_layers, C, F, maps,
                                                                                          d_band_issue, d_band_desc);
            mcs_count_launch(1);
            e = cudaGetLastError();
        }
    }
    if (e == cudaSuccess && n_warp_tiles > 0) {
        e = cudaMalloc(&d_desc, sizeof(uint32_t) * MCS_CELL_W * MCS_CELL_H * (size_t)n_warp_tiles);
        if (e == cudaSuccess) {
            mcs_tile_desc_kernel<<<n_warp_tiles, 32 * MCS_TILED_WARPS>>>(d_tiles, d_layers, C, d_desc);
            mcs_count_launch(1);
            e = cudaGetLastError();
        }
        if (e == cudaSuccess && n_fast > 0) {
            e = cudaMalloc(&d_fast, (size_t)fast_stride * n_fast);
            if (e == cudaSuccess) {
                mcs_tile_fast_kernel<<<n_fast, 256>>>(d_tiles + n_band, d_layers, n_fast, d_fast, fast_stride, fast_passes, nullptr);
                mcs_count_launch(1);
                e = cudaGetLastError();
            }
        }
        if (e == cudaSuccess) e = cudaDeviceSynchronize();
    }
    if (e != cudaSuccess) {
        why(plan, "tile upload failed: %s", cudaGetErrorString(e));
        cudaFree(d_tiles);
        cudaFree(d_layers);
        if (d_work) cudaFree(d_work);
        if (d_desc) cudaFree(d_desc);
        if (d_fast) cudaFree(d_fast);
        if (d_issue) cudaFree(d_issue);
        if (d_band_issue) cudaFree(d_band_issue);
        if (d_band_desc) cudaFree(d_band_desc);
        return;
    }
    plan->d_band_issue = d_band_issue;
    plan->d_band_desc = d_band_desc;
    plan->n_band = n_band;
    plan->band_max_ov = 0;
    for (int i = 0; i < n_band; ++i) plan->band_max_ov = std::max(plan->band_max_ov, (int)tile_passes[i]);
    plan->band_fused = fused ? 1 : 0;
    plan->d_issue = d_issue;
    plan->d_fast = d_fast;
    plan->fast_stride = fast_stride;
    plan->fast_passes = fast_passes;
    plan->d_desc = d_desc;
    {
        // frames per sweep of the tile table; $MCS_TILED_FRAME_BLOCK overrides (tests)
        const char* env = getenv("MCS_TILED_FRAME_BLOCK");
        const int v = env ? atoi(env) : 0;
        plan->frame_block = v > 0 ? v : MCS_FRAME_BLOCK_DEFAULT;
    }
    plan->d_work = d_work;
    plan->d_tiles = d_tiles;
    plan->d_layers = d_layers;
    plan->n_tiles = n_tiles;
    plan->box_bytes = (box_bytes + 127) & ~127;
    for (int k = 0; k < plan->n_layers; ++k) {
        const bool none = win[k][0] >= win[k][2] || win[k][1] >= win[k][3];
        for (int j = 0; j < 4; ++j) plan->src_win[k][j] = none ? 0 : win[k][j];
    }
    for (int k = 0; k < plan->n_layers; ++k) {
        plan->h_row_span[k] = static_cast<int*>(malloc(sizeof(int) * span[k].size() + 1));
        if (plan->h_row_span[k]) memcpy(plan->h_row_span[k], span[k].data(), sizeof(int) * span[k].size());
    }
    plan->src_win_valid = 1;
    plan->tiled_ok = 1;
}
