// points.cu -- the refine stage's point renderer: render_point (nerf/refine_utils.py:306-333), i.e. pytorch3d rasterize_points +
// compositing.alpha_composite restated for square images.
//
//   mi3d_point_render_forward : count -> scan -> fill (bin points into 16x16 pixel tiles, lists stay on the device) ->
//                               one CTA per tile: K-best (z, index) per pixel in registers, then the alpha composite
//   mi3d_point_render_backward: one thread per point walks its pixel footprint, finds its slot in each pixel's idx list and sums
//                               g_out * T_k * a_k in a fixed order (no atomics: bit-identical run to run)
//
// The per-pixel order key is (z, point index), a total order, so the result does not depend on the order in which the fill pass
// (atomic cursors) lays a tile's list out.  Compiled with -fmad=false: idx / dists are bit-identical to oracle/points_ref.py.
#include "../../include/mi3d.h"
#include "mi3d_common.cuh"

namespace {

constexpr int TILE = 16;               // tile side in pixels; one raster CTA of TILE*TILE threads per tile
constexpr int BATCH = TILE * TILE;     // points staged through shared memory per round
constexpr uint32_t MAX_K = 16;
constexpr uint32_t MAX_S = 8192;
constexpr unsigned long long EMPTY = ~0ull;

__device__ __forceinline__ bool point_valid(float x, float y, float z) { return isfinite(x) && isfinite(y) && isfinite(z) && z >= 0.f; }

// NDC centre of pixel i (row 0 / column 0 maps to +1): pytorch3d's -1 + (2 (S-1-i) + 1) / S, evaluated in double, rounded once
__device__ __forceinline__ float pix_ndc(int i, int S) { return (float)(-1.0 + (2.0 * (S - 1 - i) + 1.0) / (double)S); }

// inclusive pixel range [lo, hi] along one axis that can hold a pixel centre within rpix pixels of NDC coordinate v: the exact
// range widened by one pixel each side (float rounding), clipped to the image; empty when lo > hi
__device__ __forceinline__ void footprint_axis(float v, float rpix, int S, int& lo, int& hi) {
    const float c = (float)(S - 1) - ((v + 1.f) * (float)S - 1.f) * 0.5f;
    lo = (int)fminf(fmaxf(floorf(c - rpix) - 1.f, 0.f), (float)S);
    hi = (int)fmaxf(fminf(ceilf(c + rpix) + 1.f, (float)(S - 1)), -1.f);
}

__device__ __forceinline__ float rpix_of(float radius, int S) { return radius * (float)S * 0.5f; }

// host twin of the footprint bound: tiles a point can touch, per axis (span of the device footprint is < 2 rpix + 5 pixels)
static uint32_t tiles_per_point_axis(uint32_t S, float radius) {
    const double span = 2.0 * ceil((double)radius * S * 0.5) + 6.0;
    const uint32_t n = (uint32_t)((span + 14.0) / TILE) + 1;
    const uint32_t ntile = mi3d_ceil_div(S, TILE);
    return n < ntile ? n : ntile;
}

struct Ws { uint32_t *counts, *offsets, *cursor, *list; size_t cap, bytes; };

static Ws carve(void* base, uint32_t P, uint32_t S, float radius) {
    const uint32_t nt = mi3d_ceil_div(S, TILE), T = nt * nt;
    const uint32_t tpp = tiles_per_point_axis(S, radius);
    Ws w;
    w.cap = (size_t)P * tpp * tpp;
    auto al = [](size_t b) { return (b + 255) & ~(size_t)255; };
    char* p = (char*)base;
    size_t off = 0;
    w.counts = (uint32_t*)(p + off);  off += al((size_t)T * 4);
    w.offsets = (uint32_t*)(p + off); off += al(((size_t)T + 1) * 4);
    w.cursor = (uint32_t*)(p + off);  off += al((size_t)T * 4);
    w.list = (uint32_t*)(p + off);    off += al(w.cap * 4);
    w.bytes = off;
    return w;
}

// pass 1: entries per tile
__global__ void k_pr_count(const float* __restrict__ pts, uint32_t P, int S, float radius, uint32_t* __restrict__ counts) {
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    const float x = pts[3 * (size_t)p], y = pts[3 * (size_t)p + 1], z = pts[3 * (size_t)p + 2];
    if (!point_valid(x, y, z)) return;
    int x0, x1, y0, y1;
    const float rp = rpix_of(radius, S);
    footprint_axis(x, rp, S, x0, x1);
    footprint_axis(y, rp, S, y0, y1);
    if (x0 > x1 || y0 > y1) return;
    const int nt = (S + TILE - 1) / TILE;
    for (int ty = y0 / TILE; ty <= y1 / TILE; ty++)
        for (int tx = x0 / TILE; tx <= x1 / TILE; tx++) atomicAdd(&counts[ty * nt + tx], 1u);
}

// pass 2: exclusive scan of the T tile counts (one CTA) -> offsets[T + 1] and the fill cursors
__global__ void __launch_bounds__(1024) k_pr_scan(const uint32_t* __restrict__ counts, uint32_t T, uint32_t* __restrict__ offsets,
                                                  uint32_t* __restrict__ cursor) {
    __shared__ uint32_t warp_sums[32];
    const uint32_t per = mi3d_ceil_div(T, blockDim.x);
    const uint32_t b = threadIdx.x * per, e = min(b + per, T);
    uint32_t s = 0;
    for (uint32_t i = b; i < e; i++) s += counts[i];
    // block-wide exclusive scan of the per-thread sums
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t incl = s;
    #pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += v;
    }
    if (lane == 31) warp_sums[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        uint32_t w = lane < blockDim.x / 32 ? warp_sums[lane] : 0;
        #pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t v = __shfl_up_sync(0xffffffffu, w, o);
            if (lane >= o) w += v;
        }
        warp_sums[lane] = w;
    }
    __syncthreads();
    uint32_t run = incl - s + (warp > 0 ? warp_sums[warp - 1] : 0);
    for (uint32_t i = b; i < e; i++) {
        offsets[i] = run;
        cursor[i] = run;
        run += counts[i];
    }
    if (threadIdx.x == blockDim.x - 1) offsets[T] = run;
}

// pass 3: point indices into their tiles' lists (arrival order is free: the raster key is a total order)
__global__ void k_pr_fill(const float* __restrict__ pts, uint32_t P, int S, float radius, uint32_t* __restrict__ cursor,
                          uint32_t* __restrict__ list) {
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    const float x = pts[3 * (size_t)p], y = pts[3 * (size_t)p + 1], z = pts[3 * (size_t)p + 2];
    if (!point_valid(x, y, z)) return;
    int x0, x1, y0, y1;
    const float rp = rpix_of(radius, S);
    footprint_axis(x, rp, S, x0, x1);
    footprint_axis(y, rp, S, y0, y1);
    if (x0 > x1 || y0 > y1) return;
    const int nt = (S + TILE - 1) / TILE;
    for (int ty = y0 / TILE; ty <= y1 / TILE; ty++)
        for (int tx = x0 / TILE; tx <= x1 / TILE; tx++) list[atomicAdd(&cursor[ty * nt + tx], 1u)] = p;
}

// alpha of one selected point from its squared NDC distance: the reference's 1 - sqrt(clamp(0.1 d / r^2, 1e-3, 1))
__device__ __forceinline__ float pr_alpha(float d, float r2) { return 1.f - sqrtf(mi3d_clampf(0.1f * d / r2, 1e-3f, 1.f)); }

// pass 4: one CTA per tile, one thread per pixel.  The tile's list streams through shared memory; each pixel keeps its K smallest
// keys (z bits << 32 | index; z >= 0, so the float bits order like the floats) sorted in registers, then composites.
template <int K>
__global__ void __launch_bounds__(BATCH) k_pr_raster(const float* __restrict__ pts, const float* __restrict__ feats, int C, int S,
                                                    float radius, const uint32_t* __restrict__ offsets, const uint32_t* __restrict__ list,
                                                    int* __restrict__ idx, float* __restrict__ dists, float* __restrict__ out) {
    __shared__ float2 s_xy[BATCH];
    __shared__ unsigned long long s_key[BATCH];
    const int nt = (S + TILE - 1) / TILE;
    const int xi = blockIdx.x * TILE + (threadIdx.x % TILE), yi = blockIdx.y * TILE + (threadIdx.x / TILE);
    const bool live = xi < S && yi < S;
    const float xf = pix_ndc(xi, S), yf = pix_ndc(yi, S), r2 = radius * radius;
    unsigned long long key[K];
    float dk[K];
    #pragma unroll
    for (int k = 0; k < K; k++) { key[k] = EMPTY; dk[k] = -1.f; }

    const uint32_t t = blockIdx.y * nt + blockIdx.x, b = offsets[t], e = offsets[t + 1];
    for (uint32_t base = b; base < e; base += BATCH) {
        const uint32_t n = min((uint32_t)BATCH, e - base);
        __syncthreads();
        if (threadIdx.x < n) {
            const uint32_t p = list[base + threadIdx.x];
            s_xy[threadIdx.x] = make_float2(pts[3 * (size_t)p], pts[3 * (size_t)p + 1]);
            const float z = pts[3 * (size_t)p + 2] + 0.f;   // -0 -> +0
            s_key[threadIdx.x] = ((unsigned long long)__float_as_uint(z) << 32) | p;
        }
        __syncthreads();
        if (!live) continue;
        for (uint32_t j = 0; j < n; j++) {
            const float dx = xf - s_xy[j].x, dy = yf - s_xy[j].y;
            const float d2 = dx * dx + dy * dy;
            const unsigned long long kj = s_key[j];
            if (d2 <= r2 && kj < key[K - 1]) {
                #pragma unroll
                for (int k = K - 1; k > 0; k--) {
                    const bool up = kj < key[k - 1];
                    if (up) { key[k] = key[k - 1]; dk[k] = dk[k - 1]; }
                    else if (kj < key[k]) { key[k] = kj; dk[k] = d2; }
                }
                if (kj < key[0]) { key[0] = kj; dk[0] = d2; }
            }
        }
    }
    if (!live) return;

    const size_t pix = (size_t)yi * S + xi, SS = (size_t)S * S;
    int id[K];
    float w[K];
    float T = 1.f;
    #pragma unroll
    for (int k = 0; k < K; k++) {
        id[k] = key[k] == EMPTY ? -1 : (int)(uint32_t)key[k];
        idx[pix * K + k] = id[k];
        dists[pix * K + k] = dk[k];
        const float a = pr_alpha(dk[k], r2);
        w[k] = T * a;
        T = T * (1.f - a);
    }
    for (int c = 0; c < C; c++) {
        float acc = 0.f;
        #pragma unroll
        for (int k = 0; k < K; k++)
            if (id[k] >= 0) acc += w[k] * __ldg(feats + (size_t)id[k] * C + c);
        out[c * SS + pix] = acc;
    }
}

// backward: g_feats[p] = sum over the (pixel, slot k) holding p of g_out[:, pixel] * T_k a_k, pixels in row-major footprint order
__global__ void k_pr_backward(const float* __restrict__ g_out, const float* __restrict__ pts, const int* __restrict__ idx,
                              const float* __restrict__ dists, uint32_t P, int C, int S, int K, float radius, float* __restrict__ g_feats) {
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    float* g = g_feats + (size_t)p * C;
    for (int c = 0; c < C; c++) g[c] = 0.f;
    const float x = pts[3 * (size_t)p], y = pts[3 * (size_t)p + 1], z = pts[3 * (size_t)p + 2];
    if (!point_valid(x, y, z)) return;
    int x0, x1, y0, y1;
    const float rp = rpix_of(radius, S), r2 = radius * radius;
    footprint_axis(x, rp, S, x0, x1);
    footprint_axis(y, rp, S, y0, y1);
    const size_t SS = (size_t)S * S;
    for (int yi = y0; yi <= y1; yi++)
        for (int xi = x0; xi <= x1; xi++) {
            const size_t pix = (size_t)yi * S + xi;
            const int* ip = idx + pix * K;
            int slot = -1;
            for (int k = 0; k < K; k++)
                if (ip[k] == (int)p) { slot = k; break; }
            if (slot < 0) continue;
            const float* dp = dists + pix * K;
            float T = 1.f, w = 0.f;
            for (int k = 0; k <= slot; k++) {
                const float a = pr_alpha(dp[k], r2);
                w = T * a;
                T = T * (1.f - a);
            }
            for (int c = 0; c < C; c++) g[c] += g_out[c * SS + pix] * w;
        }
}

bool args_ok(uint32_t P, uint32_t C, uint32_t S, uint32_t K, float radius) {
    return P >= 1 && P <= 0x7fffffffu && C >= 1 && S >= 1 && S <= MAX_S && K >= 1 && K <= MAX_K && isfinite(radius) && radius > 0.f;
}

template <int K>
void launch_raster(dim3 grid, cudaStream_t st, const float* pts, const float* feats, int C, int S, float radius, const Ws& w, int* idx,
                   float* dists, float* out) {
    k_pr_raster<K><<<grid, BATCH, 0, st>>>(pts, feats, C, S, radius, w.offsets, w.list, idx, dists, out);
}

}  // namespace

extern "C" {

size_t mi3d_point_render_workspace_bytes(uint32_t P, uint32_t S, uint32_t K, float radius) {
    if (!args_ok(P, 1, S, K, radius)) return 0;
    return carve(nullptr, P, S, radius).bytes;
}

int mi3d_point_render_forward(const float* pts_ndc, const float* feats, uint32_t P, uint32_t C, uint32_t S, uint32_t K, float radius,
                              int* idx, float* dists, float* out, void* workspace, size_t workspace_bytes, mi3d_stream_t stream) {
    if (!args_ok(P, C, S, K, radius) || !pts_ndc || !feats || !idx || !dists || !out || !workspace) return MI3D_ERR_ARG;
    const Ws w = carve(workspace, P, S, radius);
    if (workspace_bytes < w.bytes) return MI3D_ERR_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    const uint32_t nt = mi3d_ceil_div(S, TILE), T = nt * nt;
    MI3D_CHECK(cudaMemsetAsync(w.counts, 0, (size_t)T * 4, st));
    const uint32_t pb = mi3d_ceil_div(P, 256);
    k_pr_count<<<pb, 256, 0, st>>>(pts_ndc, P, (int)S, radius, w.counts);
    k_pr_scan<<<1, 1024, 0, st>>>(w.counts, T, w.offsets, w.cursor);
    k_pr_fill<<<pb, 256, 0, st>>>(pts_ndc, P, (int)S, radius, w.cursor, w.list);
    const dim3 grid(nt, nt);
    switch (K) {
#define PR_CASE(k) case k: launch_raster<k>(grid, st, pts_ndc, feats, (int)C, (int)S, radius, w, idx, dists, out); break;
        PR_CASE(1) PR_CASE(2) PR_CASE(3) PR_CASE(4) PR_CASE(5) PR_CASE(6) PR_CASE(7) PR_CASE(8)
        PR_CASE(9) PR_CASE(10) PR_CASE(11) PR_CASE(12) PR_CASE(13) PR_CASE(14) PR_CASE(15) PR_CASE(16)
#undef PR_CASE
        default: return MI3D_ERR_ARG;
    }
    MI3D_RETURN_LAUNCH();
}

int mi3d_point_render_backward(const float* g_out, const float* pts_ndc, const int* idx, const float* dists, uint32_t P, uint32_t C,
                               uint32_t S, uint32_t K, float radius, float* g_feats, mi3d_stream_t stream) {
    if (!args_ok(P, C, S, K, radius) || !g_out || !pts_ndc || !idx || !dists || !g_feats) return MI3D_ERR_ARG;
    k_pr_backward<<<mi3d_ceil_div(P, 256), 256, 0, (cudaStream_t)stream>>>(g_out, pts_ndc, idx, dists, P, (int)C, (int)S, (int)K, radius,
                                                                          g_feats);
    MI3D_RETURN_LAUNCH();
}

}  // extern "C"
