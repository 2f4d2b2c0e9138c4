// texbake.cu -- texture-space half of the mesh exporter (N5): UV rasteriser, texel positions, export activation +
// quantise + scatter, exact nearest-covered-texel seam fill.  Every stage is integer or per-texel independent, so the
// bake is bit-reproducible (no float atomics).
#include "common.cuh"

namespace {

constexpr int kMinT = 16, kMaxT = 8192;

// fixed point: 8 sub-texel bits; texel (r, c) has its centre at (256c+128, 256r+128)
__device__ __forceinline__ int64_t edge_fn(int64_t ax, int64_t ay, int64_t bx, int64_t by, int64_t px, int64_t py) {
    return (bx - ax) * (py - ay) - (by - ay) * (px - ax);
}
// top-left rule: a centre on the edge a->b belongs to the triangle iff (dy > 0) or (dy == 0 and dx < 0), i.e. iff the
// centre nudged by -(1, eps) is inside.  Two CCW triangles traverse a shared edge in opposite directions, so exactly one
// of them owns a centre on it.
__device__ __forceinline__ bool edge_in(int64_t e, int64_t dx, int64_t dy) {
    return e > 0 || (e == 0 && (dy > 0 || (dy == 0 && dx < 0)));
}
__device__ __forceinline__ int64_t floordiv(int64_t a, int64_t b) {   // b > 0
    return a >= 0 ? a / b : -((-a + b - 1) / b);
}

__global__ void raster_init_kernel(int64_t n, int32_t* __restrict__ owner, float* __restrict__ bary,
                                   uint8_t* __restrict__ mask) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    owner[i] = -1;
    mask[i] = 0;
    bary[3 * i] = 0.0f; bary[3 * i + 1] = 0.0f; bary[3 * i + 2] = 0.0f;
}

// one warp per face walks the texel centres of its bounding box
__global__ void __launch_bounds__(256) uv_raster_kernel(const int2* __restrict__ uv, const int3* __restrict__ tri,
                                                        int64_t n_faces, int T, int32_t* __restrict__ owner,
                                                        float* __restrict__ bary, uint8_t* __restrict__ mask) {
    int64_t f = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    int lane = threadIdx.x & 31;
    if (f >= n_faces) return;
    int3 t = tri[f];
    int2 a = uv[t.x], b = uv[t.y], c = uv[t.z];
    int64_t x0 = a.x, y0 = a.y, x1 = b.x, y1 = b.y, x2 = c.x, y2 = c.y;
    int64_t area = (x1 - x0) * (y2 - y0) - (x2 - x0) * (y1 - y0);
    if (area <= 0) return;                                   // degenerate (or flipped by snapping): covers nothing
    int64_t xmin = min(x0, min(x1, x2)), xmax = max(x0, max(x1, x2));
    int64_t ymin = min(y0, min(y1, y2)), ymax = max(y0, max(y1, y2));
    const int64_t zero = 0, last = T - 1;
    int64_t c_lo = max(floordiv(xmin - 128 + 255, 256), zero), c_hi = min(floordiv(xmax - 128, 256), last);
    int64_t r_lo = max(floordiv(ymin - 128 + 255, 256), zero), r_hi = min(floordiv(ymax - 128, 256), last);
    if (c_hi < c_lo || r_hi < r_lo) return;
    int64_t nw = c_hi - c_lo + 1, cnt = nw * (r_hi - r_lo + 1);
    double inv = 1.0 / (double)area;
    for (int64_t k = lane; k < cnt; k += 32) {
        int64_t r = r_lo + k / nw, cc = c_lo + k % nw;
        int64_t px = 256 * cc + 128, py = 256 * r + 128;
        int64_t e01 = edge_fn(x0, y0, x1, y1, px, py);
        int64_t e12 = edge_fn(x1, y1, x2, y2, px, py);
        int64_t e20 = edge_fn(x2, y2, x0, y0, px, py);
        if (edge_in(e01, x1 - x0, y1 - y0) && edge_in(e12, x2 - x1, y2 - y1) && edge_in(e20, x0 - x2, y0 - y2)) {
            int64_t id = r * T + cc;
            owner[id] = (int32_t)f;
            mask[id] = 1;
            bary[3 * id] = (float)((double)e12 * inv);
            bary[3 * id + 1] = (float)((double)e20 * inv);
            bary[3 * id + 2] = (float)((double)e01 * inv);
        }
    }
}

__global__ void texel_positions_kernel(const int32_t* __restrict__ texels, int64_t n, const int32_t* __restrict__ owner,
                                       const float* __restrict__ bary, const float* __restrict__ v_pos,
                                       const int32_t* __restrict__ t_pos_idx, float* __restrict__ points) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int64_t t = texels[i];
    int64_t f = owner[t];
    f3 p = mk3(0.0f, 0.0f, 0.0f);
#pragma unroll
    for (int k = 0; k < 3; ++k) p = p + bary[3 * t + k] * ld3(v_pos, t_pos_idx[3 * f + k]);
    st3(points, i, p);
}

// dreammat_material.py:765-797 (DreamMatMaterial.export) + the reference's uv_padding quantisation (uint8)(x*255)
__global__ void material_export_kernel(dm_material_cfg cfg, const float* __restrict__ features, int64_t n,
                                       float* __restrict__ out, const int32_t* __restrict__ texels,
                                       uint8_t* __restrict__ kd, uint8_t* __restrict__ pm, uint8_t* __restrict__ pr) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float v[5];
#pragma unroll
    for (int k = 0; k < 5; ++k) v[k] = sigmoidf_(features[5 * i + k]);
    v[3] = v[3] * (cfg.max_metallic - cfg.min_metallic) + cfg.min_metallic;
    v[4] = sqrtf(v[4] * (cfg.max_roughness - cfg.min_roughness) + cfg.min_roughness + 1e-7f);
    if (out) {
#pragma unroll
        for (int k = 0; k < 5; ++k) out[5 * i + k] = v[k];
    }
    if (texels) {
        int64_t t = texels[i];
        kd[3 * t] = (uint8_t)(v[0] * 255.f);
        kd[3 * t + 1] = (uint8_t)(v[1] * 255.f);
        kd[3 * t + 2] = (uint8_t)(v[2] * 255.f);
        pm[t] = (uint8_t)(v[3] * 255.f);
        pr[t] = (uint8_t)(v[4] * 255.f);
    }
}

// ---- exact Euclidean distance transform (Meijster et al. 2000), integer arithmetic throughout.
// Phase 1, one thread per column: vertical distance g to the nearest covered texel of the column and its row (a tie
// between the one above and the one below goes to the one above).
__global__ void edt_cols_kernel(const uint8_t* __restrict__ mask, int T, int32_t* __restrict__ g,
                                int32_t* __restrict__ srow) {
    int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= T) return;
    const int INF = 2 * T;
    int last = -1;
    for (int r = 0; r < T; ++r) {
        if (mask[(int64_t)r * T + c]) last = r;
        srow[(int64_t)r * T + c] = last;
    }
    int next = -1;
    for (int r = T - 1; r >= 0; --r) {
        int64_t id = (int64_t)r * T + c;
        if (mask[id]) next = r;
        int up = srow[id];
        int du = up >= 0 ? r - up : INF, dd = next >= 0 ? next - r : INF;
        bool down = dd < du;
        g[id] = down ? dd : du;
        srow[id] = down ? next : up;
    }
}

// Phase 2, one thread per row: lower envelope of the parabolas (x-u)^2 + g(u)^2 over the columns u; ties keep the
// leftmost column.  s/t are per-row stacks laid out [q*T + row] so that a warp's accesses coalesce.
__global__ void edt_rows_kernel(const int32_t* __restrict__ g, const int32_t* __restrict__ srow, int T,
                                int32_t* __restrict__ s, int32_t* __restrict__ t, int32_t* __restrict__ src) {
    int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= T) return;
    const int64_t INF = 2 * (int64_t)T;
    const int32_t* gr = g + (int64_t)r * T;
    auto G2 = [&](int u) -> int64_t { int64_t v = gr[u]; return v * v; };
    auto F = [&](int64_t x, int i) -> int64_t { return (x - i) * (x - i) + G2(i); };
    int q = 0;
    s[r] = 0; t[r] = 0;
    for (int u = 1; u < T; ++u) {
        while (q >= 0 && F(t[(int64_t)q * T + r], s[(int64_t)q * T + r]) > F(t[(int64_t)q * T + r], u)) --q;
        if (q < 0) {
            q = 0;
            s[r] = u;
        } else {
            int i = s[(int64_t)q * T + r];
            int64_t w = 1 + floordiv((int64_t)u * u - (int64_t)i * i + G2(u) - G2(i), 2 * (int64_t)(u - i));
            if (w < T) {
                ++q;
                s[(int64_t)q * T + r] = u;
                t[(int64_t)q * T + r] = (int32_t)w;
            }
        }
    }
    for (int u = T - 1; u >= 0; --u) {
        int sc = s[(int64_t)q * T + r];
        int64_t id = (int64_t)r * T + u;
        src[id] = gr[sc] >= INF ? -1 : (int32_t)((int64_t)srow[(int64_t)r * T + sc] * T + sc);
        if (u == t[(int64_t)q * T + r]) --q;
    }
}

__global__ void seam_fill_kernel(const int32_t* __restrict__ src, int64_t n, const uint8_t* __restrict__ kd,
                                 const uint8_t* __restrict__ pm, const uint8_t* __restrict__ pr, float* __restrict__ kd_f,
                                 float* __restrict__ pm_f, float* __restrict__ pr_f) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int64_t s = src[i];
    bool ok = s >= 0;
    kd_f[3 * i] = ok ? kd[3 * s] / 255.0f : 0.0f;
    kd_f[3 * i + 1] = ok ? kd[3 * s + 1] / 255.0f : 0.0f;
    kd_f[3 * i + 2] = ok ? kd[3 * s + 2] / 255.0f : 0.0f;
    pm_f[i] = ok ? pm[s] / 255.0f : 0.0f;
    pr_f[i] = ok ? pr[s] / 255.0f : 0.0f;
}

}  // namespace

extern "C" int dm_uv_raster(const int32_t* uv_fixed, const int32_t* tri_uv, int64_t n_faces, int T, int32_t* owner,
                            float* bary, uint8_t* mask, void* stream) {
    DM_REQUIRE(uv_fixed && tri_uv && owner && bary && mask, "null pointer");
    DM_REQUIRE(T >= kMinT && T <= kMaxT, "texture size must be in [16, 8192]");
    DM_REQUIRE(n_faces > 0, "empty mesh");
    cudaStream_t st = (cudaStream_t)stream;
    int64_t n = (int64_t)T * T;
    raster_init_kernel<<<(unsigned)dm_ceil_div(n, 256), 256, 0, st>>>(n, owner, bary, mask);
    DM_CHECK_LAUNCH();
    uv_raster_kernel<<<(unsigned)dm_ceil_div(n_faces * 32, 256), 256, 0, st>>>((const int2*)uv_fixed, (const int3*)tri_uv,
                                                                              n_faces, T, owner, bary, mask);
    DM_CHECK_LAUNCH();
    return DM_OK;
}

extern "C" int dm_texel_positions(const int32_t* texels, int64_t n, const int32_t* owner, const float* bary,
                                  const float* v_pos, const int32_t* t_pos_idx, float* points, void* stream) {
    DM_REQUIRE(texels && owner && bary && v_pos && t_pos_idx && points, "null pointer");
    DM_REQUIRE(n > 0, "no covered texel");
    texel_positions_kernel<<<(unsigned)dm_ceil_div(n, 256), 256, 0, (cudaStream_t)stream>>>(texels, n, owner, bary, v_pos,
                                                                                           t_pos_idx, points);
    DM_CHECK_LAUNCH();
    return DM_OK;
}

extern "C" int dm_material_export(const dm_material_cfg* cfg, const float* features, int64_t n, float* out,
                                  const int32_t* texels, uint8_t* map_kd, uint8_t* map_pm, uint8_t* map_pr, void* stream) {
    DM_REQUIRE(cfg && features, "null pointer");
    DM_REQUIRE(out || texels, "nothing to write");
    DM_REQUIRE(!texels || (map_kd && map_pm && map_pr), "null map pointer");
    DM_REQUIRE(n > 0, "empty input");
    material_export_kernel<<<(unsigned)dm_ceil_div(n, 256), 256, 0, (cudaStream_t)stream>>>(*cfg, features, n, out, texels,
                                                                                           map_kd, map_pm, map_pr);
    DM_CHECK_LAUNCH();
    return DM_OK;
}

extern "C" int dm_seam_fill(const uint8_t* mask, int T, const uint8_t* map_kd, const uint8_t* map_pm,
                            const uint8_t* map_pr, int32_t* scratch, int32_t* src, float* kd_out, float* pm_out,
                            float* pr_out, void* stream) {
    DM_REQUIRE(mask && map_kd && map_pm && map_pr && scratch && src && kd_out && pm_out && pr_out, "null pointer");
    DM_REQUIRE(T >= kMinT && T <= kMaxT, "texture size must be in [16, 8192]");
    cudaStream_t st = (cudaStream_t)stream;
    int64_t n = (int64_t)T * T;
    int32_t *g = scratch, *srow = scratch + n, *s = scratch + 2 * n, *t = scratch + 3 * n;
    // one thread per column / row: warp-sized blocks spread the T sequential scans over as many SMs as possible
    unsigned nb = (unsigned)dm_ceil_div(T, 32);
    edt_cols_kernel<<<nb, 32, 0, st>>>(mask, T, g, srow);
    DM_CHECK_LAUNCH();
    edt_rows_kernel<<<nb, 32, 0, st>>>(g, srow, T, s, t, src);
    DM_CHECK_LAUNCH();
    seam_fill_kernel<<<(unsigned)dm_ceil_div(n, 256), 256, 0, st>>>(src, n, map_kd, map_pm, map_pr, kd_out, pm_out, pr_out);
    DM_CHECK_LAUNCH();
    return DM_OK;
}
