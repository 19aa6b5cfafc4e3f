// Mean and max aggregation for the attention layers (gaddconv / gmulconv with cfg.gnn.agg = 'mean' / 'max').
//
// The heads = 1 max composes kernels that exist: the attention weights alpha (gat_alpha / segment_softmax), the weighted
// max (spmm_max.cu) and the softmax backward passes (gat_mp.cu).  What is new here:
//   max_winner_sddmm   dalpha[s, k] = sum over the columns c of head k that slot s won (arg[i, c] == s) of
//                      g[i, c] * h[nbr[s], c]: the gradient of the attention weights through the max.  One warp per
//                      target row; lanes that won for the same (slot, head) are grouped with __match_any_sync and their
//                      products are summed by the group's lowest lane in lane order, chunk after chunk, so the sum runs
//                      in column order and is bitwise repeatable (no atomics).  The work per row is O(f), not O(deg).
//   gat_alpha_heads / gat_dz_heads / gat_src_sum_heads
//                      the per-(slot, head) attention weights, the softmax backward and the per-source sums of dz for
//                      heads > 1 (the heads = 1 passes of gat_mp.cu take one weight per slot)
//   spmm_row_max_heads(_bwd)
//                      the weighted max and its masked CSC backward with weight w[s * heads + c / (f / heads)], one warp
//                      per row (the sliced-ELL max stays heads = 1, as the fused sum does)
//   rows_epilogue      out = x / indeg (mean) + per-head rank-1 terms + bias: the mean's scaling of out and of the
//                      incoming gradient, and the score terms da_src att_src + da_tgt att_tgt that the max backward adds
#include <math_constants.h>

#include "common.cuh"

namespace gg {

constexpr int kAaWarps = 8;
constexpr int kAaThreads = kAaWarps * 32;

__device__ __forceinline__ float aa_warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float aa_warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

__global__ void __launch_bounds__(kAaThreads) max_winner_sddmm_kernel(
    const int32_t* __restrict__ rowptr, const int32_t* __restrict__ nbr, const int32_t* __restrict__ arg, int64_t ld_arg,
    const float* __restrict__ g, int64_t ldg, const float* __restrict__ h, int64_t ldh, int64_t n, int f, int c, int heads,
    float* __restrict__ dalpha) {
    __shared__ float sv[kAaWarps][32];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int64_t row = (int64_t)blockIdx.x * kAaWarps + w;
    if (row >= n) return;
    const int64_t beg = __ldg(rowptr + row), end = __ldg(rowptr + row + 1);
    for (int64_t s = beg * heads + lane; s < end * heads; s += 32) dalpha[s] = 0.f;
    __syncwarp();
    for (int c0 = 0; c0 < f; c0 += 32) {
        const int col = c0 + lane;
        int64_t key = -1;
        float v = 0.f;
        if (col < f) {
            const int s = __ldg(arg + row * ld_arg + col);
            if (s >= 0) {
                key = (int64_t)s * heads + col / c;
                v = __ldg(g + row * ldg + col) * __ldg(h + (int64_t)__ldg(nbr + s) * ldh + col);
            }
        }
        const unsigned grp = __match_any_sync(0xffffffffu, key);
        sv[w][lane] = v;
        __syncwarp();
        if (key >= 0 && lane == __ffs(grp) - 1) {
            float acc = 0.f;
            for (unsigned m = grp; m; m &= m - 1) acc += sv[w][__ffs(m) - 1];
            dalpha[key] += acc;
        }
        __syncwarp();
    }
}

// one warp per target row, heads one after the other: alpha[s, k] = softmax over the row of leaky_relu(a_tgt + a_src)
__global__ void __launch_bounds__(kAaThreads) gat_alpha_heads_kernel(
    const int32_t* __restrict__ rowptr, const int32_t* __restrict__ nbr, const float* __restrict__ a_tgt,
    const float* __restrict__ a_src, int64_t n, int heads, float slope, float* __restrict__ alpha) {
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * kAaWarps + (threadIdx.x >> 5);
    if (row >= n) return;
    const int beg = __ldg(rowptr + row), end = __ldg(rowptr + row + 1);
    for (int k = 0; k < heads; ++k) {
        const float at = __ldg(a_tgt + row * heads + k);
        float m = -CUDART_INF_F;
        for (int s = beg + lane; s < end; s += 32) {
            const float z = at + __ldg(a_src + (int64_t)__ldg(nbr + s) * heads + k);
            m = fmaxf(m, z > 0.f ? z : slope * z);
        }
        m = aa_warp_max(m);
        float sum = 0.f;
        for (int s = beg + lane; s < end; s += 32) {
            const float z = at + __ldg(a_src + (int64_t)__ldg(nbr + s) * heads + k);
            sum += expf((z > 0.f ? z : slope * z) - m);
        }
        const float inv = 1.0f / (aa_warp_sum(sum) + 1e-16f);
        for (int s = beg + lane; s < end; s += 32) {
            const float z = at + __ldg(a_src + (int64_t)__ldg(nbr + s) * heads + k);
            alpha[(int64_t)s * heads + k] = expf((z > 0.f ? z : slope * z) - m) * inv;
        }
    }
}

// one warp per target row: D = sum alpha dalpha, dz = alpha (dalpha - D) lrelu'(z), da_tgt = sum dz, per head
__global__ void __launch_bounds__(kAaThreads) gat_dz_heads_kernel(
    const int32_t* __restrict__ rowptr, const int32_t* __restrict__ nbr, const float* __restrict__ a_tgt,
    const float* __restrict__ a_src, const float* __restrict__ alpha, const float* __restrict__ dalpha, int64_t n, int heads,
    float slope, float* __restrict__ dz, float* __restrict__ da_tgt) {
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * kAaWarps + (threadIdx.x >> 5);
    if (row >= n) return;
    const int beg = __ldg(rowptr + row), end = __ldg(rowptr + row + 1);
    for (int k = 0; k < heads; ++k) {
        const float at = __ldg(a_tgt + row * heads + k);
        float d = 0.f;
        for (int s = beg + lane; s < end; s += 32) {
            const int64_t e = (int64_t)s * heads + k;
            d = fmaf(__ldg(alpha + e), __ldg(dalpha + e), d);
        }
        d = aa_warp_sum(d);
        float acc = 0.f;
        for (int s = beg + lane; s < end; s += 32) {
            const int64_t e = (int64_t)s * heads + k;
            const float z = at + __ldg(a_src + (int64_t)__ldg(nbr + s) * heads + k);
            const float v = __ldg(alpha + e) * (__ldg(dalpha + e) - d) * (z > 0.f ? 1.f : slope);
            dz[e] = v;
            acc += v;
        }
        acc = aa_warp_sum(acc);
        if (lane == 0) da_tgt[row * heads + k] = acc;
    }
}

// one warp per source row of the CSC layout: da_src[j, k] = sum over j's out-edges of dz[csr slot, k]
__global__ void __launch_bounds__(kAaThreads) gat_src_sum_heads_kernel(
    const int32_t* __restrict__ rowptr_t, const int32_t* __restrict__ map, const float* __restrict__ dz, int64_t n, int heads,
    float* __restrict__ da_src) {
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * kAaWarps + (threadIdx.x >> 5);
    if (row >= n) return;
    const int beg = __ldg(rowptr_t + row), end = __ldg(rowptr_t + row + 1);
    for (int k = 0; k < heads; ++k) {
        float acc = 0.f;
        for (int t = beg + lane; t < end; t += 32) acc += __ldg(dz + (int64_t)__ldg(map + t) * heads + k);
        acc = aa_warp_sum(acc);
        if (lane == 0) da_src[row * heads + k] = acc;
    }
}

// the weighted max with one weight per (slot, head): the same strict `>` scan as spmm_row_max_kernel
__global__ void __launch_bounds__(kAaThreads) spmm_row_max_heads_kernel(
    const int32_t* __restrict__ rowptr, const int32_t* __restrict__ nbr, const float* __restrict__ w, int heads, int c,
    const float* __restrict__ x, int64_t ldx, float* __restrict__ out, int64_t ldo, int32_t* __restrict__ arg, int64_t ld_arg,
    int64_t n, int f, const float* __restrict__ bias) {
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * kAaWarps + (threadIdx.x >> 5);
    if (row >= n) return;
    const int beg = __ldg(rowptr + row), end = __ldg(rowptr + row + 1);
    for (int col = lane; col < f; col += 32) {
        const int k = col / c;
        float m = -CUDART_INF_F;
        int s = -1;
        for (int e = beg; e < end; ++e) {
            const float v = __ldg(w + (int64_t)e * heads + k) * __ldg(x + (int64_t)__ldg(nbr + e) * ldx + col);
            if (v > m) {
                m = v;
                s = e;
            }
        }
        float r = s >= 0 ? m : 0.f;
        if (bias) r += __ldg(bias + col);
        out[row * ldo + col] = r;
        arg[row * ld_arg + col] = s;
    }
}

// dx[j, col] = sum over j's CSC slots t whose edge won its target's column of w[csr slot, head(col)] * g[target, col]
__global__ void __launch_bounds__(kAaThreads) spmm_row_max_heads_bwd_kernel(
    const int32_t* __restrict__ rowptr, const int32_t* __restrict__ nbr, const int32_t* __restrict__ csc2csr,
    const float* __restrict__ w, int heads, int c, const float* __restrict__ g, int64_t ldg, const int32_t* __restrict__ arg,
    int64_t ld_arg, int64_t n, int f, float* __restrict__ dx, int64_t ldd) {
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * kAaWarps + (threadIdx.x >> 5);
    if (row >= n) return;
    const int beg = __ldg(rowptr + row), end = __ldg(rowptr + row + 1);
    for (int col = lane; col < f; col += 32) {
        const int k = col / c;
        float acc = 0.f;
        for (int t = beg; t < end; ++t) {
            const int64_t i = __ldg(nbr + t);
            const int s = __ldg(csc2csr + t);
            if (__ldg(arg + i * ld_arg + col) == s)
                acc = fmaf(__ldg(w + (int64_t)s * heads + k), __ldg(g + i * ldg + col), acc);
        }
        dx[row * ldd + col] = acc;
    }
}

// out[i, col] = x[i, col] (/ indeg(i) when rowptr is given, 0 rows stay 0) + s1[i, k] v1[col] + s2[i, k] v2[col]
//               + bias[col], k = col / c.  Element-wise: out may alias x.
__global__ void __launch_bounds__(kAaThreads) rows_epilogue_kernel(
    const float* x, int64_t ldx, int64_t n, int f, const int32_t* __restrict__ rowptr, int heads, int c,
    const float* __restrict__ s1, const float* __restrict__ v1, const float* __restrict__ s2, const float* __restrict__ v2,
    const float* __restrict__ bias, float* out, int64_t ldo) {
    const int64_t total = n * (int64_t)f;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t i = e / f;
        const int col = (int)(e - i * f);
        float r = x[i * ldx + col];
        if (rowptr) {
            const int deg = __ldg(rowptr + i + 1) - __ldg(rowptr + i);
            r *= deg > 0 ? 1.0f / (float)deg : 1.0f;
        }
        if (s1) {
            const int64_t ik = i * heads + col / c;
            r = fmaf(__ldg(s1 + ik), __ldg(v1 + col), r);
            r = fmaf(__ldg(s2 + ik), __ldg(v2 + col), r);
        }
        if (bias) r += __ldg(bias + col);
        out[i * ldo + col] = r;
    }
}

static inline int aa_row_grid(int64_t n) { return (int)ceil_div(n, kAaWarps); }

}  // namespace gg

using namespace gg;

extern "C" {

int gg_max_winner_sddmm_f32(const int32_t* rowptr, const int32_t* nbr, const int32_t* arg, int64_t ld_arg, const float* g,
                            int64_t ldg, const float* h, int64_t ldh, int64_t num_rows, int heads, int64_t f, float* dalpha,
                            gg_stream_t stream) {
    GG_REQUIRE(num_rows >= 0 && f >= 0 && heads >= 1, "gg_max_winner_sddmm_f32: bad size");
    if (num_rows == 0) return GG_OK;
    GG_REQUIRE(rowptr && nbr && arg && g && h && dalpha, "gg_max_winner_sddmm_f32: null pointer");
    GG_REQUIRE(f % heads == 0 && f > 0 && f < (1 << 30) && num_rows < ((int64_t)1 << 31),
               "gg_max_winner_sddmm_f32: f=%lld does not split into %d heads", (long long)f, heads);
    GG_REQUIRE(ld_arg >= f && ldg >= f && ldh >= f, "gg_max_winner_sddmm_f32: leading dimension smaller than f");
    max_winner_sddmm_kernel<<<aa_row_grid(num_rows), kAaThreads, 0, as_stream(stream)>>>(
        rowptr, nbr, arg, ld_arg, g, ldg, h, ldh, num_rows, (int)f, (int)(f / heads), heads, dalpha);
    GG_LAUNCHED();
    return GG_OK;
}

int gg_gat_alpha_heads_f32(const int32_t* rowptr, const int32_t* nbr, const float* a_tgt, const float* a_src,
                           int64_t num_rows, int heads, float slope, float* alpha, gg_stream_t stream) {
    GG_REQUIRE(num_rows >= 0 && heads >= 1, "gg_gat_alpha_heads_f32: bad size");
    if (num_rows == 0) return GG_OK;
    GG_REQUIRE(rowptr && nbr && a_tgt && a_src && alpha, "gg_gat_alpha_heads_f32: null pointer");
    GG_REQUIRE(num_rows < ((int64_t)1 << 31), "gg_gat_alpha_heads_f32: size out of range");
    gat_alpha_heads_kernel<<<aa_row_grid(num_rows), kAaThreads, 0, as_stream(stream)>>>(rowptr, nbr, a_tgt, a_src,
                                                                                          num_rows, heads, slope, alpha);
    GG_LAUNCHED();
    return GG_OK;
}

int gg_gat_dz_heads_f32(const int32_t* rowptr, const int32_t* nbr, const float* a_tgt, const float* a_src,
                        const float* alpha, const float* dalpha, int64_t num_rows, int heads, float slope, float* dz,
                        float* da_tgt, gg_stream_t stream) {
    GG_REQUIRE(num_rows >= 0 && heads >= 1, "gg_gat_dz_heads_f32: bad size");
    if (num_rows == 0) return GG_OK;
    GG_REQUIRE(rowptr && nbr && a_tgt && a_src && alpha && dalpha && dz && da_tgt, "gg_gat_dz_heads_f32: null pointer");
    GG_REQUIRE(num_rows < ((int64_t)1 << 31), "gg_gat_dz_heads_f32: size out of range");
    gat_dz_heads_kernel<<<aa_row_grid(num_rows), kAaThreads, 0, as_stream(stream)>>>(
        rowptr, nbr, a_tgt, a_src, alpha, dalpha, num_rows, heads, slope, dz, da_tgt);
    GG_LAUNCHED();
    return GG_OK;
}

int gg_gat_src_sum_heads_f32(const int32_t* rowptr_t, const int32_t* slot_map, const float* dz, int64_t num_rows,
                             int heads, float* da_src, gg_stream_t stream) {
    GG_REQUIRE(num_rows >= 0 && heads >= 1, "gg_gat_src_sum_heads_f32: bad size");
    if (num_rows == 0) return GG_OK;
    GG_REQUIRE(rowptr_t && slot_map && dz && da_src, "gg_gat_src_sum_heads_f32: null pointer");
    GG_REQUIRE(num_rows < ((int64_t)1 << 31), "gg_gat_src_sum_heads_f32: size out of range");
    gat_src_sum_heads_kernel<<<aa_row_grid(num_rows), kAaThreads, 0, as_stream(stream)>>>(rowptr_t, slot_map, dz, num_rows,
                                                                                            heads, da_src);
    GG_LAUNCHED();
    return GG_OK;
}

int gg_spmm_row_max_heads_f32(const int32_t* rowptr, const int32_t* nbr, const float* w, int heads, const float* x,
                              int64_t ldx, float* out, int64_t ldo, int32_t* arg, int64_t ld_arg, int64_t num_rows, int64_t f,
                              const float* bias, gg_stream_t stream) {
    GG_REQUIRE(num_rows >= 0 && f >= 0 && heads >= 1, "gg_spmm_row_max_heads_f32: bad size");
    if (num_rows == 0 || f == 0) return GG_OK;
    GG_REQUIRE(rowptr && nbr && w && x && out && arg, "gg_spmm_row_max_heads_f32: null pointer");
    GG_REQUIRE(f % heads == 0 && f < (1 << 30) && num_rows < ((int64_t)1 << 31),
               "gg_spmm_row_max_heads_f32: f=%lld does not split into %d heads", (long long)f, heads);
    GG_REQUIRE(ldx >= f && ldo >= f && ld_arg >= f, "gg_spmm_row_max_heads_f32: leading dimension smaller than f");
    spmm_row_max_heads_kernel<<<aa_row_grid(num_rows), kAaThreads, 0, as_stream(stream)>>>(
        rowptr, nbr, w, heads, (int)(f / heads), x, ldx, out, ldo, arg, ld_arg, num_rows, (int)f, bias);
    GG_LAUNCHED();
    return GG_OK;
}

int gg_spmm_row_max_heads_bwd_f32(const int32_t* rowptr, const int32_t* nbr, const int32_t* csc2csr, const float* w,
                                  int heads, const float* g, int64_t ldg, const int32_t* arg, int64_t ld_arg, int64_t num_rows,
                                  int64_t f, float* dx, int64_t ldd, gg_stream_t stream) {
    GG_REQUIRE(num_rows >= 0 && f >= 0 && heads >= 1, "gg_spmm_row_max_heads_bwd_f32: bad size");
    if (num_rows == 0 || f == 0) return GG_OK;
    GG_REQUIRE(rowptr && nbr && csc2csr && w && g && arg && dx, "gg_spmm_row_max_heads_bwd_f32: null pointer");
    GG_REQUIRE(f % heads == 0 && f < (1 << 30) && num_rows < ((int64_t)1 << 31),
               "gg_spmm_row_max_heads_bwd_f32: f=%lld does not split into %d heads", (long long)f, heads);
    GG_REQUIRE(ldg >= f && ld_arg >= f && ldd >= f, "gg_spmm_row_max_heads_bwd_f32: leading dimension smaller than f");
    spmm_row_max_heads_bwd_kernel<<<aa_row_grid(num_rows), kAaThreads, 0, as_stream(stream)>>>(
        rowptr, nbr, csc2csr, w, heads, (int)(f / heads), g, ldg, arg, ld_arg, num_rows, (int)f, dx, ldd);
    GG_LAUNCHED();
    return GG_OK;
}

int gg_rows_epilogue_f32(const float* x, int64_t ldx, int64_t num_rows, int64_t f, const int32_t* rowptr, int heads,
                         const float* s1, const float* v1, const float* s2, const float* v2, const float* bias, float* out,
                         int64_t ldo, gg_stream_t stream) {
    GG_REQUIRE(num_rows >= 0 && f >= 0 && heads >= 1, "gg_rows_epilogue_f32: bad size");
    if (num_rows == 0 || f == 0) return GG_OK;
    GG_REQUIRE(x && out && (!s1 || (v1 && s2 && v2)), "gg_rows_epilogue_f32: null pointer");
    GG_REQUIRE(f % heads == 0 && f < (1 << 30), "gg_rows_epilogue_f32: f=%lld does not split into %d heads", (long long)f,
               heads);
    GG_REQUIRE(ldx >= f && ldo >= f, "gg_rows_epilogue_f32: leading dimension smaller than f");
    const int64_t blocks = ceil_div(num_rows * f, kAaThreads);
    const int grid = (int)(blocks < 16 * kNumSMs ? blocks : 16 * kNumSMs);
    rows_epilogue_kernel<<<grid, kAaThreads, 0, as_stream(stream)>>>(x, ldx, num_rows, (int)f, rowptr, heads,
                                                                     (int)(f / heads), s1, v1, s2, v2, bias, out, ldo);
    GG_LAUNCHED();
    return GG_OK;
}

}  // extern "C"
