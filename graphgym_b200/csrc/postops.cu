// Fused layer post-ops (SURVEY §8f item 1): what GraphGym's GeneralLayer / GNNStackStage run after a message-passing layer
// (ref: graphgym/models/layer.py:26-46, graphgym/models/gnn.py:76-81):
//     BatchNorm1d (train: batch statistics, eval: running statistics)  ->  activation  ->  optional row-wise L2 normalise
// In eager torch these are 3-4 full passes over [N, F] forward and about twice that backward.  Here:
//   forward   gg_bn_stats_f32     one pass: per-column mean / biased variance (shifted sums per CTA, merged in fp64 in a
//                                 fixed order; running statistics updated in the same finalize kernel)
//             gg_postops_fwd_f32  one pass: normalise + affine + activation (+ L2: the row's norm is reduced in the warp
//                                 that owns the row, the second sweep re-reads the row from L1)
//   backward  gg_postops_bwd_reduce_f32  one pass: column sums of dA and dA * xhat (dgamma, dbeta; train-mode BN only)
//             gg_postops_bwd_apply_f32   one pass: dY
// where dA (gradient at the pre-activation) is recomputed per row from the saved OUTPUT: the activation's gate is the
// sign of the output (ReLU / leaky ReLU, slope > 0), the L2 backward needs <go, out> per row and the saved row norm.
// No atomics: every column reduction is per-CTA partials + a fixed-order merge => deterministic.
//
// The skip blocks of GNNSkipStage (ref: graphgym/models/gnn.py GNNSkipBlock) end in "BN, + the block input (or
// concatenate it), activation"; the same kernels take that residual operand (gg_postops_skip_*_f32, res_mode):
//   SUM     out = l2?(act(BN(y) + res))                             res [n, f]
//   PREFIX  out = l2?([act(res) | act(BN(y))])                      res [n, p], out [n, p + f], the L2 over all p + f
// The backward writes dres = dA beside dy (SUM: the f columns; PREFIX: the p prefix columns) and dy = BN-backward(dA);
// the L2 row dot covers the whole output row, the dgamma / dbeta column sums the f columns only.
#include "common.cuh"

namespace gg {

constexpr int kPoThreads = 256;
constexpr int kPoWarps = kPoThreads / 32;

struct PostArgs {
    const float* y;       // layer output (pre-BN) [n, ld_y]
    int64_t ld_y;
    const float* out;     // post-op output [n, ld_o] (backward: saved)
    int64_t ld_o;
    const float* go;      // backward: gradient wrt out
    int64_t ld_go;
    float* dst;           // forward: out; backward apply: dY
    int64_t ld_dst;
    int64_t n;
    int f;
    const float* mean;    // nullable: no BN
    const float* invstd;
    const float* gamma;   // nullable: no affine
    const float* beta;
    int act;              // GG_ACT_NONE / GG_ACT_RELU / GG_ACT_LRELU
    float slope;
    int l2;               // row-wise L2 normalise (eps 1e-12)
    float* rownorm;       // [n] max(||r||, eps) (forward: written when l2; backward: read)
    int train;            // backward: batch-statistics BN (the mean / variance depend on y)
    const float* dgamma;  // backward apply (train): column sums from the reduce pass
    const float* dbeta;
    float* partial;       // reduce pass: [grid, 2, f]
    int res_mode;         // GG_SKIP_NONE / GG_SKIP_SUM / GG_SKIP_PREFIX
    const float* res;     // forward: the skip operand [n, ld_res] (SUM: f columns, PREFIX: p columns)
    int64_t ld_res;
    int p;                // PREFIX: width of the carried columns; the f columns of out and go start at column p (else 0)
    float* dres;          // backward apply: gradient wrt res [n, ld_dres]
    int64_t ld_dres;
};

__device__ __forceinline__ float po_act(float a, int act, float slope) {
    if (act == GG_ACT_RELU) return a > 0.f ? a : 0.f;
    if (act == GG_ACT_LRELU) return a > 0.f ? a : a * slope;
    return a;
}
__device__ __forceinline__ float po_act_grad(float o, int act, float slope) {  // from the sign of the OUTPUT
    if (act == GG_ACT_RELU) return o > 0.f ? 1.f : 0.f;
    if (act == GG_ACT_LRELU) return o > 0.f ? 1.f : slope;
    return 1.f;
}
template <int V>
__device__ __forceinline__ void po_ld(float (&v)[V], const float* p) {
    if constexpr (V == 4) {
        const float4 t = *reinterpret_cast<const float4*>(p);
        v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
    } else {
        v[0] = *p;
    }
}
template <int V>
__device__ __forceinline__ void po_st(float* p, const float (&v)[V]) {
    if constexpr (V == 4) *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
    else *p = v[0];
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ---- statistics ----------------------------------------------------------------------------------------------------
// Shifted sums per column, s1 = sum(x - K), s2 = sum((x - K)^2) with K = row 0 of y (one shift for the whole matrix, so
// the CTAs' partials simply add; keeps s2 - s1^2/n well conditioned when |mean| >> std).  A warp walks rows — one
// coalesced row segment per load, 4 rows in flight — and keeps its columns' sums in registers; the CTA's 8 warps are
// combined through shared memory in a fixed order.  part[b] = {s1[f], s2[f]}.
template <int V>
__global__ void __launch_bounds__(kPoThreads) bn_stats_partial_kernel(const float* __restrict__ y, int64_t ld, int64_t n,
                                                                      int f, int64_t chunk, float* __restrict__ part) {
    extern __shared__ float sh[];   // [kPoWarps][2][f]
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int64_t r0 = (int64_t)blockIdx.x * chunk;
    const int64_t r1 = r0 + chunk < n ? r0 + chunk : n;
    float* mine = sh + (int64_t)wid * 2 * f;
    for (int c0 = lane * V; c0 < f; c0 += 32 * V) {   // column groups this lane owns
        float K[V], s1[V], s2[V];
#pragma unroll
        for (int q = 0; q < V; ++q) { K[q] = __ldg(y + c0 + q); s1[q] = 0.f; s2[q] = 0.f; }
        int64_t r = r0 + wid;
        for (; r + 3 * kPoWarps < r1; r += 4 * kPoWarps) {
            float v[4][V];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const float* p = y + (r + (int64_t)u * kPoWarps) * ld + c0;
                if (V == 4) *reinterpret_cast<float4*>(v[u]) = *reinterpret_cast<const float4*>(p);
                else v[u][0] = *p;
            }
#pragma unroll
            for (int u = 0; u < 4; ++u)
#pragma unroll
                for (int q = 0; q < V; ++q) {
                    const float d = v[u][q] - K[q];
                    s1[q] += d;
                    s2[q] = fmaf(d, d, s2[q]);
                }
        }
        for (; r < r1; r += kPoWarps) {
            float v[V];
            const float* p = y + r * ld + c0;
            if (V == 4) *reinterpret_cast<float4*>(v) = *reinterpret_cast<const float4*>(p);
            else v[0] = *p;
#pragma unroll
            for (int q = 0; q < V; ++q) {
                const float d = v[q] - K[q];
                s1[q] += d;
                s2[q] = fmaf(d, d, s2[q]);
            }
        }
#pragma unroll
        for (int q = 0; q < V; ++q) { mine[c0 + q] = s1[q]; mine[f + c0 + q] = s2[q]; }
    }
    __syncthreads();
    float* pb = part + (int64_t)blockIdx.x * 2 * f;
    for (int c = threadIdx.x; c < 2 * f; c += kPoThreads) {
        float acc = 0.f;
#pragma unroll
        for (int w = 0; w < kPoWarps; ++w) acc += sh[(int64_t)w * 2 * f + c];   // fixed order
        pb[c] = acc;
    }
}

// the CTAs' partials add up in fp64 in CTA order; also the running-statistics update of BatchNorm1d
// (running = (1 - m) running + m stat, the variance unbiased).
__global__ void __launch_bounds__(256) bn_stats_final_kernel(const float* __restrict__ part, const float* __restrict__ y,
                                                             int blocks, int64_t n, int f, float eps,
                                                             float* __restrict__ mean, float* __restrict__ invstd,
                                                             float* __restrict__ running_mean,
                                                             float* __restrict__ running_var, float momentum) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= f) return;
    double s1 = 0.0, s2 = 0.0;
    for (int b = 0; b < blocks; ++b) {
        s1 += (double)part[(int64_t)b * 2 * f + c];
        s2 += (double)part[(int64_t)b * 2 * f + f + c];
    }
    const double cnt = (double)n;
    const double mu = (double)y[c] + s1 / cnt;
    double m2 = s2 - s1 * s1 / cnt;
    if (m2 < 0.0) m2 = 0.0;
    const double var = m2 / cnt;
    mean[c] = (float)mu;
    invstd[c] = (float)(1.0 / sqrt(var + (double)eps));
    if (running_mean) running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * (float)mu;
    if (running_var) {
        const double unbiased = cnt > 1 ? m2 / (cnt - 1.0) : var;
        running_var[c] = (1.f - momentum) * running_var[c] + momentum * (float)unbiased;
    }
}

// ---- forward -----------------------------------------------------------------------------------------------------
// one warp per row; lanes stride the columns.  The per-column constants (mean, invstd * gamma, beta) are staged in shared
// memory once per CTA — reading them with four __ldg per element made the first version instruction-bound (603 M
// instructions, 1.75 TB/s at F = 128, profiles/r02_sell_postops_ncu_raw.csv).
struct PoCols {
    const float* mu;    // shared-memory arrays [f]
    const float* isg;
    const float* beta;
};
__device__ __forceinline__ PoCols po_stage_cols(const PostArgs& a, float* sh) {
    float* mu = sh;
    float* isg = sh + a.f;
    float* be = sh + 2 * a.f;
    for (int c = threadIdx.x; c < a.f; c += blockDim.x) {
        mu[c] = a.mean ? a.mean[c] : 0.f;
        isg[c] = a.mean ? a.invstd[c] * (a.gamma ? a.gamma[c] : 1.f) : 1.f;
        be[c] = (a.mean && a.gamma) ? a.beta[c] : 0.f;
    }
    __syncthreads();
    return PoCols{mu, isg, be};
}

template <int V>
__global__ void __launch_bounds__(kPoThreads) postops_fwd_kernel(const __grid_constant__ PostArgs a) {
    extern __shared__ float sh[];
    const PoCols pc = po_stage_cols(a, sh);
    const int lane = threadIdx.x & 31;
    const int64_t warps = (int64_t)gridDim.x * kPoWarps;
    constexpr int kKeep = 4;   // column groups of a row a lane keeps in registers (f <= 512 with V = 4)
    for (int64_t r = (int64_t)blockIdx.x * kPoWarps + (threadIdx.x >> 5); r < a.n; r += warps) {
        const float* yr = a.y + r * a.ld_y;
        const float* rr = a.res + r * a.ld_res;       // only read when res_mode != NONE
        float* prow = a.dst + r * a.ld_dst;           // PREFIX: act(res) in [0, p)
        float* orow = prow + a.p;
        float keep[kKeep][V];
        float ss = 0.f;
        if (a.res_mode == GG_SKIP_PREFIX) {
            for (int c = lane * V; c < a.p; c += 32 * V) {
                float v[V];
                po_ld<V>(v, rr + c);
#pragma unroll
                for (int q = 0; q < V; ++q) {
                    v[q] = po_act(v[q], a.act, a.slope);
                    ss = fmaf(v[q], v[q], ss);
                }
                if (!a.l2) po_st<V>(prow + c, v);
            }
        }
        int k = 0;
        for (int c = lane * V; c < a.f; c += 32 * V, ++k) {
            float v[V], s[V];
#pragma unroll
            for (int q = 0; q < V; ++q) s[q] = -0.f;   // x + (-0) == x bitwise: no residual leaves the result as it was
            po_ld<V>(v, yr + c);
            if (a.res_mode == GG_SKIP_SUM) po_ld<V>(s, rr + c);
#pragma unroll
            for (int q = 0; q < V; ++q) {
                v[q] = po_act(fmaf(v[q] - pc.mu[c + q], pc.isg[c + q], pc.beta[c + q]) + s[q], a.act, a.slope);
                ss = fmaf(v[q], v[q], ss);
            }
            if (!a.l2) {
                po_st<V>(orow + c, v);
            } else if (k < kKeep) {
#pragma unroll
                for (int q = 0; q < V; ++q) keep[k][q] = v[q];
            }
        }
        if (!a.l2) continue;
        const float nrm = fmaxf(sqrtf(warp_sum(ss)), 1e-12f);   // F.normalize: x / max(||x||, eps)
        if (lane == 0) a.rownorm[r] = nrm;
        const float scale = 1.f / nrm;
        if (a.res_mode == GG_SKIP_PREFIX) {   // the carried columns are recomputed from the (L1-resident) res row
            for (int c = lane * V; c < a.p; c += 32 * V) {
                float v[V];
                po_ld<V>(v, rr + c);
#pragma unroll
                for (int q = 0; q < V; ++q) v[q] = po_act(v[q], a.act, a.slope) * scale;
                po_st<V>(prow + c, v);
            }
        }
        k = 0;
        for (int c = lane * V; c < a.f; c += 32 * V, ++k) {
            float v[V];
            if (k < kKeep) {
#pragma unroll
                for (int q = 0; q < V; ++q) v[q] = keep[k][q] * scale;
            } else {   // very wide rows: recompute from the (L1-resident) row
                float s[V];
#pragma unroll
                for (int q = 0; q < V; ++q) s[q] = -0.f;
                po_ld<V>(v, yr + c);
                if (a.res_mode == GG_SKIP_SUM) po_ld<V>(s, rr + c);
#pragma unroll
                for (int q = 0; q < V; ++q)
                    v[q] = po_act(fmaf(v[q] - pc.mu[c + q], pc.isg[c + q], pc.beta[c + q]) + s[q], a.act, a.slope) *
                           scale;
            }
            po_st<V>(orow + c, v);
        }
    }
}

// ---- backward ------------------------------------------------------------------------------------------------------
// dA for the columns of one row a lane owns: L2 backward (needs the row's <go, out>, over the whole row: PREFIX columns
// included), then the activation's gate
template <int V>
__device__ __forceinline__ float po_row_dot(const PostArgs& a, int64_t r, int lane) {
    if (!a.l2) return 0.f;
    const float* gr = a.go + r * a.ld_go;
    const float* orow = a.out + r * a.ld_o;
    const int w = a.p + a.f;
    float d = 0.f;
    for (int c = lane * V; c < w; c += 32 * V) {
        if (V == 4) {
            const float4 g = *reinterpret_cast<const float4*>(gr + c), o = *reinterpret_cast<const float4*>(orow + c);
            d = fmaf(g.x, o.x, fmaf(g.y, o.y, fmaf(g.z, o.z, fmaf(g.w, o.w, d))));
        } else {
            d = fmaf(gr[c], orow[c], d);
        }
    }
    return warp_sum(d);
}
__device__ __forceinline__ float po_da(const PostArgs& a, float g, float o, float dot, float inv_norm) {
    if (a.l2) g = (g - o * dot) * inv_norm;   // d/dr of r / max(||r||, eps)   (rows at the eps clamp: ||r|| ~ 0, o ~ 0)
    return g * po_act_grad(o, a.act, a.slope);
}

// column sums of dA and dA * xhat over the CTA's rows -> partial[blockIdx][{0,1}][f]
template <int V>
__global__ void __launch_bounds__(kPoThreads) postops_bwd_reduce_kernel(const __grid_constant__ PostArgs a, int64_t chunk) {
    extern __shared__ float sh[];   // [kPoWarps][2][f] sums, then mean[f], invstd[f]
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    float* mine = sh + (int64_t)wid * 2 * a.f;
    float* s_mu = sh + (int64_t)kPoWarps * 2 * a.f;
    float* s_is = s_mu + a.f;
    for (int c = threadIdx.x; c < a.f; c += kPoThreads) { s_mu[c] = a.mean[c]; s_is[c] = a.invstd[c]; }
    for (int c = lane; c < 2 * a.f; c += 32) mine[c] = 0.f;
    __syncthreads();
    const int64_t r0 = (int64_t)blockIdx.x * chunk;
    const int64_t r1 = r0 + chunk < a.n ? r0 + chunk : a.n;
    for (int64_t r = r0 + wid; r < r1; r += kPoWarps) {
        const float dot = po_row_dot<V>(a, r, lane);
        const float inv_norm = a.l2 ? 1.f / a.rownorm[r] : 1.f;
        const float* gr = a.go + r * a.ld_go + a.p;   // the f columns only (PREFIX: after the carried ones)
        const float* orow = a.out + r * a.ld_o + a.p;
        const float* yr = a.y + r * a.ld_y;
        for (int c = lane * V; c < a.f; c += 32 * V) {
            float g[V], o[V], yv[V];
            if (V == 4) {
                *reinterpret_cast<float4*>(g) = *reinterpret_cast<const float4*>(gr + c);
                *reinterpret_cast<float4*>(o) = *reinterpret_cast<const float4*>(orow + c);
                *reinterpret_cast<float4*>(yv) = *reinterpret_cast<const float4*>(yr + c);
            } else {
                g[0] = gr[c]; o[0] = orow[c]; yv[0] = yr[c];
            }
#pragma unroll
            for (int q = 0; q < V; ++q) {
                const float da = po_da(a, g[q], o[q], dot, inv_norm);
                const float xhat = (yv[q] - s_mu[c + q]) * s_is[c + q];
                mine[c + q] += da;                       // a lane owns its columns: no conflicts inside the warp
                mine[a.f + c + q] = fmaf(da, xhat, mine[a.f + c + q]);
            }
        }
    }
    __syncthreads();
    float* pb = a.partial + (int64_t)blockIdx.x * 2 * a.f;
    for (int c = threadIdx.x; c < 2 * a.f; c += kPoThreads) {
        float s = 0.f;
#pragma unroll
        for (int w = 0; w < kPoWarps; ++w) s += sh[(int64_t)w * 2 * a.f + c];   // fixed order
        pb[c] = s;
    }
}

__global__ void __launch_bounds__(256) postops_bwd_final_kernel(const float* __restrict__ partial, int blocks, int f,
                                                                float* __restrict__ dgamma, float* __restrict__ dbeta) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= f) return;
    double sb = 0.0, sg = 0.0;
    for (int b = 0; b < blocks; ++b) {
        sb += partial[(int64_t)b * 2 * f + c];
        sg += partial[(int64_t)b * 2 * f + f + c];
    }
    dbeta[c] = (float)sb;
    dgamma[c] = (float)sg;
}

template <int V>
__global__ void __launch_bounds__(kPoThreads) postops_bwd_apply_kernel(const __grid_constant__ PostArgs a) {
    extern __shared__ float sh[];   // mean, invstd * gamma, invstd, dbeta / n, dgamma / n   [5][f]
    float* s_mu = sh;
    float* s_isg = sh + a.f;
    float* s_is = sh + 2 * a.f;
    float* s_db = sh + 3 * a.f;
    float* s_dg = sh + 4 * a.f;
    if (a.mean) {
        const float inv_cnt = 1.f / (float)a.n;
        for (int c = threadIdx.x; c < a.f; c += kPoThreads) {
            s_mu[c] = a.mean[c];
            s_is[c] = a.invstd[c];
            s_isg[c] = a.invstd[c] * (a.gamma ? a.gamma[c] : 1.f);
            s_db[c] = a.train ? a.dbeta[c] * inv_cnt : 0.f;
            s_dg[c] = a.train ? a.dgamma[c] * inv_cnt : 0.f;
        }
        __syncthreads();
    }
    const int lane = threadIdx.x & 31;
    const int64_t warps = (int64_t)gridDim.x * kPoWarps;
    for (int64_t r = (int64_t)blockIdx.x * kPoWarps + (threadIdx.x >> 5); r < a.n; r += warps) {
        const float dot = po_row_dot<V>(a, r, lane);
        const float inv_norm = a.l2 ? 1.f / a.rownorm[r] : 1.f;
        const float* gr = a.go + r * a.ld_go + a.p;   // the f columns (PREFIX: after the carried ones)
        const float* orow = a.out + r * a.ld_o + a.p;
        const float* yr = a.y + r * a.ld_y;
        float* drow = a.dst + r * a.ld_dst;
        float* rrow = a.dres + r * a.ld_dres;         // only written when res_mode != NONE
        for (int c = lane * V; c < a.f; c += 32 * V) {
            float g[V], o[V], yv[V], da[V];
            if (V == 4) {
                *reinterpret_cast<float4*>(g) = *reinterpret_cast<const float4*>(gr + c);
                *reinterpret_cast<float4*>(o) = *reinterpret_cast<const float4*>(orow + c);
                if (a.mean && a.train) *reinterpret_cast<float4*>(yv) = *reinterpret_cast<const float4*>(yr + c);
            } else {
                g[0] = gr[c]; o[0] = orow[c];
                if (a.mean && a.train) yv[0] = yr[c];
            }
#pragma unroll
            for (int q = 0; q < V; ++q) {
                float d = po_da(a, g[q], o[q], dot, inv_norm);
                da[q] = d;                                // dA (SUM: dres)
                if (a.mean) {
                    if (a.train) {
                        const float xhat = (yv[q] - s_mu[c + q]) * s_is[c + q];
                        d = d - s_db[c + q] - xhat * s_dg[c + q];
                    }
                    d *= s_isg[c + q];
                }
                g[q] = d;
            }
            if (V == 4) *reinterpret_cast<float4*>(drow + c) = *reinterpret_cast<float4*>(g);
            else drow[c] = g[0];
            if (a.res_mode == GG_SKIP_SUM) po_st<V>(rrow + c, da);
        }
        if (a.res_mode == GG_SKIP_PREFIX) {           // dres = dA on the carried columns
            for (int c = lane * V; c < a.p; c += 32 * V) {
                float g[V], o[V];
                po_ld<V>(g, gr - a.p + c);
                po_ld<V>(o, orow - a.p + c);
#pragma unroll
                for (int q = 0; q < V; ++q) g[q] = po_da(a, g[q], o[q], dot, inv_norm);
                po_st<V>(rrow + c, g);
            }
        }
    }
}

static inline bool po_vec_ok(const void* p, int64_t ld) {
    return !p || ((reinterpret_cast<uintptr_t>(p) & 15) == 0 && ld % 4 == 0);
}
static inline int po_row_grid(int64_t n) {
    int64_t b = ceil_div(n, kPoWarps);
    if (b > (int64_t)kNumSMs * 8) b = (int64_t)kNumSMs * 8;
    return (int)(b < 1 ? 1 : b);
}
static inline int po_chunks(int64_t n, int64_t* chunk) {   // CTAs of a column reduction and their rows
    int64_t blocks = ceil_div(n, 64);
    if (blocks > (int64_t)kNumSMs * 4) blocks = (int64_t)kNumSMs * 4;
    if (blocks < 1) blocks = 1;
    *chunk = ceil_div(n, blocks);
    return (int)ceil_div(n, *chunk > 0 ? *chunk : 1);
}

}  // namespace gg

using namespace gg;

extern "C" {

size_t gg_postops_workspace_bytes(int64_t n, int64_t f) {
    int64_t chunk;
    const int blocks = po_chunks(n > 0 ? n : 1, &chunk);
    return 256 + align_up((size_t)blocks * 3 * (size_t)(f > 0 ? f : 1) * sizeof(float), 256);
}

int gg_bn_stats_f32(const float* y, int64_t ld, int64_t n, int64_t f, float eps, float* mean, float* invstd,
                    float* running_mean, float* running_var, float momentum, void* workspace, size_t workspace_bytes,
                    gg_stream_t stream) {
    GG_REQUIRE(n >= 1 && f >= 1 && f < ((int64_t)1 << 20), "gg_bn_stats_f32: needs n >= 1, 1 <= f < 2^20");
    GG_REQUIRE(y && mean && invstd && workspace && ld >= f, "gg_bn_stats_f32: bad operands");
    if (workspace_bytes < gg_postops_workspace_bytes(n, f)) {
        set_error("gg_bn_stats_f32: workspace %zu < %zu", workspace_bytes, gg_postops_workspace_bytes(n, f));
        return GG_ERR_WORKSPACE;
    }
    cudaStream_t st = as_stream(stream);
    int64_t chunk;
    const int blocks = po_chunks(n, &chunk);
    float* part = static_cast<float*>(workspace);
    const size_t smem = (size_t)kPoWarps * 2 * f * sizeof(float);
    GG_REQUIRE(smem <= 200 * 1024, "gg_bn_stats_f32: f=%lld too wide for the column reduction", (long long)f);
    if (f % 4 == 0 && po_vec_ok(y, ld)) {
        GG_CUDA(cudaFuncSetAttribute(bn_stats_partial_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        bn_stats_partial_kernel<4><<<blocks, kPoThreads, smem, st>>>(y, ld, n, (int)f, chunk, part);
    } else {
        GG_CUDA(cudaFuncSetAttribute(bn_stats_partial_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        bn_stats_partial_kernel<1><<<blocks, kPoThreads, smem, st>>>(y, ld, n, (int)f, chunk, part);
    }
    GG_LAUNCHED();
    bn_stats_final_kernel<<<(int)ceil_div(f, 256), 256, 0, st>>>(part, y, blocks, n, (int)f, eps, mean, invstd,
                                                                running_mean, running_var, momentum);
    GG_LAUNCHED();
    return GG_OK;
}

static int po_check(const char* who, int64_t n, int64_t f, int act) {
    GG_REQUIRE(n >= 0 && f >= 1 && f < ((int64_t)1 << 20), "%s: bad sizes", who);
    GG_REQUIRE(act == GG_ACT_NONE || act == GG_ACT_RELU || act == GG_ACT_LRELU, "%s: act=%d", who, act);
    return GG_OK;
}

// forward and backward of both the plain post-ops (res_mode NONE) and the skip epilogue
static int po_fwd(const char* who, const float* y, int64_t ld_y, const float* res, int64_t ld_res, int64_t n, int64_t f,
                  int64_t p, int mode, const float* mean, const float* invstd, const float* gamma, const float* beta,
                  int act, float slope, int l2norm, float* out, int64_t ld_out, float* rownorm, gg_stream_t stream) {
    int rc = po_check(who, n, f, act);
    if (rc != GG_OK) return rc;
    if (n == 0) return GG_OK;
    GG_REQUIRE(y && out && ld_y >= f && ld_out >= p + f && (!mean || invstd) && (!gamma || beta) && (!l2norm || rownorm),
               "%s: bad operands", who);
    GG_REQUIRE(mode == GG_SKIP_NONE || (res && ld_res >= (mode == GG_SKIP_SUM ? f : p)), "%s: bad residual", who);
    PostArgs a{};
    a.y = y; a.ld_y = ld_y; a.dst = out; a.ld_dst = ld_out; a.n = n; a.f = (int)f; a.mean = mean; a.invstd = invstd;
    a.gamma = gamma; a.beta = beta; a.act = act; a.slope = slope; a.l2 = l2norm; a.rownorm = rownorm;
    a.res_mode = mode; a.res = res; a.ld_res = ld_res; a.p = (int)p;
    const bool vec = f % 4 == 0 && p % 4 == 0 && po_vec_ok(y, ld_y) && po_vec_ok(out, ld_out) && po_vec_ok(res, ld_res);
    const size_t smem = (size_t)3 * f * sizeof(float);
    GG_REQUIRE(smem <= 200 * 1024, "%s: f=%lld too wide", who, (long long)f);
    if (vec) {
        GG_CUDA(cudaFuncSetAttribute(postops_fwd_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        postops_fwd_kernel<4><<<po_row_grid(n), kPoThreads, smem, as_stream(stream)>>>(a);
    } else {
        GG_CUDA(cudaFuncSetAttribute(postops_fwd_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        postops_fwd_kernel<1><<<po_row_grid(n), kPoThreads, smem, as_stream(stream)>>>(a);
    }
    GG_LAUNCHED();
    return GG_OK;
}

static int po_bwd(const char* who, const float* go, int64_t ld_go, const float* out, int64_t ld_out, const float* y,
                  int64_t ld_y, int64_t n, int64_t f, int64_t p, int mode, const float* mean, const float* invstd,
                  const float* gamma, int train, int act, float slope, int l2norm, const float* rownorm, float* dy,
                  int64_t ld_dy, float* dres, int64_t ld_dres, float* dgamma, float* dbeta, void* workspace,
                  size_t workspace_bytes, gg_stream_t stream) {
    int rc = po_check(who, n, f, act);
    if (rc != GG_OK) return rc;
    if (n == 0) return GG_OK;
    GG_REQUIRE(go && out && dy && ld_go >= p + f && ld_out >= p + f && ld_dy >= f &&
                   (!mean || (invstd && y && ld_y >= f)) && (!l2norm || rownorm) &&
                   (!mean || (dgamma && dbeta && workspace)),
               "%s: bad operands", who);
    GG_REQUIRE(mode == GG_SKIP_NONE || (dres && ld_dres >= (mode == GG_SKIP_SUM ? f : p)), "%s: bad residual", who);
    if (mean && workspace_bytes < gg_postops_workspace_bytes(n, f)) {
        set_error("%s: workspace %zu < %zu", who, workspace_bytes, gg_postops_workspace_bytes(n, f));
        return GG_ERR_WORKSPACE;
    }
    cudaStream_t st = as_stream(stream);
    PostArgs a{};
    a.y = y; a.ld_y = ld_y; a.out = out; a.ld_o = ld_out; a.go = go; a.ld_go = ld_go; a.dst = dy; a.ld_dst = ld_dy;
    a.n = n; a.f = (int)f; a.mean = mean; a.invstd = invstd; a.gamma = gamma; a.act = act; a.slope = slope;
    a.l2 = l2norm; a.rownorm = const_cast<float*>(rownorm); a.train = train; a.dgamma = dgamma; a.dbeta = dbeta;
    a.partial = static_cast<float*>(workspace);
    a.res_mode = mode; a.p = (int)p; a.dres = dres; a.ld_dres = ld_dres;
    const bool vec = f % 4 == 0 && p % 4 == 0 && po_vec_ok(go, ld_go) && po_vec_ok(out, ld_out) && po_vec_ok(y, ld_y) &&
                     po_vec_ok(dy, ld_dy) && po_vec_ok(dres, ld_dres);
    if (mean) {   // dgamma / dbeta (also in eval mode: the affine parameters still get gradients)
        int64_t chunk;
        const int blocks = po_chunks(n, &chunk);
        const size_t smem = (size_t)(kPoWarps * 2 + 2) * f * sizeof(float);
        GG_REQUIRE(smem <= 200 * 1024, "%s: f=%lld too wide for the column reduction", who, (long long)f);
        if (vec) {
            GG_CUDA(cudaFuncSetAttribute(postops_bwd_reduce_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            postops_bwd_reduce_kernel<4><<<blocks, kPoThreads, smem, st>>>(a, chunk);
        } else {
            GG_CUDA(cudaFuncSetAttribute(postops_bwd_reduce_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            postops_bwd_reduce_kernel<1><<<blocks, kPoThreads, smem, st>>>(a, chunk);
        }
        GG_LAUNCHED();
        postops_bwd_final_kernel<<<(int)ceil_div(f, 256), 256, 0, st>>>(a.partial, blocks, (int)f, dgamma, dbeta);
        GG_LAUNCHED();
    }
    const size_t smem_apply = (size_t)5 * f * sizeof(float);
    GG_REQUIRE(smem_apply <= 200 * 1024, "%s: f=%lld too wide", who, (long long)f);
    if (vec) {
        GG_CUDA(cudaFuncSetAttribute(postops_bwd_apply_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_apply));
        postops_bwd_apply_kernel<4><<<po_row_grid(n), kPoThreads, smem_apply, st>>>(a);
    } else {
        GG_CUDA(cudaFuncSetAttribute(postops_bwd_apply_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_apply));
        postops_bwd_apply_kernel<1><<<po_row_grid(n), kPoThreads, smem_apply, st>>>(a);
    }
    GG_LAUNCHED();
    return GG_OK;
}

int gg_postops_fwd_f32(const float* y, int64_t ld_y, int64_t n, int64_t f, const float* mean, const float* invstd,
                       const float* gamma, const float* beta, int act, float slope, int l2norm, float* out,
                       int64_t ld_out, float* rownorm, gg_stream_t stream) {
    return po_fwd("gg_postops_fwd_f32", y, ld_y, nullptr, 0, n, f, 0, GG_SKIP_NONE, mean, invstd, gamma, beta, act, slope,
                  l2norm, out, ld_out, rownorm, stream);
}

int gg_postops_bwd_f32(const float* go, int64_t ld_go, const float* out, int64_t ld_out, const float* y, int64_t ld_y,
                       int64_t n, int64_t f, const float* mean, const float* invstd, const float* gamma, int train,
                       int act, float slope, int l2norm, const float* rownorm, float* dy, int64_t ld_dy, float* dgamma,
                       float* dbeta, void* workspace, size_t workspace_bytes, gg_stream_t stream) {
    return po_bwd("gg_postops_bwd_f32", go, ld_go, out, ld_out, y, ld_y, n, f, 0, GG_SKIP_NONE, mean, invstd, gamma, train,
                  act, slope, l2norm, rownorm, dy, ld_dy, nullptr, 0, dgamma, dbeta, workspace, workspace_bytes, stream);
}

static int po_skip_check(const char* who, int mode, int64_t p) {
    GG_REQUIRE((mode == GG_SKIP_SUM && p == 0) || (mode == GG_SKIP_PREFIX && p >= 1 && p < ((int64_t)1 << 20)),
               "%s: mode=%d with p=%lld (SUM takes p = 0, PREFIX 1 <= p < 2^20)", who, mode, (long long)p);
    return GG_OK;
}

int gg_postops_skip_fwd_f32(const float* y, int64_t ld_y, const float* res, int64_t ld_res, int64_t n, int64_t f,
                            int64_t p, int mode, const float* mean, const float* invstd, const float* gamma,
                            const float* beta, int act, float slope, int l2norm, float* out, int64_t ld_out,
                            float* rownorm, gg_stream_t stream) {
    int rc = po_skip_check("gg_postops_skip_fwd_f32", mode, p);
    if (rc != GG_OK) return rc;
    return po_fwd("gg_postops_skip_fwd_f32", y, ld_y, res, ld_res, n, f, p, mode, mean, invstd, gamma, beta, act, slope,
                  l2norm, out, ld_out, rownorm, stream);
}

int gg_postops_skip_bwd_f32(const float* go, int64_t ld_go, const float* out, int64_t ld_out, const float* y,
                            int64_t ld_y, int64_t n, int64_t f, int64_t p, int mode, const float* mean,
                            const float* invstd, const float* gamma, int train, int act, float slope, int l2norm,
                            const float* rownorm, float* dy, int64_t ld_dy, float* dres, int64_t ld_dres, float* dgamma,
                            float* dbeta, void* workspace, size_t workspace_bytes, gg_stream_t stream) {
    int rc = po_skip_check("gg_postops_skip_bwd_f32", mode, p);
    if (rc != GG_OK) return rc;
    return po_bwd("gg_postops_skip_bwd_f32", go, ld_go, out, ld_out, y, ld_y, n, f, p, mode, mean, invstd, gamma, train,
                  act, slope, l2norm, rownorm, dy, ld_dy, dres, ld_dres, dgamma, dbeta, workspace, workspace_bytes, stream);
}

}  // extern "C"
