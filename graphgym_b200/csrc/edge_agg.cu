// Edge-feature message passing (generaledgeconv / generalsampleedgeconv, ref: graphgym/contrib/layer/generalconv.py,
// GeneralEdgeConvLayer).  The message on edge e = (j -> i) is [x_i |] x_j | a_e times W^T; with W split by column blocks
// into W_i, W_j, W_a it is h_i[i] + h_j[j] + a_e W_a^T, h = x W^T node-level GEMMs.  No [E, F] tensor is formed:
//   edge_row_reduce   out[i] = sum over the CSR slots s of row i of a[perm[s]] (/ indeg(i) for the mean), slot order:
//                     the edge term of the add / mean aggregation before its [N, edge_dim] x [edge_dim, F] GEMM.  One
//                     warp per row, lanes over the edge_dim columns.
//   edge_rows_self    out[i] = y[i] + r_i h[i] + z[i], r_i = indeg(i) (add) or [indeg(i) > 0] (mean): the h_i term
//                     and the self term of the add / mean aggregation, and (y = z = 0) the h_i gradient.
//   edge_max          out[i,c] = max over the slots s of row i of h_j[nbr[s],c] + sum_k a[perm[s],k] W_a[c,k], + h_i[i,c]
//                     where the row has a slot, 0 otherwise; + self_scale x_self + bias.  arg = the first slot reaching
//                     the maximum (strict `>` in slot order, -1 for an empty row), as spmm_max.cu.  The edge term is
//                     formed per slot in registers from a W_a column tile staged in shared memory.  Two paths, chosen
//                     as spmm_max's: sliced ELL (f % 4 == 0; the slot_of units give the slot, perm the edge; split rows
//                     combined by the fix-up in piece order) and one warp per row (any f).
//   max_mask          out = g where arg >= 0, else 0: the gradient of h_i through the max.
//   edge_max_winner   da[perm[s], k] = sum over the columns c that slot s of row i won of g[i,c] W_a[c,k], in column
//                     order; 0 for an edge that won no column.  One warp per row; every edge is written once.
//   edge_max_wgrad    dW_a[c,k] = sum_i g[i,c] a[perm[arg[i,c]], k]: per-block partials over row ranges, summed in
//                     block order by a second kernel.
// No atomics on data: every kernel is bitwise run-to-run deterministic.
#include <math_constants.h>

#include "common.cuh"

namespace gg {

constexpr int kEaWarps = 8;
constexpr int kEaThreads = kEaWarps * 32;
constexpr int kEaRows = 8;            // virtual rows per sliced-ELL chunk (= spmm_sell.cu)
constexpr int kEaTile = 128;          // columns per launch of the sliced-ELL max
constexpr int kEaMaxKd = 256;         // edge_dim limit of the max (W_a tile in shared memory)
constexpr int32_t kEaNoRow = INT32_MIN;
constexpr int kEaWgradThreads = 256;

static inline int ea_row_grid(int64_t n) { return (int)ceil_div(n, kEaWarps); }

// ---- add / mean -----------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kEaThreads) edge_row_reduce_kernel(
    const int32_t* __restrict__ rowptr, const int32_t* __restrict__ perm, int64_t n, const float* __restrict__ a,
    int64_t lda, int k, int mean, float* __restrict__ out, int64_t ldo) {
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * kEaWarps + (threadIdx.x >> 5);
    if (row >= n) return;
    const int beg = __ldg(rowptr + row), end = __ldg(rowptr + row + 1);
    for (int c = lane; c < k; c += 32) {
        float acc = 0.f;
        int s = beg;
        for (; s + 4 <= end; s += 4) {   // four rows in flight, added in slot order
            const int64_t e0 = __ldg(perm + s), e1 = __ldg(perm + s + 1), e2 = __ldg(perm + s + 2), e3 = __ldg(perm + s + 3);
            const float v0 = __ldg(a + e0 * lda + c), v1 = __ldg(a + e1 * lda + c), v2 = __ldg(a + e2 * lda + c),
                        v3 = __ldg(a + e3 * lda + c);
            acc += v0; acc += v1; acc += v2; acc += v3;
        }
        for (; s < end; ++s) acc += __ldg(a + (int64_t)__ldg(perm + s) * lda + c);
        if (mean && end > beg) acc /= (float)(end - beg);
        out[row * ldo + c] = acc;
    }
}

__global__ void __launch_bounds__(256) edge_rows_self_kernel(
    const int32_t* __restrict__ rowptr, int64_t n, int f, int mean, const float* y, int64_t ldy,
    const float* __restrict__ h, int64_t ldh, const float* __restrict__ z, int64_t ldz, float* out, int64_t ldo) {
    const int64_t total = n * f;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = e / f, c = e - r * f;
        float v = y ? y[r * ldy + c] : 0.f;
        if (h) {
            const int deg = __ldg(rowptr + r + 1) - __ldg(rowptr + r);
            v = fmaf(mean ? (deg > 0 ? 1.f : 0.f) : (float)deg, __ldg(h + r * ldh + c), v);
        }
        if (z) v += __ldg(z + r * ldz + c);
        out[r * ldo + c] = v;
    }
}

__global__ void __launch_bounds__(256) max_mask_kernel(const float* __restrict__ g, int64_t ldg,
                                                       const int32_t* __restrict__ arg, int64_t ld_arg, int64_t n, int f,
                                                       float* __restrict__ out, int64_t ldo) {
    const int64_t total = n * f;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = e / f, c = e - r * f;
        out[r * ldo + c] = __ldg(arg + r * ld_arg + c) >= 0 ? __ldg(g + r * ldg + c) : 0.f;
    }
}

static inline int ea_elem_grid(int64_t total) {
    int64_t b = ceil_div(total, 256);
    if (b > (int64_t)kNumSMs * 16) b = (int64_t)kNumSMs * 16;
    return (int)(b < 1 ? 1 : b);
}

// ---- max: shared pieces ---------------------------------------------------------------------------------------
struct EdgeMaxArgs {
    const uint32_t* chunk_ptr;
    int chunks;
    const int4* idx4;
    const int4* slot4;
    const int32_t* perm;
    const int32_t* vdst;
    const int32_t* hub_rows;
    const int32_t* hub_pptr;
    int hubs;
    const float* hj;
    int64_t ldj;
    const float* hi;        // nullable: + h_i where the row has a slot
    int64_t ldi;
    const float* a;
    int64_t lda;
    int kd;
    const float* wa;        // [f, kd] rows of ldw
    int64_t ldw;
    float* out;
    int64_t ldo;
    int32_t* arg;
    int64_t ld_arg;
    int f;
    const float* x_self;    // nullable
    int64_t ld_self;
    float self_scale;
    const float* bias;      // nullable
    float* pval;
    int32_t* pslot;
    int* counter;
    int l2_hint;
};

__device__ __forceinline__ void ea_take(float& m, int& s, float v, int slot, bool ok) {
    if (ok && v > m) {
        m = v;
        s = slot;
    }
}
__device__ __forceinline__ int4 ea_ldg_i4(const int4* p, uint64_t pol) {
    int4 r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.s32 {%0,%1,%2,%3}, [%4], %5;"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p), "l"(pol));
    return r;
}

// W_a rows [c0, c0 + tf) transposed into shared memory: sw[k * tf + c] = W_a[c0 + c, k]
__device__ __forceinline__ void ea_stage_wa(float* sw, const float* wa, int64_t ldw, int tf, int kd) {
    for (int t = threadIdx.x; t < tf * kd; t += blockDim.x) {
        const int c = t / kd, k = t - c * kd;
        sw[k * tf + c] = __ldg(wa + (int64_t)c * ldw + k);
    }
    __syncthreads();
}

// out = (m + h_i, or 0 where no slot won) + self_scale * x_self + bias; arg = the winning slots
__device__ __forceinline__ void ea_epilogue4(const EdgeMaxArgs& a, int row, int gl, float4 m, const int4& s, uint64_t pol) {
    if (a.hi) {
        const float4 h = __ldg(reinterpret_cast<const float4*>(a.hi + (int64_t)row * a.ldi) + gl);
        m.x += h.x; m.y += h.y; m.z += h.z; m.w += h.w;
    }
    float4 r = make_float4(s.x >= 0 ? m.x : 0.f, s.y >= 0 ? m.y : 0.f, s.z >= 0 ? m.z : 0.f, s.w >= 0 ? m.w : 0.f);
    if (a.x_self) fma4(r, a.self_scale, __ldg(reinterpret_cast<const float4*>(a.x_self + (int64_t)row * a.ld_self) + gl));
    if (a.bias) add4(r, __ldg(reinterpret_cast<const float4*>(a.bias) + gl));
    stg_f4_hint(reinterpret_cast<float4*>(a.out + (int64_t)row * a.ldo) + gl, r, pol);
    reinterpret_cast<int4*>(a.arg + (int64_t)row * a.ld_arg)[gl] = s;
}

// ---- max, sliced ELL ------------------------------------------------------------------------------------------
// spmm_sell_max_kernel's walk (a warp per chunk of 8 virtual rows, G lanes per row, one float4 of columns per lane) with
// the edge term added to every gathered message before the strict `>`.
template <int G>
__global__ void __launch_bounds__(kEaThreads) edge_sell_max_kernel(const __grid_constant__ EdgeMaxArgs a) {
    extern __shared__ float sw[];
    constexpr int S = 32 / G;
    constexpr int P = kEaRows / S;
    const int lane = threadIdx.x & 31;
    const int grp = lane / G, gl = lane % G;
    const int nvec = a.f >> 2;
    const bool act = gl < nvec;
    const int vl = act ? gl : nvec - 1;
    const char* __restrict__ xg = reinterpret_cast<const char*>(a.hj) + vl * 16;
    const uint32_t row_bytes = (uint32_t)a.ldj * 4u;
    const uint64_t pol_keep = l2_policy(a.l2_hint ? 1 : 0), pol_stream = l2_policy(a.l2_hint ? 2 : 0);
    const float4 ninf4 = make_float4(-CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F);
    const int4 none4 = make_int4(-1, -1, -1, -1);
    const int kd = a.kd;
    ea_stage_wa(sw, a.wa, a.ldw, a.f, kd);
    const float4* __restrict__ swv = reinterpret_cast<const float4*>(sw) + vl;   // column vector vl of row k: swv[k * nvec]
    // message of slot `slot` (edge perm[slot]) from source j: h_j[j] + a_e W_a^T for this lane's four columns
    auto message = [&](int j, int slot) {
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (j >= 0) {
            v = ldg_nc_f4_hint(reinterpret_cast<const float4*>(xg + (uint64_t)(uint32_t)j * row_bytes), pol_keep);
            const float* __restrict__ ar = a.a + (int64_t)__ldg(a.perm + slot) * a.lda;
            float4 p = make_float4(0.f, 0.f, 0.f, 0.f);
            for (int k = 0; k < kd; ++k) fma4(p, __ldg(ar + k), swv[k * nvec]);
            v.x += p.x; v.y += p.y; v.z += p.z; v.w += p.w;
        }
        return v;
    };

    int chunk = 0;
    if (lane == 0) chunk = atomicAdd(a.counter, 1);
    chunk = __shfl_sync(0xffffffffu, chunk, 0);
    while (chunk < a.chunks) {
        int next = 0;
        if (lane == 0) next = atomicAdd(a.counter, 1);
        const uint32_t base = __ldg(a.chunk_ptr + chunk);
        const int nk = (int)(__ldg(a.chunk_ptr + chunk + 1) - base) / kEaRows;
        const int4* __restrict__ ip = a.idx4 + base + grp;
        const int4* __restrict__ sp = a.slot4 + base + grp;
        int4 ia = nk > 0 ? ea_ldg_i4(ip, pol_stream) : none4;
        for (int p = 0; p < P; ++p) {
            float4 m = ninf4;
            int4 s = none4;
            for (int k4 = 0; k4 < nk; ++k4) {
                int4 na = none4;
                if (k4 + 1 < nk) na = ea_ldg_i4(ip + ((k4 + 1) * P + p) * S, pol_stream);
                else if (p + 1 < P) na = ea_ldg_i4(ip + (p + 1) * S, pol_stream);
                const int u = (k4 * P + p) * S;
                const int4 sa = ea_ldg_i4(sp + u, pol_stream);
                const float4 v0 = message(ia.x, sa.x), v1 = message(ia.y, sa.y), v2 = message(ia.z, sa.z),
                             v3 = message(ia.w, sa.w);
                ea_take(m.x, s.x, v0.x, sa.x, ia.x >= 0); ea_take(m.y, s.y, v0.y, sa.x, ia.x >= 0);
                ea_take(m.z, s.z, v0.z, sa.x, ia.x >= 0); ea_take(m.w, s.w, v0.w, sa.x, ia.x >= 0);
                ea_take(m.x, s.x, v1.x, sa.y, ia.y >= 0); ea_take(m.y, s.y, v1.y, sa.y, ia.y >= 0);
                ea_take(m.z, s.z, v1.z, sa.y, ia.y >= 0); ea_take(m.w, s.w, v1.w, sa.y, ia.y >= 0);
                ea_take(m.x, s.x, v2.x, sa.z, ia.z >= 0); ea_take(m.y, s.y, v2.y, sa.z, ia.z >= 0);
                ea_take(m.z, s.z, v2.z, sa.z, ia.z >= 0); ea_take(m.w, s.w, v2.w, sa.z, ia.z >= 0);
                ea_take(m.x, s.x, v3.x, sa.w, ia.w >= 0); ea_take(m.y, s.y, v3.y, sa.w, ia.w >= 0);
                ea_take(m.z, s.z, v3.z, sa.w, ia.w >= 0); ea_take(m.w, s.w, v3.w, sa.w, ia.w >= 0);
                ia = na;
            }
            const int d = __ldg(a.vdst + (int64_t)chunk * kEaRows + p * S + grp);
            if (act) {
                if (d >= 0) ea_epilogue4(a, d, gl, m, s, pol_stream);
                else if (d != kEaNoRow) {
                    const int64_t o = (int64_t)(-d - 1) * a.f;
                    reinterpret_cast<float4*>(a.pval + o)[gl] = m;
                    reinterpret_cast<int4*>(a.pslot + o)[gl] = s;
                }
            }
        }
        chunk = __shfl_sync(0xffffffffu, next, 0);
    }
}

// split rows: the pieces' (max, slot) in piece order with the same strict `>`, then the epilogue
__global__ void __launch_bounds__(256) edge_sell_max_fixup_kernel(const __grid_constant__ EdgeMaxArgs a) {
    const int nvec = a.f >> 2;
    const int64_t total = (int64_t)a.hubs * nvec;
    const uint64_t pol = l2_policy(0);
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int h = (int)(e / nvec), gl = (int)(e - (int64_t)h * nvec);
        const int p0 = __ldg(a.hub_pptr + h), p1 = __ldg(a.hub_pptr + h + 1);
        float4 m = make_float4(-CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F);
        int4 s = make_int4(-1, -1, -1, -1);
        for (int p = p0; p < p1; ++p) {
            const float4 v = reinterpret_cast<const float4*>(a.pval + (int64_t)p * a.f)[gl];
            const int4 q = reinterpret_cast<const int4*>(a.pslot + (int64_t)p * a.f)[gl];
            ea_take(m.x, s.x, v.x, q.x, q.x >= 0);
            ea_take(m.y, s.y, v.y, q.y, q.y >= 0);
            ea_take(m.z, s.z, v.z, q.z, q.z >= 0);
            ea_take(m.w, s.w, v.w, q.w, q.w >= 0);
        }
        ea_epilogue4(a, __ldg(a.hub_rows + h), gl, m, s, pol);
    }
}

static inline size_t ea_smem(int tf, int kd) { return (size_t)tf * kd * sizeof(float); }

template <int G>
static int ea_launch_sell_tile(const EdgeMaxArgs& a, cudaStream_t st) {
    const size_t smem = ea_smem(a.f, a.kd);
    GG_CUDA(cudaFuncSetAttribute(edge_sell_max_kernel<G>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = (int)((200u << 10) / (smem + 1024));
    per_sm = per_sm < 1 ? 1 : (per_sm > 5 ? 5 : per_sm);
    int64_t grid = ceil_div(a.chunks, kEaWarps);
    if (grid > (int64_t)kNumSMs * per_sm) grid = (int64_t)kNumSMs * per_sm;
    edge_sell_max_kernel<G><<<(int)(grid < 1 ? 1 : grid), kEaThreads, smem, st>>>(a);
    count_launch();
    if (a.hubs > 0) {
        edge_sell_max_fixup_kernel<<<ea_elem_grid((int64_t)a.hubs * (a.f >> 2)), 256, 0, st>>>(a);
        count_launch();
    }
    return GG_OK;
}

// ---- max, one warp per row (any f) ----------------------------------------------------------------------------
// block (8 warps, column tile of 32): lane c of the warp of row i scans the row's slots in order
__global__ void __launch_bounds__(kEaThreads) edge_row_max_kernel(
    const int32_t* __restrict__ rowptr, const int32_t* __restrict__ nbr, const int32_t* __restrict__ perm,
    const float* __restrict__ hj, int64_t ldj, const float* __restrict__ hi, int64_t ldi, const float* __restrict__ ea,
    int64_t lda, int kd, const float* __restrict__ wa, int64_t ldw, float* __restrict__ out, int64_t ldo,
    int32_t* __restrict__ arg, int64_t ld_arg, int64_t n, int f, const float* __restrict__ x_self, int64_t ld_self,
    float self_scale, const float* __restrict__ bias) {
    extern __shared__ float sw[];   // [kd][32]
    const int lane = threadIdx.x & 31;
    const int c0 = blockIdx.y * 32;
    const int tf = f - c0 < 32 ? f - c0 : 32;
    for (int t = threadIdx.x; t < 32 * kd; t += blockDim.x) {
        const int c = t / kd, k = t - c * kd;
        sw[k * 32 + c] = c < tf ? __ldg(wa + (int64_t)(c0 + c) * ldw + k) : 0.f;
    }
    __syncthreads();
    const int64_t row = (int64_t)blockIdx.x * kEaWarps + (threadIdx.x >> 5);
    if (row >= n || lane >= tf) return;
    const int c = c0 + lane;
    const int beg = __ldg(rowptr + row), end = __ldg(rowptr + row + 1);
    float m = -CUDART_INF_F;
    int s = -1;
    for (int k = beg; k < end; ++k) {
        const float* __restrict__ ar = ea + (int64_t)__ldg(perm + k) * lda;
        float p = 0.f;
        for (int q = 0; q < kd; ++q) p = fmaf(__ldg(ar + q), sw[q * 32 + lane], p);
        ea_take(m, s, __ldg(hj + (int64_t)__ldg(nbr + k) * ldj + c) + p, k, true);
    }
    if (hi) m += __ldg(hi + row * ldi + c);
    float r = s >= 0 ? m : 0.f;
    if (x_self) r = fmaf(self_scale, __ldg(x_self + row * ld_self + c), r);
    if (bias) r += __ldg(bias + c);
    out[row * ldo + c] = r;
    arg[row * ld_arg + c] = s;
}

// ---- max backward, edge side ----------------------------------------------------------------------------------
// one warp per row: slots in order; the columns a slot won are found by ballots over the arg row, then lanes over k sum
// g[i,c] W_a[c,k] over those columns in column order
__global__ void __launch_bounds__(kEaThreads) edge_max_winner_kernel(
    const int32_t* __restrict__ rowptr, const int32_t* __restrict__ perm, const int32_t* __restrict__ arg, int64_t ld_arg,
    const float* __restrict__ g, int64_t ldg, const float* __restrict__ wa, int64_t ldw, int64_t n, int f, int kd,
    float* __restrict__ da, int64_t ldda) {
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * kEaWarps + (threadIdx.x >> 5);
    if (row >= n) return;
    const int beg = __ldg(rowptr + row), end = __ldg(rowptr + row + 1);
    const int32_t* __restrict__ ar = arg + row * ld_arg;
    const float* __restrict__ gr = g + row * ldg;
    for (int s = beg; s < end; ++s) {
        bool won = false;
        for (int c0 = 0; c0 < f && !won; c0 += 32) {
            const int c = c0 + lane;
            won = __any_sync(0xffffffffu, c < f && __ldg(ar + c) == s);
        }
        float* __restrict__ dst = da + (int64_t)__ldg(perm + s) * ldda;
        if (!won) {
            for (int k = lane; k < kd; k += 32) dst[k] = 0.f;
            continue;
        }
        for (int k0 = 0; k0 < kd; k0 += 32) {
            const int k = k0 + lane;
            float acc = 0.f;
            for (int c0 = 0; c0 < f; c0 += 32) {
                const int c = c0 + lane;
                unsigned mask = __ballot_sync(0xffffffffu, c < f && __ldg(ar + c) == s);
                for (; mask; mask &= mask - 1) {
                    const int cc = c0 + __ffs(mask) - 1;
                    if (k < kd) acc = fmaf(__ldg(gr + cc), __ldg(wa + (int64_t)cc * ldw + k), acc);
                }
            }
            if (k < kd) dst[k] = acc;
        }
    }
}

// partial[b, c * kd + k] = sum over the rows of block-row range b of g[i,c] a[perm[arg[i,c]], k]
__global__ void __launch_bounds__(kEaWgradThreads) edge_max_wgrad_partial_kernel(
    const int32_t* __restrict__ perm, const int32_t* __restrict__ arg, int64_t ld_arg, const float* __restrict__ g,
    int64_t ldg, const float* __restrict__ ea, int64_t lda, int64_t n, int f, int kd, int64_t rows_per_block,
    float* __restrict__ part) {
    const int64_t fk = (int64_t)f * kd;
    const int64_t p = (int64_t)blockIdx.y * kEaWgradThreads + threadIdx.x;
    if (p >= fk) return;
    const int c = (int)(p / kd), k = (int)(p - (int64_t)c * kd);
    const int64_t r0 = (int64_t)blockIdx.x * rows_per_block;
    const int64_t r1 = r0 + rows_per_block < n ? r0 + rows_per_block : n;
    float acc = 0.f;
    for (int64_t i = r0; i < r1; ++i) {
        const int s = __ldg(arg + i * ld_arg + c);
        if (s >= 0) acc = fmaf(__ldg(g + i * ldg + c), __ldg(ea + (int64_t)__ldg(perm + s) * lda + k), acc);
    }
    part[(int64_t)blockIdx.x * fk + p] = acc;
}

__global__ void __launch_bounds__(256) edge_max_wgrad_reduce_kernel(const float* __restrict__ part, int blocks, int f,
                                                                    int kd, float* __restrict__ dw, int64_t lddw) {
    const int64_t fk = (int64_t)f * kd;
    for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < fk; p += (int64_t)gridDim.x * blockDim.x) {
        float acc = 0.f;
        for (int b = 0; b < blocks; ++b) acc += part[(int64_t)b * fk + p];
        const int64_t c = p / kd, k = p - c * kd;
        dw[c * lddw + k] = acc;
    }
}

// (row blocks, rows per block) of the dW_a partials: about 8 resident blocks per SM in all
static inline void ea_wgrad_split(int64_t n, int64_t f, int64_t kd, int64_t* blocks, int64_t* rows) {
    const int64_t tiles = ceil_div(f * kd, kEaWgradThreads);
    int64_t b = (int64_t)kNumSMs * 8 / (tiles > 0 ? tiles : 1);
    const int64_t cap = ceil_div(n, 64);
    if (b > cap) b = cap;
    if (b < 1) b = 1;
    *rows = ceil_div(n, b);
    *blocks = ceil_div(n, *rows);
}

static inline bool ea_al16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

}  // namespace gg

using namespace gg;

extern "C" {

int gg_edge_row_reduce_f32(const int32_t* rowptr, const int32_t* perm, int64_t num_rows, const float* a, int64_t lda,
                           int64_t k, int mean, float* out, int64_t ldo, gg_stream_t stream) {
    GG_REQUIRE(num_rows >= 0 && k >= 0, "gg_edge_row_reduce_f32: negative size");
    if (num_rows == 0 || k == 0) return GG_OK;
    GG_REQUIRE(rowptr && out, "gg_edge_row_reduce_f32: null pointer");   // perm / a: null for a layout without slots
    GG_REQUIRE(lda >= k && ldo >= k && num_rows < ((int64_t)1 << 31) && k < (1 << 30),
               "gg_edge_row_reduce_f32: bad leading dimension or size");
    edge_row_reduce_kernel<<<ea_row_grid(num_rows), kEaThreads, 0, as_stream(stream)>>>(rowptr, perm, num_rows, a, lda,
                                                                                         (int)k, mean, out, ldo);
    GG_LAUNCHED();
    return GG_OK;
}

int gg_edge_rows_self_f32(const int32_t* rowptr, int64_t num_rows, int64_t f, int mean, const float* y, int64_t ldy,
                          const float* h, int64_t ldh, const float* z, int64_t ldz, float* out, int64_t ldo,
                          gg_stream_t stream) {
    GG_REQUIRE(num_rows >= 0 && f >= 0, "gg_edge_rows_self_f32: negative size");
    if (num_rows == 0 || f == 0) return GG_OK;
    GG_REQUIRE(rowptr && out, "gg_edge_rows_self_f32: null pointer");
    GG_REQUIRE(ldo >= f && (!h || ldh >= f) && (!y || ldy >= f) && (!z || ldz >= f) && f < (1 << 30),
               "gg_edge_rows_self_f32: bad leading dimension");
    edge_rows_self_kernel<<<ea_elem_grid(num_rows * f), 256, 0, as_stream(stream)>>>(rowptr, num_rows, (int)f, mean, y, ldy,
                                                                                    h, ldh, z, ldz, out, ldo);
    GG_LAUNCHED();
    return GG_OK;
}

int gg_max_mask_f32(const float* g, int64_t ldg, const int32_t* arg, int64_t ld_arg, int64_t num_rows, int64_t f,
                    float* out, int64_t ldo, gg_stream_t stream) {
    GG_REQUIRE(num_rows >= 0 && f >= 0, "gg_max_mask_f32: negative size");
    if (num_rows == 0 || f == 0) return GG_OK;
    GG_REQUIRE(g && arg && out, "gg_max_mask_f32: null pointer");
    GG_REQUIRE(ldg >= f && ld_arg >= f && ldo >= f && f < (1 << 30), "gg_max_mask_f32: bad leading dimension");
    max_mask_kernel<<<ea_elem_grid(num_rows * f), 256, 0, as_stream(stream)>>>(g, ldg, arg, ld_arg, num_rows, (int)f, out,
                                                                              ldo);
    GG_LAUNCHED();
    return GG_OK;
}

int gg_edge_max_sell_f32(const uint32_t* chunk_ptr, int64_t chunks, const int32_t* idx, const int32_t* slot_of,
                         const int32_t* perm, const int32_t* vdst, const int32_t* hub_rows, const int32_t* hub_pptr,
                         int64_t hubs, int64_t partial_rows, const float* h_j, int64_t ldj, const float* h_i, int64_t ldi,
                         const float* a, int64_t lda, int64_t kd, const float* w_a, int64_t ldw, float* out, int64_t ldo,
                         int32_t* arg, int64_t ld_arg, int64_t num_rows, int64_t f, const float* x_self, int64_t ld_self,
                         float self_scale, const float* bias, void* workspace, size_t workspace_bytes, int flags,
                         gg_stream_t stream) {
    GG_REQUIRE(num_rows >= 0 && f >= 0 && chunks >= 0 && hubs >= 0 && partial_rows >= 0 && kd >= 0,
               "gg_edge_max_sell_f32: negative size");
    if (num_rows == 0 || f == 0) return GG_OK;
    if (f % 4 != 0 || kd > kEaMaxKd) {
        set_error("gg_edge_max_sell_f32: needs f %% 4 == 0 and edge_dim <= %d (got f %lld, edge_dim %lld)", kEaMaxKd,
                  (long long)f, (long long)kd);
        return GG_ERR_UNSUPPORTED;
    }
    GG_REQUIRE(chunk_ptr && idx && slot_of && vdst && h_j && out && arg && workspace && (kd == 0 || w_a) &&
                   (hubs == 0 || (hub_rows && hub_pptr)),
               "gg_edge_max_sell_f32: null pointer");
    GG_REQUIRE(chunks < ((int64_t)1 << 31) && num_rows < ((int64_t)1 << 31), "gg_edge_max_sell_f32: sizes out of range");
    GG_REQUIRE(ldj >= f && ldj < ((int64_t)1 << 30) && ldo >= f && ld_arg >= f && ldj % 4 == 0 && ldo % 4 == 0 &&
                   ld_arg % 4 == 0 && lda >= kd && ldw >= kd && ea_al16(h_j) && ea_al16(out) && ea_al16(arg) &&
                   ea_al16(idx) && ea_al16(slot_of) && (!h_i || (ldi >= f && ldi % 4 == 0 && ea_al16(h_i))) &&
                   (!x_self || (ld_self >= f && ld_self % 4 == 0 && ea_al16(x_self))) && (!bias || ea_al16(bias)),
               "gg_edge_max_sell_f32: rows and unit arrays must be 16-byte aligned");
    if (workspace_bytes < gg_spmm_sell_max_workspace_bytes(partial_rows, f)) {
        set_error("gg_edge_max_sell_f32: workspace %zu < %zu", workspace_bytes,
                  gg_spmm_sell_max_workspace_bytes(partial_rows, f));
        return GG_ERR_WORKSPACE;
    }
    const int64_t tf0 = f < kEaTile ? f : kEaTile;
    const int64_t tiles = ceil_div(f, kEaTile);
    Carver cv(workspace);
    EdgeMaxArgs e{};
    int* counters = cv.take<int>(tiles);
    e.pval = cv.take<float>((size_t)partial_rows * tf0);
    e.pslot = cv.take<int32_t>((size_t)partial_rows * tf0);
    e.chunk_ptr = chunk_ptr; e.chunks = (int)chunks;
    e.idx4 = reinterpret_cast<const int4*>(idx); e.slot4 = reinterpret_cast<const int4*>(slot_of);
    e.perm = perm; e.vdst = vdst; e.hub_rows = hub_rows; e.hub_pptr = hub_pptr; e.hubs = (int)hubs;
    e.ldj = ldj; e.ldi = ldi; e.a = a; e.lda = lda; e.kd = (int)kd; e.ldw = ldw;
    e.ldo = ldo; e.ld_arg = ld_arg; e.ld_self = ld_self; e.self_scale = self_scale;
    e.l2_hint = (flags & 4) ? 1 : 0;
    cudaStream_t st = as_stream(stream);
    GG_CUDA(cudaMemsetAsync(counters, 0, (size_t)tiles * sizeof(int), st));
    for (int64_t t = 0; t < tiles; ++t) {
        const int64_t c0 = t * kEaTile;
        EdgeMaxArgs b = e;
        b.f = (int)(f - c0 < kEaTile ? f - c0 : kEaTile);
        b.counter = counters + t;
        b.hj = h_j + c0;
        b.hi = h_i ? h_i + c0 : nullptr;
        b.wa = w_a ? w_a + c0 * ldw : nullptr;
        b.out = out + c0;
        b.arg = arg + c0;
        b.x_self = x_self ? x_self + c0 : nullptr;
        b.bias = bias ? bias + c0 : nullptr;
        const int nvec = b.f / 4;
        int rc;
        if (nvec <= 4) rc = ea_launch_sell_tile<4>(b, st);
        else if (nvec <= 8) rc = ea_launch_sell_tile<8>(b, st);
        else if (nvec <= 16) rc = ea_launch_sell_tile<16>(b, st);
        else rc = ea_launch_sell_tile<32>(b, st);
        if (rc != GG_OK) return rc;
    }
    GG_CUDA(cudaPeekAtLastError());
    return GG_OK;
}

int gg_edge_max_row_f32(const int32_t* rowptr, const int32_t* nbr, const int32_t* perm, const float* h_j, int64_t ldj,
                        const float* h_i, int64_t ldi, const float* a, int64_t lda, int64_t kd, const float* w_a,
                        int64_t ldw, float* out, int64_t ldo, int32_t* arg, int64_t ld_arg, int64_t num_rows, int64_t f,
                        const float* x_self, int64_t ld_self, float self_scale, const float* bias, gg_stream_t stream) {
    GG_REQUIRE(num_rows >= 0 && f >= 0 && kd >= 0, "gg_edge_max_row_f32: negative size");
    if (num_rows == 0 || f == 0) return GG_OK;
    if (kd > kEaMaxKd) {
        set_error("gg_edge_max_row_f32: needs edge_dim <= %d (got %lld)", kEaMaxKd, (long long)kd);
        return GG_ERR_UNSUPPORTED;
    }
    // nbr / perm / a may be null for a layout without slots
    GG_REQUIRE(rowptr && h_j && out && arg && (kd == 0 || w_a), "gg_edge_max_row_f32: null pointer");
    GG_REQUIRE(ldj >= f && ldo >= f && ld_arg >= f && lda >= kd && ldw >= kd && (!h_i || ldi >= f) &&
                   (!x_self || ld_self >= f),
               "gg_edge_max_row_f32: leading dimension smaller than f");
    GG_REQUIRE(num_rows < ((int64_t)1 << 31) && f < (1 << 30), "gg_edge_max_row_f32: size out of range");
    const dim3 grid((unsigned)ea_row_grid(num_rows), (unsigned)ceil_div(f, 32));
    const size_t smem = (size_t)32 * (kd > 0 ? kd : 1) * sizeof(float);
    GG_CUDA(cudaFuncSetAttribute(edge_row_max_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    edge_row_max_kernel<<<grid, kEaThreads, smem, as_stream(stream)>>>(rowptr, nbr, perm, h_j, ldj, h_i, ldi, a, lda, (int)kd,
                                                                       w_a, ldw, out, ldo, arg, ld_arg, num_rows, (int)f,
                                                                       x_self, ld_self, self_scale, bias);
    GG_LAUNCHED();
    return GG_OK;
}

int gg_edge_max_winner_f32(const int32_t* rowptr, const int32_t* perm, const int32_t* arg, int64_t ld_arg, const float* g,
                           int64_t ldg, const float* w_a, int64_t ldw, int64_t num_rows, int64_t f, int64_t kd, float* da,
                           int64_t ldda, gg_stream_t stream) {
    GG_REQUIRE(num_rows >= 0 && f >= 0 && kd >= 0, "gg_edge_max_winner_f32: negative size");
    if (num_rows == 0 || kd == 0) return GG_OK;
    GG_REQUIRE(rowptr && arg && g && w_a, "gg_edge_max_winner_f32: null pointer");   // perm / da: null without slots
    GG_REQUIRE(ld_arg >= f && ldg >= f && ldw >= kd && ldda >= kd && f < (1 << 30) && kd < (1 << 30) &&
                   num_rows < ((int64_t)1 << 31),
               "gg_edge_max_winner_f32: bad leading dimension or size");
    edge_max_winner_kernel<<<ea_row_grid(num_rows), kEaThreads, 0, as_stream(stream)>>>(
        rowptr, perm, arg, ld_arg, g, ldg, w_a, ldw, num_rows, (int)f, (int)kd, da, ldda);
    GG_LAUNCHED();
    return GG_OK;
}

size_t gg_edge_max_wgrad_workspace_bytes(int64_t num_rows, int64_t f, int64_t kd) {
    if (num_rows <= 0 || f <= 0 || kd <= 0) return 256;
    int64_t blocks, rows;
    ea_wgrad_split(num_rows, f, kd, &blocks, &rows);
    return align_up((size_t)blocks * (size_t)f * (size_t)kd * sizeof(float), 256);
}

int gg_edge_max_wgrad_f32(const int32_t* perm, const int32_t* arg, int64_t ld_arg, const float* g, int64_t ldg,
                          const float* a, int64_t lda, int64_t num_rows, int64_t f, int64_t kd, float* dw, int64_t lddw,
                          void* workspace, size_t workspace_bytes, gg_stream_t stream) {
    GG_REQUIRE(num_rows >= 0 && f >= 0 && kd >= 0, "gg_edge_max_wgrad_f32: negative size");
    if (f == 0 || kd == 0) return GG_OK;
    GG_REQUIRE(dw && lddw >= kd, "gg_edge_max_wgrad_f32: bad output");
    cudaStream_t st = as_stream(stream);
    if (num_rows == 0) {
        GG_CUDA(cudaMemset2DAsync(dw, (size_t)lddw * sizeof(float), 0, (size_t)kd * sizeof(float), (size_t)f, st));
        return GG_OK;
    }
    GG_REQUIRE(arg && g && workspace, "gg_edge_max_wgrad_f32: null pointer");   // perm / a: null without slots
    GG_REQUIRE(ld_arg >= f && ldg >= f && lda >= kd && f * kd < ((int64_t)1 << 31) && num_rows < ((int64_t)1 << 31),
               "gg_edge_max_wgrad_f32: bad leading dimension or size");
    if (workspace_bytes < gg_edge_max_wgrad_workspace_bytes(num_rows, f, kd)) {
        set_error("gg_edge_max_wgrad_f32: workspace %zu < %zu", workspace_bytes,
                  gg_edge_max_wgrad_workspace_bytes(num_rows, f, kd));
        return GG_ERR_WORKSPACE;
    }
    int64_t blocks, rows;
    ea_wgrad_split(num_rows, f, kd, &blocks, &rows);
    float* part = static_cast<float*>(workspace);
    const dim3 grid((unsigned)blocks, (unsigned)ceil_div(f * kd, kEaWgradThreads));
    edge_max_wgrad_partial_kernel<<<grid, kEaWgradThreads, 0, st>>>(perm, arg, ld_arg, g, ldg, a, lda, num_rows, (int)f,
                                                                   (int)kd, rows, part);
    count_launch();
    edge_max_wgrad_reduce_kernel<<<ea_elem_grid(f * kd), 256, 0, st>>>(part, (int)blocks, (int)f, (int)kd, dw, lddw);
    GG_LAUNCHED();
    return GG_OK;
}

}  // extern "C"
