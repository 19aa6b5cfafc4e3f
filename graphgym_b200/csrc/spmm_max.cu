// Max aggregation (GraphGym cfg.gnn.agg = 'max'; PyG MessagePassing(aggr='max') = torch_scatter.scatter_max):
//   out[i,c] = max over the in-edges e = (j -> i) of m_e = w_e * x[j,c]      (0 for a row without in-edges)
//              + self_scale * x_self[i,c] + bias[c]
//   arg[i,c] = CSR slot of the FIRST in-edge that reaches the maximum (strict `>` in slot order; -1 for an empty row)
//   dx[j,c]  = sum over e = (j -> i) with arg[i,c] == slot(e) of w_e * g[i,c]  (+ self_scale * g[j,c])
// Ties go to the first edge in edge order, as in torch_scatter's CPU kernel (its CUDA kernel lets racing writes pick one):
// a CSR slot order is the stable order of the edited edge list, so "first edge" = "smallest slot".
//
// Two paths, selected where ops.spmm leaves the sliced-ELL path for the sum:
//   sliced ELL (f % 4 == 0, 16-byte rows): the layout of spmm_sell.cu.  A warp owns a chunk of 8 virtual rows, G lanes per
//     row, one float4 of columns per lane.  The forward keeps a running (max, slot) per column and reads the slot_of units
//     alongside the index units; padding entries (idx = -1) are skipped — a padding 0 would beat every negative maximum.
//     The backward walks the CSC layout: every entry carries the target i, the CSR slot of the same edge (composed map)
//     and the CSC-ordered weight, and gathers g[i] and arg[i] (16 bytes each) to add w * g where the arg names the edge.
//     Unlike spmm_sell_kernel, a group walks its chunk's rows one after the other with a single (max, slot) pair or sum:
//     interleaving the 8 rows would need 8 of them per lane (64 registers at G = 32) on top of the arg gathers.
//     Split rows write (value, slot) / sum partials; the fix-ups combine the pieces in order with the same strict `>` /
//     sum, so the result is bitwise that of one scan over the row, and apply the epilogue.  Widths above 128 run the same
//     kernels per column tile of <= 128 through the leading dimensions.
//   row (any f, any alignment; small graphs): one warp per row, lanes over the columns, slots in order; the backward walks
//     the CSC rows through the csc -> csr slot map.
// No atomics on data: every value is computed by one lane in a fixed order, so forward and backward are bitwise
// run-to-run deterministic.  NaN / inf inputs are not specified.
#include <math_constants.h>

#include "common.cuh"

namespace gg {

constexpr int kMaxRows = 8;        // virtual rows per chunk (= spmm_sell.cu)
constexpr int kMaxThreads = 256;
constexpr int kMaxTile = 128;      // columns per launch of the sliced-ELL kernels
constexpr int32_t kMaxNoRow = INT32_MIN;
constexpr int32_t kMaxHubBit = 1 << 30;   // gg_sell_hub_hint's marker bit (spmm_sell.cu)

struct MaxArgs {
    const uint32_t* chunk_ptr;
    int chunks;
    const int4* idx4;
    const int4* slot4;       // fwd: slot_of (CSR slot of every entry); bwd: CSR slot of the same edge (composed map)
    const float4* w4;        // nullable
    const int32_t* vdst;
    const int32_t* hub_rows;
    const int32_t* hub_pptr;
    int hubs;
    const float* x;          // fwd: gathered features; bwd: g
    int64_t ldx;
    const int32_t* arg_in;   // bwd: arg of the forward
    int64_t ld_arg_in;
    float* out;              // fwd: out; bwd: dx
    int64_t ldo;
    int32_t* arg;            // fwd
    int64_t ld_arg;
    int f;
    const float* x_self;     // nullable (bwd: g)
    int64_t ld_self;
    float self_scale;
    const float* bias;       // fwd, nullable
    float* pval;             // [partial rows, f]
    int32_t* pslot;          // fwd: [partial rows, f]
    int* counter;
    int l2_hint;
    int hub_hint;
};

__device__ __forceinline__ void max_take(float& m, int& s, float v, int slot, bool ok) {
    if (ok && v > m) {
        m = v;
        s = slot;
    }
}
__device__ __forceinline__ void max_take4(float4& m, int4& s, const float4& v, int slot, bool ok) {
    max_take(m.x, s.x, v.x, slot, ok);
    max_take(m.y, s.y, v.y, slot, ok);
    max_take(m.z, s.z, v.z, slot, ok);
    max_take(m.w, s.w, v.w, slot, ok);
}
__device__ __forceinline__ float4 mul4(float w, const float4& v) {
    return make_float4(w * v.x, w * v.y, w * v.z, w * v.w);
}
__device__ __forceinline__ int4 ldg_i4_pol(const int4* p, uint64_t pol) {
    int4 r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.s32 {%0,%1,%2,%3}, [%4], %5;"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p), "l"(pol));
    return r;
}

// out = (max, or 0 where no edge won) + self_scale * x_self + bias; arg = the winning slots
__device__ __forceinline__ void max_epilogue(const MaxArgs& a, int row, int gl, const float4& m, const int4& s,
                                             uint64_t pol) {
    float4 r = make_float4(s.x >= 0 ? m.x : 0.f, s.y >= 0 ? m.y : 0.f, s.z >= 0 ? m.z : 0.f, s.w >= 0 ? m.w : 0.f);
    if (a.x_self) fma4(r, a.self_scale, __ldg(reinterpret_cast<const float4*>(a.x_self + (int64_t)row * a.ld_self) + gl));
    if (a.bias) add4(r, __ldg(reinterpret_cast<const float4*>(a.bias) + gl));
    stg_f4_hint(reinterpret_cast<float4*>(a.out + (int64_t)row * a.ldo) + gl, r, pol);
    reinterpret_cast<int4*>(a.arg + (int64_t)row * a.ld_arg)[gl] = s;
}

__device__ __forceinline__ int max_next_chunk(const MaxArgs& a, int lane) {
    int c = 0;
    if (lane == 0) c = atomicAdd(a.counter, 1);
    return __shfl_sync(0xffffffffu, c, 0);
}

// ---- sliced ELL, forward -------------------------------------------------------------------------------------
template <int G, bool WEIGHTED>
__global__ void __launch_bounds__(kMaxThreads) spmm_sell_max_kernel(const __grid_constant__ MaxArgs a) {
    constexpr int S = 32 / G;              // rows per pass
    constexpr int P = kMaxRows / S;        // rows of the chunk per group
    const int lane = threadIdx.x & 31;
    const int grp = lane / G, gl = lane % G;
    const int nvec = a.f >> 2;
    const bool act = gl < nvec;
    // lanes past the row's last vector gather a duplicate of it and never store
    const char* __restrict__ xg = reinterpret_cast<const char*>(a.x) + (act ? gl : nvec - 1) * 16;
    const uint32_t row_bytes = (uint32_t)a.ldx * 4u;
    const uint64_t pol_keep = l2_policy(a.l2_hint ? 1 : 0), pol_stream = l2_policy(a.l2_hint ? 2 : 0);
    const bool hub_hint = a.hub_hint != 0;
    const float4 ninf4 = make_float4(-CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F);
    const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
    const int4 none4 = make_int4(-1, -1, -1, -1);
    auto gather = [&](int j) {
        float4 v = zero4;
        if (j >= 0) {
            const uint64_t pol = (hub_hint && !(j & kMaxHubBit)) ? pol_stream : pol_keep;
            v = ldg_nc_f4_hint(reinterpret_cast<const float4*>(xg + (uint64_t)(uint32_t)(j & ~kMaxHubBit) * row_bytes), pol);
        }
        return v;
    };

    int chunk = max_next_chunk(a, lane);
    while (chunk < a.chunks) {
        int next = 0;
        if (lane == 0) next = atomicAdd(a.counter, 1);   // in flight while this chunk is processed
        const uint32_t base = __ldg(a.chunk_ptr + chunk);
        const int nk = (int)(__ldg(a.chunk_ptr + chunk + 1) - base) / kMaxRows;   // 4-slot units per row
        // unit k4 of the group's p-th row (chunk row p * S + grp) is unit k4 * 8 + p * S + grp of the chunk
        const int4* __restrict__ ip = a.idx4 + base + grp;
        const int4* __restrict__ sp = a.slot4 + base + grp;
        const float4* __restrict__ wp = a.w4 + base + grp;
        int4 ia = nk > 0 ? ldg_i4_pol(ip, pol_stream) : none4;
        for (int p = 0; p < P; ++p) {
            float4 m = ninf4;
            int4 s = none4;
            for (int k4 = 0; k4 < nk; ++k4) {
                // the next unit's indices (this row's next one, else the next row's first) are requested first
                int4 na = none4;
                if (k4 + 1 < nk) na = ldg_i4_pol(ip + ((k4 + 1) * P + p) * S, pol_stream);
                else if (p + 1 < P) na = ldg_i4_pol(ip + (p + 1) * S, pol_stream);
                const int u = (k4 * P + p) * S;
                const int4 sa = ldg_i4_pol(sp + u, pol_stream);
                float4 v0 = gather(ia.x), v1 = gather(ia.y), v2 = gather(ia.z), v3 = gather(ia.w);
                if (WEIGHTED) {   // m_e = fl(w_e * x): one rounding, as the reference's message
                    const float4 wa = ldg_nc_f4_hint(wp + u, pol_stream);
                    v0 = mul4(wa.x, v0); v1 = mul4(wa.y, v1); v2 = mul4(wa.z, v2); v3 = mul4(wa.w, v3);
                }
                max_take4(m, s, v0, sa.x, ia.x >= 0);
                max_take4(m, s, v1, sa.y, ia.y >= 0);
                max_take4(m, s, v2, sa.z, ia.z >= 0);
                max_take4(m, s, v3, sa.w, ia.w >= 0);
                ia = na;
            }
            const int d = __ldg(a.vdst + (int64_t)chunk * kMaxRows + p * S + grp);
            if (act) {
                if (d >= 0) max_epilogue(a, d, gl, m, s, pol_stream);
                else if (d != kMaxNoRow) {
                    const int64_t o = (int64_t)(-d - 1) * a.f;
                    reinterpret_cast<float4*>(a.pval + o)[gl] = m;
                    reinterpret_cast<int4*>(a.pslot + o)[gl] = s;
                }
            }
        }
        chunk = __shfl_sync(0xffffffffu, next, 0);
    }
}

// split rows: the pieces' (max, slot) in piece order with the same strict `>`, then the epilogue; one thread per vector
__global__ void __launch_bounds__(256) spmm_sell_max_fixup_kernel(const __grid_constant__ MaxArgs a) {
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
            max_take(m.x, s.x, v.x, q.x, q.x >= 0);
            max_take(m.y, s.y, v.y, q.y, q.y >= 0);
            max_take(m.z, s.z, v.z, q.z, q.z >= 0);
            max_take(m.w, s.w, v.w, q.w, q.w >= 0);
        }
        max_epilogue(a, __ldg(a.hub_rows + h), gl, m, s, pol);
    }
}

// ---- sliced ELL, backward (CSC layout) -----------------------------------------------------------------------
__device__ __forceinline__ void max_bwd_store(const MaxArgs& a, int d, int gl, float4 r, uint64_t pol) {
    if (d >= 0) {
        if (a.x_self) fma4(r, a.self_scale, __ldg(reinterpret_cast<const float4*>(a.x_self + (int64_t)d * a.ld_self) + gl));
        stg_f4_hint(reinterpret_cast<float4*>(a.out + (int64_t)d * a.ldo) + gl, r, pol);
    } else if (d != kMaxNoRow) {
        reinterpret_cast<float4*>(a.pval + (int64_t)(-d - 1) * a.f)[gl] = r;
    }
}

template <int G, bool WEIGHTED>
__global__ void __launch_bounds__(kMaxThreads) spmm_sell_max_bwd_kernel(const __grid_constant__ MaxArgs a) {
    constexpr int S = 32 / G;
    constexpr int P = kMaxRows / S;
    const int lane = threadIdx.x & 31;
    const int grp = lane / G, gl = lane % G;
    const int nvec = a.f >> 2;
    const bool act = gl < nvec;
    const int vl = act ? gl : nvec - 1;
    const char* __restrict__ gp = reinterpret_cast<const char*>(a.x) + vl * 16;
    const char* __restrict__ ap = reinterpret_cast<const char*>(a.arg_in) + vl * 16;
    const uint64_t g_bytes = (uint64_t)a.ldx * 4u, a_bytes = (uint64_t)a.ld_arg_in * 4u;
    const uint64_t pol_keep = l2_policy(a.l2_hint ? 1 : 0), pol_stream = l2_policy(a.l2_hint ? 2 : 0);
    const int4 none4 = make_int4(-1, -1, -1, -1);
    // target i's g row and arg row (padding, i = -1: nothing gathered, an arg that matches no slot)
    auto gather = [&](int i, float4& gv, int4& av) {
        gv = make_float4(0.f, 0.f, 0.f, 0.f);
        av = make_int4(-2, -2, -2, -2);
        if (i >= 0) {
            gv = ldg_nc_f4_hint(reinterpret_cast<const float4*>(gp + (uint64_t)(uint32_t)i * g_bytes), pol_keep);
            av = ldg_i4_pol(reinterpret_cast<const int4*>(ap + (uint64_t)(uint32_t)i * a_bytes), pol_keep);
        }
    };
    // + w * g[i] in the columns whose arg is this entry's CSR slot e
    auto take = [&](float4& acc, const float4& gv, const int4& av, int e, float w) {
        if (WEIGHTED) {
            acc.x = av.x == e ? fmaf(w, gv.x, acc.x) : acc.x;
            acc.y = av.y == e ? fmaf(w, gv.y, acc.y) : acc.y;
            acc.z = av.z == e ? fmaf(w, gv.z, acc.z) : acc.z;
            acc.w = av.w == e ? fmaf(w, gv.w, acc.w) : acc.w;
        } else {
            acc.x = av.x == e ? acc.x + gv.x : acc.x;
            acc.y = av.y == e ? acc.y + gv.y : acc.y;
            acc.z = av.z == e ? acc.z + gv.z : acc.z;
            acc.w = av.w == e ? acc.w + gv.w : acc.w;
        }
    };

    int chunk = max_next_chunk(a, lane);
    while (chunk < a.chunks) {
        int next = 0;
        if (lane == 0) next = atomicAdd(a.counter, 1);
        const uint32_t base = __ldg(a.chunk_ptr + chunk);
        const int nk = (int)(__ldg(a.chunk_ptr + chunk + 1) - base) / kMaxRows;
        const int4* __restrict__ ip = a.idx4 + base + grp;
        const int4* __restrict__ sp = a.slot4 + base + grp;
        const float4* __restrict__ wp = a.w4 + base + grp;
        int4 ia = nk > 0 ? ldg_i4_pol(ip, pol_stream) : none4;
        for (int p = 0; p < P; ++p) {
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
            for (int k4 = 0; k4 < nk; ++k4) {
                int4 na = none4;
                if (k4 + 1 < nk) na = ldg_i4_pol(ip + ((k4 + 1) * P + p) * S, pol_stream);
                else if (p + 1 < P) na = ldg_i4_pol(ip + (p + 1) * S, pol_stream);
                const int u = (k4 * P + p) * S;
                const int4 sa = ldg_i4_pol(sp + u, pol_stream);
                float4 wa = make_float4(1.f, 1.f, 1.f, 1.f);
                if (WEIGHTED) wa = ldg_nc_f4_hint(wp + u, pol_stream);
                float4 g0, g1, g2, g3;
                int4 a0, a1, a2, a3;
                gather(ia.x, g0, a0); gather(ia.y, g1, a1); gather(ia.z, g2, a2); gather(ia.w, g3, a3);
                take(acc, g0, a0, sa.x, wa.x);
                take(acc, g1, a1, sa.y, wa.y);
                take(acc, g2, a2, sa.z, wa.z);
                take(acc, g3, a3, sa.w, wa.w);
                ia = na;
            }
            const int d = __ldg(a.vdst + (int64_t)chunk * kMaxRows + p * S + grp);
            if (act) max_bwd_store(a, d, gl, acc, pol_stream);
        }
        chunk = __shfl_sync(0xffffffffu, next, 0);
    }
}

// split rows: partial sums in piece order, then + self_scale * g[j]
__global__ void __launch_bounds__(256) spmm_sell_max_bwd_fixup_kernel(const __grid_constant__ MaxArgs a) {
    const int nvec = a.f >> 2;
    const int64_t total = (int64_t)a.hubs * nvec;
    const uint64_t pol = l2_policy(0);
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int h = (int)(e / nvec), gl = (int)(e - (int64_t)h * nvec);
        const int p0 = __ldg(a.hub_pptr + h), p1 = __ldg(a.hub_pptr + h + 1);
        float4 r = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int p = p0; p < p1; ++p) add4(r, reinterpret_cast<const float4*>(a.pval + (int64_t)p * a.f)[gl]);
        max_bwd_store(a, __ldg(a.hub_rows + h), gl, r, pol);
    }
}

static inline int max_grid(int64_t total, int per_block, int cap) {
    int64_t b = ceil_div(total, per_block);
    if (b > cap) b = cap;
    return (int)(b < 1 ? 1 : b);
}

template <int G>
static void launch_max_tile(const MaxArgs& a, bool bwd, cudaStream_t st) {
    const int grid = max_grid(a.chunks, kMaxThreads / 32, kNumSMs * 5);   // 40-64 registers: 5 blocks per SM
    if (bwd) {
        if (a.w4) spmm_sell_max_bwd_kernel<G, true><<<grid, kMaxThreads, 0, st>>>(a);
        else spmm_sell_max_bwd_kernel<G, false><<<grid, kMaxThreads, 0, st>>>(a);
    } else {
        if (a.w4) spmm_sell_max_kernel<G, true><<<grid, kMaxThreads, 0, st>>>(a);
        else spmm_sell_max_kernel<G, false><<<grid, kMaxThreads, 0, st>>>(a);
    }
    count_launch();
    if (a.hubs > 0) {
        const int g2 = max_grid((int64_t)a.hubs * (a.f >> 2), 256, kNumSMs * 8);
        if (bwd) spmm_sell_max_bwd_fixup_kernel<<<g2, 256, 0, st>>>(a);
        else spmm_sell_max_fixup_kernel<<<g2, 256, 0, st>>>(a);
        count_launch();
    }
}

// one launch (+ fix-up) per column tile of <= 128; `a` holds the whole-width pointers
static int launch_max_tiles(MaxArgs a, int64_t f, bool bwd, cudaStream_t st) {
    int* counters = a.counter;
    const int64_t tiles = ceil_div(f, kMaxTile);
    GG_CUDA(cudaMemsetAsync(counters, 0, (size_t)tiles * sizeof(int), st));
    for (int64_t t = 0; t < tiles; ++t) {
        const int64_t c0 = t * kMaxTile;
        const int tf = (int)(f - c0 < kMaxTile ? f - c0 : kMaxTile);
        MaxArgs b = a;
        b.f = tf;
        b.counter = counters + t;
        b.x = a.x + c0;
        b.out = a.out + c0;
        if (a.arg) b.arg = a.arg + c0;
        if (a.arg_in) b.arg_in = a.arg_in + c0;
        if (a.x_self) b.x_self = a.x_self + c0;
        if (a.bias) b.bias = a.bias + c0;
        const int nvec = tf / 4;
        if (nvec <= 4) launch_max_tile<4>(b, bwd, st);
        else if (nvec <= 8) launch_max_tile<8>(b, bwd, st);
        else if (nvec <= 16) launch_max_tile<16>(b, bwd, st);
        else launch_max_tile<32>(b, bwd, st);
    }
    GG_CUDA(cudaPeekAtLastError());
    return GG_OK;
}

// ---- row path (any f, any alignment) --------------------------------------------------------------------------
constexpr int kMaxRowWarps = 8;

template <bool WEIGHTED>
__global__ void __launch_bounds__(kMaxRowWarps * 32) spmm_row_max_kernel(
    const int32_t* __restrict__ rowptr, const int32_t* __restrict__ nbr, const float* __restrict__ w, const float* __restrict__ x,
    int64_t ldx, float* __restrict__ out, int64_t ldo, int32_t* __restrict__ arg, int64_t ld_arg, int64_t n, int f,
    const float* __restrict__ x_self, int64_t ld_self, float self_scale, const float* __restrict__ bias) {
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * kMaxRowWarps + (threadIdx.x >> 5);
    if (row >= n) return;
    const int beg = __ldg(rowptr + row), end = __ldg(rowptr + row + 1);
    for (int c = lane; c < f; c += 32) {
        float m = -CUDART_INF_F;
        int s = -1;
        for (int k = beg; k < end; ++k) {
            float v = __ldg(x + (int64_t)__ldg(nbr + k) * ldx + c);
            if (WEIGHTED) v = __ldg(w + k) * v;
            max_take(m, s, v, k, true);
        }
        float r = s >= 0 ? m : 0.f;
        if (x_self) r = fmaf(self_scale, __ldg(x_self + row * ld_self + c), r);
        if (bias) r += __ldg(bias + c);
        out[row * ldo + c] = r;
        arg[row * ld_arg + c] = s;
    }
}

template <bool WEIGHTED>
__global__ void __launch_bounds__(kMaxRowWarps * 32) spmm_row_max_bwd_kernel(
    const int32_t* __restrict__ rowptr, const int32_t* __restrict__ nbr, const int32_t* __restrict__ csc2csr,
    const float* __restrict__ w, const float* __restrict__ g, int64_t ldg, const int32_t* __restrict__ arg, int64_t ld_arg,
    int64_t n, int f, float self_scale, float* __restrict__ dx, int64_t ldd) {
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * kMaxRowWarps + (threadIdx.x >> 5);
    if (row >= n) return;
    const int beg = __ldg(rowptr + row), end = __ldg(rowptr + row + 1);
    for (int c = lane; c < f; c += 32) {
        float acc = 0.f;
        for (int k = beg; k < end; ++k) {
            const int64_t i = __ldg(nbr + k);
            if (__ldg(arg + i * ld_arg + c) == __ldg(csc2csr + k)) {
                const float gv = __ldg(g + i * ldg + c);
                acc = WEIGHTED ? fmaf(__ldg(w + k), gv, acc) : acc + gv;
            }
        }
        if (self_scale != 0.f) acc = fmaf(self_scale, __ldg(g + row * ldg + c), acc);
        dx[row * ldd + c] = acc;
    }
}

static inline bool max_al16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

}  // namespace gg

using namespace gg;

extern "C" {

size_t gg_spmm_sell_max_workspace_bytes(int64_t partial_rows, int64_t f) {
    const int64_t tf = f < kMaxTile ? f : kMaxTile;
    const int64_t tiles = f > 0 ? ceil_div(f, kMaxTile) : 1;
    const size_t part = align_up((size_t)(partial_rows > 0 ? partial_rows : 0) * (size_t)(tf > 0 ? tf : 0) * 4, 256);
    return 512 + align_up((size_t)tiles * sizeof(int), 256) + 2 * part;
}

int gg_spmm_sell_max_f32(const uint32_t* chunk_ptr, int64_t chunks, const int32_t* idx, const int32_t* slot_of,
                         const float* w_sell, const int32_t* vdst, const int32_t* hub_rows, const int32_t* hub_pptr,
                         int64_t hubs, int64_t partial_rows, const float* x, int64_t ldx, float* out, int64_t ldo,
                         int32_t* arg, int64_t ld_arg, int64_t num_rows, int64_t f, const float* x_self, int64_t ld_self,
                         float self_scale, const float* bias, void* workspace, size_t workspace_bytes, int flags,
                         gg_stream_t stream) {
    GG_REQUIRE(num_rows >= 0 && f >= 0 && chunks >= 0 && hubs >= 0 && partial_rows >= 0,
               "gg_spmm_sell_max_f32: negative size");
    if (num_rows == 0 || f == 0) return GG_OK;
    if (f % 4 != 0) {
        set_error("gg_spmm_sell_max_f32: needs f %% 4 == 0 (got %lld)", (long long)f);
        return GG_ERR_UNSUPPORTED;
    }
    GG_REQUIRE(chunk_ptr && idx && slot_of && vdst && x && out && arg && workspace && (hubs == 0 || (hub_rows && hub_pptr)),
               "gg_spmm_sell_max_f32: null pointer");
    GG_REQUIRE(chunks < ((int64_t)1 << 31) && num_rows < ((int64_t)1 << 31), "gg_spmm_sell_max_f32: sizes out of range");
    GG_REQUIRE(ldx >= f && ldx < ((int64_t)1 << 30) && ldo >= f && ld_arg >= f && ldx % 4 == 0 && ldo % 4 == 0 &&
                   ld_arg % 4 == 0 && max_al16(x) && max_al16(out) && max_al16(arg) && max_al16(idx) && max_al16(slot_of) &&
                   (!w_sell || max_al16(w_sell)) && (!x_self || (ld_self >= f && ld_self % 4 == 0 && max_al16(x_self))) &&
                   (!bias || max_al16(bias)),
               "gg_spmm_sell_max_f32: rows and unit arrays must be 16-byte aligned");
    if (workspace_bytes < gg_spmm_sell_max_workspace_bytes(partial_rows, f)) {
        set_error("gg_spmm_sell_max_f32: workspace %zu < %zu", workspace_bytes,
                  gg_spmm_sell_max_workspace_bytes(partial_rows, f));
        return GG_ERR_WORKSPACE;
    }
    const int64_t tf = f < kMaxTile ? f : kMaxTile;
    Carver c(workspace);
    MaxArgs a{};
    a.counter = c.take<int>(ceil_div(f, kMaxTile));
    a.pval = c.take<float>((size_t)partial_rows * tf);
    a.pslot = c.take<int32_t>((size_t)partial_rows * tf);
    a.chunk_ptr = chunk_ptr; a.chunks = (int)chunks;
    a.idx4 = reinterpret_cast<const int4*>(idx); a.slot4 = reinterpret_cast<const int4*>(slot_of);
    a.w4 = reinterpret_cast<const float4*>(w_sell);
    a.vdst = vdst; a.hub_rows = hub_rows; a.hub_pptr = hub_pptr; a.hubs = (int)hubs;
    a.x = x; a.ldx = ldx; a.out = out; a.ldo = ldo; a.arg = arg; a.ld_arg = ld_arg;
    a.x_self = x_self; a.ld_self = ld_self; a.self_scale = self_scale; a.bias = bias;
    a.l2_hint = (flags & 4) ? 1 : 0; a.hub_hint = (flags & 8) ? 1 : 0;
    return launch_max_tiles(a, f, false, as_stream(stream));
}

int gg_spmm_sell_max_bwd_f32(const uint32_t* chunk_ptr, int64_t chunks, const int32_t* idx, const int32_t* edge_map,
                             const float* w_sell, const int32_t* vdst, const int32_t* hub_rows, const int32_t* hub_pptr,
                             int64_t hubs, int64_t partial_rows, const float* g, int64_t ldg, const int32_t* arg,
                             int64_t ld_arg, int64_t num_rows, int64_t f, float self_scale, float* dx, int64_t ldd,
                             void* workspace, size_t workspace_bytes, int flags, gg_stream_t stream) {
    GG_REQUIRE(num_rows >= 0 && f >= 0 && chunks >= 0 && hubs >= 0 && partial_rows >= 0,
               "gg_spmm_sell_max_bwd_f32: negative size");
    if (num_rows == 0 || f == 0) return GG_OK;
    if (f % 4 != 0) {
        set_error("gg_spmm_sell_max_bwd_f32: needs f %% 4 == 0 (got %lld)", (long long)f);
        return GG_ERR_UNSUPPORTED;
    }
    GG_REQUIRE(chunk_ptr && idx && edge_map && vdst && g && arg && dx && workspace && (hubs == 0 || (hub_rows && hub_pptr)),
               "gg_spmm_sell_max_bwd_f32: null pointer");
    GG_REQUIRE(chunks < ((int64_t)1 << 31) && num_rows < ((int64_t)1 << 31), "gg_spmm_sell_max_bwd_f32: sizes out of range");
    GG_REQUIRE(ldg >= f && ld_arg >= f && ldd >= f && ldg % 4 == 0 && ld_arg % 4 == 0 && ldd % 4 == 0 && max_al16(g) &&
                   max_al16(arg) && max_al16(dx) && max_al16(idx) && max_al16(edge_map) && (!w_sell || max_al16(w_sell)),
               "gg_spmm_sell_max_bwd_f32: rows and unit arrays must be 16-byte aligned");
    if (workspace_bytes < gg_spmm_sell_max_workspace_bytes(partial_rows, f)) {
        set_error("gg_spmm_sell_max_bwd_f32: workspace %zu < %zu", workspace_bytes,
                  gg_spmm_sell_max_workspace_bytes(partial_rows, f));
        return GG_ERR_WORKSPACE;
    }
    const int64_t tf = f < kMaxTile ? f : kMaxTile;
    Carver c(workspace);
    MaxArgs a{};
    a.counter = c.take<int>(ceil_div(f, kMaxTile));
    a.pval = c.take<float>((size_t)partial_rows * tf);
    a.chunk_ptr = chunk_ptr; a.chunks = (int)chunks;
    a.idx4 = reinterpret_cast<const int4*>(idx); a.slot4 = reinterpret_cast<const int4*>(edge_map);
    a.w4 = reinterpret_cast<const float4*>(w_sell);
    a.vdst = vdst; a.hub_rows = hub_rows; a.hub_pptr = hub_pptr; a.hubs = (int)hubs;
    a.x = g; a.ldx = ldg; a.arg_in = arg; a.ld_arg_in = ld_arg; a.out = dx; a.ldo = ldd;
    a.x_self = self_scale != 0.f ? g : nullptr; a.ld_self = ldg; a.self_scale = self_scale;
    a.l2_hint = (flags & 4) ? 1 : 0;
    return launch_max_tiles(a, f, true, as_stream(stream));
}

int gg_spmm_row_max_f32(const int32_t* rowptr, const int32_t* nbr, const float* w_slot, const float* x, int64_t ldx,
                        float* out, int64_t ldo, int32_t* arg, int64_t ld_arg, int64_t num_rows, int64_t f,
                        const float* x_self, int64_t ld_self, float self_scale, const float* bias, gg_stream_t stream) {
    GG_REQUIRE(num_rows >= 0 && f >= 0, "gg_spmm_row_max_f32: negative size");
    if (num_rows == 0 || f == 0) return GG_OK;
    GG_REQUIRE(rowptr && x && out && arg, "gg_spmm_row_max_f32: null pointer");
    GG_REQUIRE(ldx >= f && ldo >= f && ld_arg >= f && (!x_self || ld_self >= f),
               "gg_spmm_row_max_f32: leading dimension smaller than f");
    GG_REQUIRE(num_rows < ((int64_t)1 << 31) && f < (1 << 30), "gg_spmm_row_max_f32: size out of range");
    const int grid = (int)ceil_div(num_rows, kMaxRowWarps);
    cudaStream_t st = as_stream(stream);
    if (w_slot)
        spmm_row_max_kernel<true><<<grid, kMaxRowWarps * 32, 0, st>>>(rowptr, nbr, w_slot, x, ldx, out, ldo, arg, ld_arg,
                                                                      num_rows, (int)f, x_self, ld_self, self_scale, bias);
    else
        spmm_row_max_kernel<false><<<grid, kMaxRowWarps * 32, 0, st>>>(rowptr, nbr, nullptr, x, ldx, out, ldo, arg, ld_arg,
                                                                       num_rows, (int)f, x_self, ld_self, self_scale, bias);
    GG_LAUNCHED();
    return GG_OK;
}

int gg_spmm_row_max_bwd_f32(const int32_t* rowptr, const int32_t* nbr, const int32_t* csc2csr, const float* w_slot,
                            const float* g, int64_t ldg, const int32_t* arg, int64_t ld_arg, int64_t num_rows, int64_t f,
                            float self_scale, float* dx, int64_t ldd, gg_stream_t stream) {
    GG_REQUIRE(num_rows >= 0 && f >= 0, "gg_spmm_row_max_bwd_f32: negative size");
    if (num_rows == 0 || f == 0) return GG_OK;
    GG_REQUIRE(rowptr && g && arg && dx, "gg_spmm_row_max_bwd_f32: null pointer");
    GG_REQUIRE(ldg >= f && ld_arg >= f && ldd >= f, "gg_spmm_row_max_bwd_f32: leading dimension smaller than f");
    GG_REQUIRE(num_rows < ((int64_t)1 << 31) && f < (1 << 30), "gg_spmm_row_max_bwd_f32: size out of range");
    const int grid = (int)ceil_div(num_rows, kMaxRowWarps);
    cudaStream_t st = as_stream(stream);
    if (w_slot)
        spmm_row_max_bwd_kernel<true><<<grid, kMaxRowWarps * 32, 0, st>>>(rowptr, nbr, csc2csr, w_slot, g, ldg, arg, ld_arg,
                                                                          num_rows, (int)f, self_scale, dx, ldd);
    else
        spmm_row_max_bwd_kernel<false><<<grid, kMaxRowWarps * 32, 0, st>>>(rowptr, nbr, csc2csr, nullptr, g, ldg, arg,
                                                                           ld_arg, num_rows, (int)f, self_scale, dx, ldd);
    GG_LAUNCHED();
    return GG_OK;
}

}  // extern "C"
