// B-spline weighted mean aggregation (splineconv; PyG 1.6 SplineConv with dim = 1, kernel_size = 2, degree = 1, open
// spline).  Edge e = (j -> i) carries a pseudo-coordinate u_e; torch_spline_conv's degree-1 basis with t = trunc(u),
// fr = u - floor(u) puts 1 - fr on kernel matrix t mod 2 and fr on (t + 1) mod 2 (non-negative mod), i.e. two coefficients
// (c0_e, c1_e) for W0 and W1.  The message c0 x_j W0 + c1 x_j W1 is linear in x, so no per-edge message is formed:
//   spread   out[i] = [sum_s w_s c0(u[perm[s]]) x[nbr[s]] | sum_s w_s c1(u[perm[s]]) x[nbr[s]]]   ([n, 2f] from [*, f]),
//            / indeg(i) with `mean`: aggregate-first order's [P0 | P1], transform-first order's [dH0 | dH1] on the CSC
//   blend    out[i] = sum_s w_s (c0 y[nbr[s], :f] + c1 y[nbr[s], f:]) (/ indeg(i)) + res[i] + bias   ([n, f] from [*, 2f]):
//            transform-first order's forward over H = [X W0 | X W1], aggregate-first order's dX over [dP0 | dP1] on the CSC
//   du       du[perm[s]] = (dc[(t+1) mod 2] - dc[t mod 2]) / indeg(i), dc_k = <a_k[i], b_k[nbr[s]]>: the pseudo-coordinate
//            gradient of torch_spline_conv's basis backward, one warp per CSR row, edge order output
// w_s: optional per-slot weight (the CSC's 1/indeg(target)).  Coefficients are formed per slot in registers from
// u[perm[slot]] (the slot_of units give the slot): no per-step re-lay and no E-sized coefficient array.
// Two paths for spread / blend, chosen as spmm_max's: sliced ELL (f % 4 == 0, 16-byte rows; the walk of spmm_sell_max_kernel
// with a sum per lane, split rows combined by a fix-up in piece order, column tiles of 128) and one warp per row (any f).
// No atomics on data: every kernel is bitwise run-to-run deterministic.
#include "common.cuh"

namespace gg {

constexpr int kSpRows = 8;          // virtual rows per sliced-ELL chunk (= spmm_sell.cu)
constexpr int kSpThreads = 256;
constexpr int kSpWarps = kSpThreads / 32;
constexpr int kSpTile = 128;        // columns per launch of the sliced-ELL kernels
constexpr int32_t kSpNoRow = INT32_MIN;

// (c0, c1) of pseudo-coordinate u: c[t & 1] = 1 - fr, c[(t & 1) ^ 1] = fr; `t & 1` is the non-negative t mod 2, which
// equals torch_spline_conv's index wherever that one is defined (u > -1).  1 - fr is formed as (floor(u) + 1) - u, one
// rounding of the exact value: 1 - (u - floor(u)) would round twice and lose the digits of a small -u for u in (-1, 0)
__device__ __forceinline__ float2 spline_coef(float u) {
    const float fl = floorf(u);
    const float fr = u - fl, om = (fl + 1.f) - u;
    return (__float2int_rz(u) & 1) ? make_float2(fr, om) : make_float2(om, fr);
}

struct SplineArgs {
    const uint32_t* chunk_ptr;
    int chunks;
    const int4* idx4;
    const int4* slot4;
    const float4* w4;        // nullable
    const int32_t* perm;
    const float* u;
    const int32_t* vdst;
    const int32_t* rowptr;   // the layout's rows: indeg for `mean`
    const int32_t* hub_rows;
    const int32_t* hub_pptr;
    int hubs;
    int mean;
    const float* x;          // gathered rows; blend: second half at x + half
    int64_t ldx;
    float* out;              // spread: second half at out + half
    int64_t ldo;
    int64_t half;
    int f;                   // columns of this tile
    const float* res;        // blend, nullable
    int64_t ld_res;
    const float* bias;       // blend, nullable
    float* pval0;            // [partial rows, f] per output half
    float* pval1;
    int* counter;
    int l2_hint;
};

__device__ __forceinline__ int4 sp_ldg_i4(const int4* p, uint64_t pol) {
    int4 r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.s32 {%0,%1,%2,%3}, [%4], %5;"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p), "l"(pol));
    return r;
}
__device__ __forceinline__ float4 scale4(const float4& v, float s) { return make_float4(v.x * s, v.y * s, v.z * s, v.w * s); }

__device__ __forceinline__ float sp_row_scale(const SplineArgs& a, int row) {
    if (!a.mean) return 1.f;
    const int deg = __ldg(a.rowptr + row + 1) - __ldg(a.rowptr + row);
    return deg > 0 ? 1.f / (float)deg : 1.f;
}

template <bool BLEND>
__device__ __forceinline__ void sp_epilogue(const SplineArgs& a, int row, int gl, float4 acc0, float4 acc1, uint64_t pol) {
    const float s = sp_row_scale(a, row);
    if (BLEND) {
        float4 r = scale4(acc0, s);
        if (a.res) add4(r, __ldg(reinterpret_cast<const float4*>(a.res + (int64_t)row * a.ld_res) + gl));
        if (a.bias) add4(r, __ldg(reinterpret_cast<const float4*>(a.bias) + gl));
        stg_f4_hint(reinterpret_cast<float4*>(a.out + (int64_t)row * a.ldo) + gl, r, pol);
    } else {
        stg_f4_hint(reinterpret_cast<float4*>(a.out + (int64_t)row * a.ldo) + gl, scale4(acc0, s), pol);
        stg_f4_hint(reinterpret_cast<float4*>(a.out + a.half + (int64_t)row * a.ldo) + gl, scale4(acc1, s), pol);
    }
}

// ---- sliced ELL ----------------------------------------------------------------------------------------------
// a warp per chunk of 8 virtual rows, G lanes per row, one float4 of columns per lane; a group walks its rows one after the
// other with one sum (blend) or two (spread) per lane
template <int G, bool BLEND, bool WEIGHTED>
__global__ void __launch_bounds__(kSpThreads) spline_sell_kernel(const __grid_constant__ SplineArgs a) {
    constexpr int S = 32 / G;
    constexpr int P = kSpRows / S;
    const int lane = threadIdx.x & 31;
    const int grp = lane / G, gl = lane % G;
    const int nvec = a.f >> 2;
    const bool act = gl < nvec;
    const char* __restrict__ xg = reinterpret_cast<const char*>(a.x) + (act ? gl : nvec - 1) * 16;
    const uint64_t row_bytes = (uint64_t)a.ldx * 4u, half_bytes = (uint64_t)a.half * 4u;
    const uint64_t pol_keep = l2_policy(a.l2_hint ? 1 : 0), pol_stream = l2_policy(a.l2_hint ? 2 : 0);
    const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
    const int4 none4 = make_int4(-1, -1, -1, -1);
    // entry (j, slot, w): spread acc0 += c0 w x_j, acc1 += c1 w x_j; blend acc0 += c0 w y_j[:f] + c1 w y_j[f:]
    auto take = [&](float4& acc0, float4& acc1, int j, int slot, float w) {
        if (j < 0) return;
        const char* r = xg + (uint64_t)(uint32_t)j * row_bytes;
        const float4 v0 = ldg_nc_f4_hint(reinterpret_cast<const float4*>(r), pol_keep);
        float4 v1 = zero4;
        if (BLEND) v1 = ldg_nc_f4_hint(reinterpret_cast<const float4*>(r + half_bytes), pol_keep);
        float2 c = spline_coef(__ldg(a.u + __ldg(a.perm + slot)));
        if (WEIGHTED) c = make_float2(c.x * w, c.y * w);
        if (BLEND) {
            fma4(acc0, c.x, v0);
            fma4(acc0, c.y, v1);
        } else {
            fma4(acc0, c.x, v0);
            fma4(acc1, c.y, v0);
        }
    };

    int chunk = 0;
    if (lane == 0) chunk = atomicAdd(a.counter, 1);
    chunk = __shfl_sync(0xffffffffu, chunk, 0);
    while (chunk < a.chunks) {
        int next = 0;
        if (lane == 0) next = atomicAdd(a.counter, 1);   // in flight while this chunk is processed
        const uint32_t base = __ldg(a.chunk_ptr + chunk);
        const int nk = (int)(__ldg(a.chunk_ptr + chunk + 1) - base) / kSpRows;
        const int4* __restrict__ ip = a.idx4 + base + grp;
        const int4* __restrict__ sp = a.slot4 + base + grp;
        const float4* __restrict__ wp = a.w4 + base + grp;
        int4 ia = nk > 0 ? sp_ldg_i4(ip, pol_stream) : none4;
        for (int p = 0; p < P; ++p) {
            float4 acc0 = zero4, acc1 = zero4;
            for (int k4 = 0; k4 < nk; ++k4) {
                int4 na = none4;
                if (k4 + 1 < nk) na = sp_ldg_i4(ip + ((k4 + 1) * P + p) * S, pol_stream);
                else if (p + 1 < P) na = sp_ldg_i4(ip + (p + 1) * S, pol_stream);
                const int u = (k4 * P + p) * S;
                const int4 sa = sp_ldg_i4(sp + u, pol_stream);
                float4 wa = make_float4(1.f, 1.f, 1.f, 1.f);
                if (WEIGHTED) wa = ldg_nc_f4_hint(wp + u, pol_stream);
                take(acc0, acc1, ia.x, sa.x, wa.x);
                take(acc0, acc1, ia.y, sa.y, wa.y);
                take(acc0, acc1, ia.z, sa.z, wa.z);
                take(acc0, acc1, ia.w, sa.w, wa.w);
                ia = na;
            }
            const int d = __ldg(a.vdst + (int64_t)chunk * kSpRows + p * S + grp);
            if (act) {
                if (d >= 0) sp_epilogue<BLEND>(a, d, gl, acc0, acc1, pol_stream);
                else if (d != kSpNoRow) {
                    const int64_t o = (int64_t)(-d - 1) * a.f;
                    reinterpret_cast<float4*>(a.pval0 + o)[gl] = acc0;
                    if (!BLEND) reinterpret_cast<float4*>(a.pval1 + o)[gl] = acc1;
                }
            }
        }
        chunk = __shfl_sync(0xffffffffu, next, 0);
    }
}

// split rows: the pieces' sums in piece order, then the epilogue; one thread per vector
template <bool BLEND>
__global__ void __launch_bounds__(256) spline_sell_fixup_kernel(const __grid_constant__ SplineArgs a) {
    const int nvec = a.f >> 2;
    const int64_t total = (int64_t)a.hubs * nvec;
    const uint64_t pol = l2_policy(0);
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int h = (int)(e / nvec), gl = (int)(e - (int64_t)h * nvec);
        const int p0 = __ldg(a.hub_pptr + h), p1 = __ldg(a.hub_pptr + h + 1);
        float4 r0 = make_float4(0.f, 0.f, 0.f, 0.f), r1 = r0;
        for (int p = p0; p < p1; ++p) add4(r0, reinterpret_cast<const float4*>(a.pval0 + (int64_t)p * a.f)[gl]);
        if (!BLEND)
            for (int p = p0; p < p1; ++p) add4(r1, reinterpret_cast<const float4*>(a.pval1 + (int64_t)p * a.f)[gl]);
        sp_epilogue<BLEND>(a, __ldg(a.hub_rows + h), gl, r0, r1, pol);
    }
}

static inline int sp_grid(int64_t total, int per_block, int cap) {
    int64_t b = ceil_div(total, per_block);
    if (b > cap) b = cap;
    return (int)(b < 1 ? 1 : b);
}

template <int G, bool BLEND>
static void sp_launch_tile(const SplineArgs& a, cudaStream_t st) {
    const int grid = sp_grid(a.chunks, kSpWarps, kNumSMs * 5);
    if (a.w4) spline_sell_kernel<G, BLEND, true><<<grid, kSpThreads, 0, st>>>(a);
    else spline_sell_kernel<G, BLEND, false><<<grid, kSpThreads, 0, st>>>(a);
    count_launch();
    if (a.hubs > 0) {
        spline_sell_fixup_kernel<BLEND><<<sp_grid((int64_t)a.hubs * (a.f >> 2), 256, kNumSMs * 8), 256, 0, st>>>(a);
        count_launch();
    }
}

// one launch (+ fix-up) per column tile of <= 128; `a` holds the whole-width pointers, `a.f` the whole width
template <bool BLEND>
static int sp_launch_tiles(SplineArgs a, cudaStream_t st) {
    const int64_t f = a.f;
    const int64_t tiles = ceil_div(f, kSpTile);
    GG_CUDA(cudaMemsetAsync(a.counter, 0, (size_t)tiles * sizeof(int), st));
    for (int64_t t = 0; t < tiles; ++t) {
        const int64_t c0 = t * kSpTile;
        SplineArgs b = a;
        b.f = (int)(f - c0 < kSpTile ? f - c0 : kSpTile);
        b.counter = a.counter + t;
        b.x = a.x + c0;
        b.out = a.out + c0;
        if (a.res) b.res = a.res + c0;
        if (a.bias) b.bias = a.bias + c0;
        const int nvec = b.f / 4;
        if (nvec <= 4) sp_launch_tile<4, BLEND>(b, st);
        else if (nvec <= 8) sp_launch_tile<8, BLEND>(b, st);
        else if (nvec <= 16) sp_launch_tile<16, BLEND>(b, st);
        else sp_launch_tile<32, BLEND>(b, st);
    }
    GG_CUDA(cudaPeekAtLastError());
    return GG_OK;
}

// ---- one warp per row (any f, any alignment) -----------------------------------------------------------------
template <bool BLEND>
__global__ void __launch_bounds__(kSpThreads) spline_row_kernel(
    const int32_t* __restrict__ rowptr, const int32_t* __restrict__ nbr, const int32_t* __restrict__ perm,
    const float* __restrict__ w, const float* __restrict__ u, const float* __restrict__ x, int64_t ldx, int64_t half,
    float* __restrict__ out, int64_t ldo, int64_t n, int f, int mean, const float* __restrict__ res, int64_t ld_res,
    const float* __restrict__ bias) {
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * kSpWarps + (threadIdx.x >> 5);
    if (row >= n) return;
    const int beg = __ldg(rowptr + row), end = __ldg(rowptr + row + 1);
    const float s = (mean && end > beg) ? 1.f / (float)(end - beg) : 1.f;
    for (int c = lane; c < f; c += 32) {
        float acc0 = 0.f, acc1 = 0.f;
        for (int k = beg; k < end; ++k) {
            const float* __restrict__ xr = x + (int64_t)__ldg(nbr + k) * ldx + c;
            float2 cf = spline_coef(__ldg(u + __ldg(perm + k)));
            if (w) {
                const float wk = __ldg(w + k);
                cf = make_float2(cf.x * wk, cf.y * wk);
            }
            const float v0 = __ldg(xr);
            if (BLEND) {
                acc0 = fmaf(cf.x, v0, acc0);
                acc0 = fmaf(cf.y, __ldg(xr + half), acc0);
            } else {
                acc0 = fmaf(cf.x, v0, acc0);
                acc1 = fmaf(cf.y, v0, acc1);
            }
        }
        if (BLEND) {
            float r = acc0 * s;
            if (res) r += __ldg(res + row * ld_res + c);
            if (bias) r += __ldg(bias + c);
            out[row * ldo + c] = r;
        } else {
            out[row * ldo + c] = acc0 * s;
            out[row * ldo + half + c] = acc1 * s;
        }
    }
}

// ---- pseudo-coordinate gradient ------------------------------------------------------------------------------
// one warp per CSR row i; per slot the lanes take the two dot products over the columns, a butterfly in a fixed order sums
// them, lane 0 writes the edge's du
__global__ void __launch_bounds__(kSpThreads) spline_du_kernel(
    const int32_t* __restrict__ rowptr, const int32_t* __restrict__ nbr, const int32_t* __restrict__ perm,
    const float* __restrict__ u, const float* __restrict__ a, int64_t lda, int64_t a_half, const float* __restrict__ b,
    int64_t ldb, int64_t b_half, int64_t n, int f, float* __restrict__ du) {
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * kSpWarps + (threadIdx.x >> 5);
    if (row >= n) return;
    const int beg = __ldg(rowptr + row), end = __ldg(rowptr + row + 1);
    if (end == beg) return;
    const float inv = 1.f / (float)(end - beg);
    const float* __restrict__ ar = a + row * lda;
    for (int k = beg; k < end; ++k) {
        const float* __restrict__ br = b + (int64_t)__ldg(nbr + k) * ldb;
        float p0 = 0.f, p1 = 0.f;
        for (int c = lane; c < f; c += 32) {
            p0 = fmaf(__ldg(ar + c), __ldg(br + c), p0);
            p1 = fmaf(__ldg(ar + a_half + c), __ldg(br + b_half + c), p1);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            p0 += __shfl_xor_sync(0xffffffffu, p0, o);
            p1 += __shfl_xor_sync(0xffffffffu, p1, o);
        }
        if (lane == 0) {
            const int64_t e = __ldg(perm + k);
            const float d = (__float2int_rz(__ldg(u + e)) & 1) ? p0 - p1 : p1 - p0;   // dc[(t+1) mod 2] - dc[t mod 2]
            du[e] = d * inv;
        }
    }
}

static inline bool sp_al16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

template <bool BLEND>
static int sp_sell(const char* name, const uint32_t* chunk_ptr, int64_t chunks, const int32_t* idx,
                   const int32_t* slot_of, const float* w_sell, const int32_t* perm, const float* u, const int32_t* vdst,
                   const int32_t* rowptr, const int32_t* hub_rows, const int32_t* hub_pptr, int64_t hubs,
                   int64_t partial_rows, const float* x, int64_t ldx, float* out, int64_t ldo, int64_t num_rows, int64_t f,
                   int mean, const float* res, int64_t ld_res, const float* bias, void* workspace, size_t workspace_bytes,
                   int flags, gg_stream_t stream) {
    GG_REQUIRE(num_rows >= 0 && f >= 0 && chunks >= 0 && hubs >= 0 && partial_rows >= 0, "%s: negative size", name);
    if (num_rows == 0 || f == 0) return GG_OK;
    if (f % 4 != 0) {
        set_error("%s: needs f %% 4 == 0 (got %lld)", name, (long long)f);
        return GG_ERR_UNSUPPORTED;
    }
    GG_REQUIRE(chunk_ptr && idx && slot_of && perm && u && vdst && rowptr && x && out && workspace &&
                   (hubs == 0 || (hub_rows && hub_pptr)),
               "%s: null pointer", name);
    GG_REQUIRE(chunks < ((int64_t)1 << 31) && num_rows < ((int64_t)1 << 31) && f < (1 << 29), "%s: sizes out of range",
               name);
    const int64_t xw = BLEND ? 2 * f : f, ow = BLEND ? f : 2 * f;
    GG_REQUIRE(ldx >= xw && ldo >= ow && ldx % 4 == 0 && ldo % 4 == 0 && sp_al16(x) && sp_al16(out) && sp_al16(idx) &&
                   sp_al16(slot_of) && (!w_sell || sp_al16(w_sell)) &&
                   (!res || (ld_res >= f && ld_res % 4 == 0 && sp_al16(res))) && (!bias || sp_al16(bias)),
               "%s: rows and unit arrays must be 16-byte aligned", name);
    if (workspace_bytes < gg_spmm_sell_max_workspace_bytes(partial_rows, f)) {
        set_error("%s: workspace %zu < %zu", name, workspace_bytes, gg_spmm_sell_max_workspace_bytes(partial_rows, f));
        return GG_ERR_WORKSPACE;
    }
    const int64_t tf = f < kSpTile ? f : kSpTile;
    Carver c(workspace);
    SplineArgs a{};
    a.counter = c.take<int>(ceil_div(f, kSpTile));
    a.pval0 = c.take<float>((size_t)partial_rows * tf);
    a.pval1 = c.take<float>((size_t)partial_rows * tf);
    a.chunk_ptr = chunk_ptr; a.chunks = (int)chunks;
    a.idx4 = reinterpret_cast<const int4*>(idx); a.slot4 = reinterpret_cast<const int4*>(slot_of);
    a.w4 = reinterpret_cast<const float4*>(w_sell);
    a.perm = perm; a.u = u; a.vdst = vdst; a.rowptr = rowptr;
    a.hub_rows = hub_rows; a.hub_pptr = hub_pptr; a.hubs = (int)hubs; a.mean = mean;
    a.x = x; a.ldx = ldx; a.out = out; a.ldo = ldo; a.half = f; a.f = (int)f;
    a.res = res; a.ld_res = ld_res; a.bias = bias;
    a.l2_hint = (flags & 4) ? 1 : 0;
    return sp_launch_tiles<BLEND>(a, as_stream(stream));
}

template <bool BLEND>
static int sp_row(const char* name, const int32_t* rowptr, const int32_t* nbr, const int32_t* perm, const float* w_slot,
                  const float* u, const float* x, int64_t ldx, float* out, int64_t ldo, int64_t num_rows, int64_t f,
                  int mean, const float* res, int64_t ld_res, const float* bias, gg_stream_t stream) {
    GG_REQUIRE(num_rows >= 0 && f >= 0, "%s: negative size", name);
    if (num_rows == 0 || f == 0) return GG_OK;
    GG_REQUIRE(rowptr && x && out, "%s: null pointer", name);   // nbr / perm / u: null for a layout without slots
    const int64_t xw = BLEND ? 2 * f : f, ow = BLEND ? f : 2 * f;
    GG_REQUIRE(ldx >= xw && ldo >= ow && (!res || ld_res >= f), "%s: leading dimension too small", name);
    GG_REQUIRE(num_rows < ((int64_t)1 << 31) && f < (1 << 29), "%s: size out of range", name);
    spline_row_kernel<BLEND><<<(int)ceil_div(num_rows, kSpWarps), kSpThreads, 0, as_stream(stream)>>>(
        rowptr, nbr, perm, w_slot, u, x, ldx, f, out, ldo, num_rows, (int)f, mean, res, ld_res, bias);
    GG_LAUNCHED();
    return GG_OK;
}

}  // namespace gg

using namespace gg;

extern "C" {

int gg_spline_spread_sell_f32(const uint32_t* chunk_ptr, int64_t chunks, const int32_t* idx, const int32_t* slot_of,
                              const float* w_sell, const int32_t* perm, const float* u, const int32_t* vdst,
                              const int32_t* rowptr, const int32_t* hub_rows, const int32_t* hub_pptr, int64_t hubs,
                              int64_t partial_rows, const float* x, int64_t ldx, float* out, int64_t ldo, int64_t num_rows,
                              int64_t f, int mean, void* workspace, size_t workspace_bytes, int flags, gg_stream_t stream) {
    return sp_sell<false>("gg_spline_spread_sell_f32", chunk_ptr, chunks, idx, slot_of, w_sell, perm, u, vdst, rowptr,
                          hub_rows, hub_pptr, hubs, partial_rows, x, ldx, out, ldo, num_rows, f, mean, nullptr, 0, nullptr,
                          workspace, workspace_bytes, flags, stream);
}

int gg_spline_blend_sell_f32(const uint32_t* chunk_ptr, int64_t chunks, const int32_t* idx, const int32_t* slot_of,
                             const float* w_sell, const int32_t* perm, const float* u, const int32_t* vdst,
                             const int32_t* rowptr, const int32_t* hub_rows, const int32_t* hub_pptr, int64_t hubs,
                             int64_t partial_rows, const float* y, int64_t ldy, float* out, int64_t ldo, int64_t num_rows,
                             int64_t f, int mean, const float* res, int64_t ld_res, const float* bias, void* workspace,
                             size_t workspace_bytes, int flags, gg_stream_t stream) {
    return sp_sell<true>("gg_spline_blend_sell_f32", chunk_ptr, chunks, idx, slot_of, w_sell, perm, u, vdst, rowptr,
                         hub_rows, hub_pptr, hubs, partial_rows, y, ldy, out, ldo, num_rows, f, mean, res, ld_res, bias,
                         workspace, workspace_bytes, flags, stream);
}

int gg_spline_spread_row_f32(const int32_t* rowptr, const int32_t* nbr, const int32_t* perm, const float* w_slot,
                             const float* u, const float* x, int64_t ldx, float* out, int64_t ldo, int64_t num_rows,
                             int64_t f, int mean, gg_stream_t stream) {
    return sp_row<false>("gg_spline_spread_row_f32", rowptr, nbr, perm, w_slot, u, x, ldx, out, ldo, num_rows, f, mean,
                         nullptr, 0, nullptr, stream);
}

int gg_spline_blend_row_f32(const int32_t* rowptr, const int32_t* nbr, const int32_t* perm, const float* w_slot,
                            const float* u, const float* y, int64_t ldy, float* out, int64_t ldo, int64_t num_rows,
                            int64_t f, int mean, const float* res, int64_t ld_res, const float* bias, gg_stream_t stream) {
    return sp_row<true>("gg_spline_blend_row_f32", rowptr, nbr, perm, w_slot, u, y, ldy, out, ldo, num_rows, f, mean, res,
                        ld_res, bias, stream);
}

int gg_spline_du_f32(const int32_t* rowptr, const int32_t* nbr, const int32_t* perm, const float* u, const float* a,
                     int64_t lda, int64_t a_half, const float* b, int64_t ldb, int64_t b_half, int64_t num_rows, int64_t f,
                     float* du, gg_stream_t stream) {
    GG_REQUIRE(num_rows >= 0 && f >= 0 && a_half >= 0 && b_half >= 0, "gg_spline_du_f32: negative size");
    if (num_rows == 0) return GG_OK;
    GG_REQUIRE(rowptr && a && b, "gg_spline_du_f32: null pointer");   // nbr / perm / u / du: null without slots
    GG_REQUIRE(lda >= a_half + f && ldb >= b_half + f && num_rows < ((int64_t)1 << 31) && f < (1 << 30),
               "gg_spline_du_f32: bad leading dimension or size");
    spline_du_kernel<<<(int)ceil_div(num_rows, kSpWarps), kSpThreads, 0, as_stream(stream)>>>(
        rowptr, nbr, perm, u, a, lda, a_half, b, ldb, b_half, num_rows, (int)f, du);
    GG_LAUNCHED();
    return GG_OK;
}

}  // extern "C"
