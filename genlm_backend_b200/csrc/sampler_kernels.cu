// Fused SMC row op for sm_100a: masked logsumexp + one categorical draw per row, one HBM pass.
//
// Replaces the per-particle torch sequence of the reference idiom (README.md:82-91, docs/index.md:61-70;
// temperature variant genlm/backend/llm/base.py:131-146):
//     masked = logp + mask;  logZ = masked.logsumexp(-1);  tok = multinomial((masked - logZ).exp(), 1)
//
// One CTA of kSThreads = 256 threads per row, four rows in flight per SM.  Thread t owns the 16-byte groups
// g = t, t + kSThreads, ... of the row and keeps an online (max, sum-exp) pair for them; after a block reduction
// (fp64) a Philox uniform picks first the owning thread, then the element among that thread's ~V/kSThreads
// elements, which are re-read from L2 (a few KB).
// The draw is an exact inverse CDF over a fixed permutation of the vocabulary, so it is distributed as
// the reference's multinomial but is not stream-identical to torch's generator.
#include <cstdint>
#include <type_traits>

#include "trie_device.cuh"
#include "philox.cuh"

namespace gt {

#ifndef GT_SAMPLER_THREADS
#define GT_SAMPLER_THREADS 256
#endif
// Threads per row; 1024 / kSThreads rows are in flight per SM.  256 (4 rows per SM) measured 12 % faster than 512 on
// B200 at 512 rows x 128k: all rows of a launch start in one wave and the block-wide tail of a row (reduction, draw,
// second pass) overlaps three other rows' streaming instead of one.
constexpr int kSThreads = GT_SAMPLER_THREADS;
constexpr float kLog2e = 1.4426950408889634f;

// 2^x for x <= 0 (flush-to-zero below 2^-126: such terms vanish against the row maximum anyway): one MUFU, without
// the range scaling of exp2f()
__device__ __forceinline__ float fast_exp2(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

struct SampleArgs {
    const void* logp; int64_t ld_logp; int64_t V; int n_rows;
    const void* mask; int mask_kind; int64_t mask_ld;
    float inv_temp; uint64_t seed, offset;
    float* logZ; int32_t* tok;
};

// Per-row view: groups of EPV elements aligned to 16 bytes in global memory.
//
// Values are handled in "working units" that cost the fewest instructions per element: with an additive mask
// y = logp * inv_temp + mask (one FFMA) and exponentials are 2^(y * log2e - ...); otherwise y is the raw log-prob
// (masked-out elements replaced by -inf) and the temperature is folded into the exponent scale SC = inv_temp * log2e,
// which is legal because inv_temp > 0 preserves the maximum.  unit() converts a working-unit value back to
// temperature-scaled natural-log units.
template <typename IN_T, int MK> struct RowView {
    static constexpr int EPV = 16 / (int)sizeof(IN_T);
    const IN_T* row;        // first element of the row
    int phase;              // element offset of `row` inside its 16-byte line
    int V;
    const void* mrow; bool mask_vec;
    static constexpr int mask_kind = MK;  // compile-time: no per-element dispatch
    float inv_temp;

    __device__ __forceinline__ int n_groups() const { return (phase + V + EPV - 1) / EPV; }
    __device__ __forceinline__ float scale() const { return MK == GT_MASK_ADD_F32 ? kLog2e : inv_temp * kLog2e; }
    __device__ __forceinline__ float unit() const { return MK == GT_MASK_ADD_F32 ? 1.f : inv_temp; }

    // working-unit value of element i (scalar path: edge groups and masks that do not line up with the row's groups)
    __device__ __forceinline__ float mask_apply(float e, int i) const {
        if constexpr (MK == GT_MASK_ADD_F32) return fmaf(e, inv_temp, __ldg(static_cast<const float*>(mrow) + i));
        else if constexpr (MK == GT_MASK_BOOL_U8) return __ldg(static_cast<const uint8_t*>(mrow) + i) ? e : -INFINITY;
        else if constexpr (MK == GT_MASK_BITS_U32) return (__ldg(static_cast<const uint32_t*>(mrow) + (i >> 5)) >> (i & 31)) & 1u ? e : -INFINITY;
        else return e;
    }

    // A group is "interior" when all of its EPV elements lie inside the row: then it is one aligned 16-byte load.
    __device__ __forceinline__ bool interior(int g) const {
        const int i0 = g * EPV - phase;
        return i0 >= 0 && i0 + EPV <= V;
    }
    // What is requested ahead of its use for one interior group: the 16 bytes of the row and the group's share of the
    // mask -- 16/32 bytes of an additive mask, EPV bytes of a byte mask, one or two words of a bit mask.  issue() only
    // requests: nothing here may consume a loaded value, or the requests of a round would serialise on each other.
    // A Cursor holds the addresses of one interior group; the groups a thread visits are a fixed number of groups
    // apart, so the loads of a round are the cursor plus compile-time offsets and advancing is a few pointer adds.
    struct Raw { uint4 v; uint4 ma, mb; uint32_t m0, m1; };
    struct Cursor {
        const IN_T* p; const unsigned char* mp;
        int i0;      // element index of the group's first element
        int sh;      // bit mask: position of that element's bit in its word (the same for every group of a thread)
        bool strad;  // bit mask: the group's bits continue in the next word (unaligned rows only)
    };
    __device__ __forceinline__ Cursor cursor(int g) const {
        Cursor c;
        c.i0 = g * EPV - phase;
        c.p = row + c.i0;
        c.sh = c.i0 & 31; c.strad = c.sh + EPV > 32;
        if (MK == GT_MASK_ADD_F32) c.mp = reinterpret_cast<const unsigned char*>(static_cast<const float*>(mrow) + c.i0);
        else if (MK == GT_MASK_BOOL_U8) c.mp = static_cast<const unsigned char*>(mrow) + c.i0;
        else if (MK == GT_MASK_BITS_U32) c.mp = reinterpret_cast<const unsigned char*>(static_cast<const uint32_t*>(mrow) + (c.i0 >> 5));
        else c.mp = nullptr;
        return c;
    }
    // dg groups further on (dg * EPV is a multiple of 32 wherever this is used with a bit mask)
    __device__ __forceinline__ void advance(Cursor& c, int dg) const {
        const int de = dg * EPV;
        c.i0 += de; c.p += de;
        if (MK == GT_MASK_ADD_F32) c.mp += (size_t)de * 4;
        else if (MK == GT_MASK_BOOL_U8) c.mp += de;
        else if (MK == GT_MASK_BITS_U32) c.mp += de >> 3;
    }
    // the group dg groups after the cursor
    template <bool VEC> __device__ __forceinline__ Raw issue(const Cursor& c, int dg) const {
        Raw r;
        const int de = dg * EPV;
        asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                     : "=r"(r.v.x), "=r"(r.v.y), "=r"(r.v.z), "=r"(r.v.w) : "l"(c.p + de));
        r.m0 = r.m1 = 0;
        r.ma = r.mb = make_uint4(0, 0, 0, 0);
        if (MK == GT_MASK_ADD_F32 && VEC) {
            const uint4* m4 = reinterpret_cast<const uint4*>(c.mp + (size_t)de * 4);
            r.ma = __ldg(m4);
            if constexpr (EPV >= 8) r.mb = __ldg(m4 + 1);
        } else if (MK == GT_MASK_BOOL_U8 && VEC) {
            const unsigned char* mp = c.mp + de;
            if constexpr (EPV <= 4) {
                r.m0 = __ldg(reinterpret_cast<const uint32_t*>(mp));
            } else {
                const uint2 t = __ldg(reinterpret_cast<const uint2*>(mp));
                r.m0 = t.x; r.m1 = t.y;
            }
        } else if (MK == GT_MASK_BITS_U32) {
            // the word that holds the group's first bit and, when the group straddles, the next one (which exists:
            // the group is interior)
            const uint32_t* mw = reinterpret_cast<const uint32_t*>(c.mp + (de >> 3));
            r.m0 = __ldg(mw);
            if (c.strad) r.m1 = __ldg(mw + 1);
        }
        return r;
    }
    // y[k] = working-unit value of element k of the group dg groups after the cursor, from an issued load
    template <bool VEC> __device__ __forceinline__ void finish(const Cursor& c, int dg, const Raw& raw, float y[EPV]) const {
        const IN_T* e = reinterpret_cast<const IN_T*>(&raw.v);
#pragma unroll
        for (int k = 0; k < EPV; ++k) y[k] = in_to_float<IN_T>(e[k]);
        if (MK == GT_MASK_ADD_F32 && VEC) {
            const float* ma = reinterpret_cast<const float*>(&raw.ma);
            const float* mb = reinterpret_cast<const float*>(&raw.mb);
#pragma unroll
            for (int k = 0; k < EPV; ++k) y[k] = fmaf(y[k], inv_temp, k < 4 ? ma[k & 3] : mb[k & 3]);
        } else if (MK == GT_MASK_BOOL_U8 && VEC) {
#pragma unroll
            for (int k = 0; k < EPV; ++k) y[k] = ((k < 4 ? raw.m0 : raw.m1) & (0xFFu << (8 * (k & 3)))) ? y[k] : -INFINITY;
        } else if (MK == GT_MASK_BITS_U32) {
            const uint32_t bits = __funnelshift_r(raw.m0, raw.m1, c.sh);  // m1 = 0 when the group does not straddle
#pragma unroll
            for (int k = 0; k < EPV; ++k) y[k] = (bits & (1u << k)) ? y[k] : -INFINITY;
        } else if (MK != GT_MASK_NONE) {
            const int i0 = c.i0 + dg * EPV;
#pragma unroll
            for (int k = 0; k < EPV; ++k) y[k] = mask_apply(y[k], i0 + k);
        }
    }
    // edge groups (first / last of an unaligned row): element-wise, -inf outside the row
    __device__ __forceinline__ void fetch_edge(int g, float y[EPV]) const {
        const int i0 = g * EPV - phase;
#pragma unroll
        for (int k = 0; k < EPV; ++k) {
            const int i = i0 + k;
            y[k] = (i >= 0 && i < V) ? mask_apply(in_to_float<IN_T>(row[i]), i) : -INFINITY;
        }
    }
    __device__ __forceinline__ void fetch(int g, float y[EPV]) const {
        if (interior(g)) {
            const Cursor c = cursor(g);
            if (mask_vec) finish<true>(c, 0, issue<true>(c, 0), y);
            else finish<false>(c, 0, issue<false>(c, 0), y);
        }
        else fetch_edge(g, y);
    }
};

// max that returns NaN when either operand is NaN (fmaxf would drop it)
__device__ __forceinline__ float fmax_nan(float a, float b) {
    float r;
    asm("max.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
    return r;
}

// Online (max, sum of 2^((y - max) * SC)) update with N more values.  A NaN among them makes s NaN for good, also while
// the running max is still -inf (a NaN logit at an allowed position of an otherwise masked stretch): torch's logsumexp
// gives NaN for such a row and multinomial raises.
template <int N> __device__ __forceinline__ void online_update(const float (&y)[N], float SC, float& m, float& s) {
    float gm = y[0];
#pragma unroll
    for (int k = 1; k < N; ++k) gm = fmax_nan(gm, y[k]);
    if (!(gm <= m)) {  // a larger value (rare once the running max has settled) or a NaN
        s *= fast_exp2((m - gm) * SC);  // m = -inf: s is still 0; gm = NaN: s becomes NaN
        m = gm;
    }
    if (m > -INFINITY) {
        const float ms = -m * SC;
        float t[N];
#pragma unroll
        for (int k = 0; k < N; ++k) t[k] = fast_exp2(fmaf(y[k], SC, ms));
#pragma unroll
        for (int w = 1; w < N; w <<= 1)  // pairwise: a short dependency chain
#pragma unroll
            for (int k = 0; k + w < N; k += 2 * w) t[k] += t[k + w];
        s += t[0];
    }
}

// Warp-wide search over arr[0..n) (shared memory).  target >= 0: first index whose inclusive prefix sum
// exceeds target.  target < 0, or rounding pushed target past the total: the last index with positive
// mass, flagged by before = -1.  idx = -1 only when nothing has mass.
__device__ __forceinline__ void warp_find(const double* arr, int n, double target, int& idx, double& before) {
    const int lane = threadIdx.x & 31;
    const int per = (n + 31) / 32;
    const int a = min(n, lane * per), b = min(n, a + per);
    double local = 0.0;
    int last_pos = -1;
    for (int i = a; i < b; ++i) { const double v = arr[i]; local += v; if (v > 0.0) last_pos = i; }
    double incl = local;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const double y = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += y;
    }
    const unsigned hit = __ballot_sync(0xffffffffu, target >= 0.0 && incl > target && last_pos >= 0);
    if (hit) {
        const int src = __ffs(hit) - 1;
        int found = -1; double bef = 0.0;
        if (lane == src) {
            double run = incl - local;
            for (int i = a; i < b; ++i) {
                const double v = arr[i];
                if (v > 0.0) { found = i; bef = run; if (run + v > target) break; }
                run += v;
            }
        }
        idx = __shfl_sync(0xffffffffu, found, src);
        before = __shfl_sync(0xffffffffu, bef, src);
    } else {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) last_pos = max(last_pos, __shfl_xor_sync(0xffffffffu, last_pos, o));
        idx = last_pos; before = -1.0;
    }
}

// Second pass of a row, executed by the whole CTA once per row: the picked thread owned groups pick, pick + NT, ...;
// candidate c of them goes to thread c % NT (one candidate per thread unless the row has more than NT^2 groups),
// a second inverse-CDF step picks the thread and it walks its candidates' elements.  (Measured both ways: inlined is
// 1-5 % faster for fp32 rows than a __noinline__ call, which spills the row view to the stack.)
template <typename IN_T, int MK, int NT>
__device__ __forceinline__ void locate_token(const RowView<IN_T, MK>& rv, int pick, double resid, float M, float SC, int ng,
                                          double* s_mass, int* s_pick, double* s_resid, int32_t* tok_out) {
    constexpr int EPV = RowView<IN_T, MK>::EPV;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int n_cand = (ng - pick + NT - 1) / NT;
    const float ms2 = -M * SC;
    double local = 0.0;
    for (int c = tid; c < n_cand; c += NT) {
        float x[EPV];
        rv.fetch(pick + c * NT, x);
#pragma unroll
        for (int k = 0; k < EPV; ++k) local += (double)fast_exp2(fmaf(x[k], SC, ms2));
    }
    s_mass[tid] = local;
    __syncthreads();
    if (warp == 0) {
        int k2; double before2;
        warp_find(s_mass, min(n_cand, NT), resid, k2, before2);
        if (lane == 0) { *s_pick = k2; *s_resid = (before2 < 0.0) ? -1.0 : resid - before2; }
    }
    __syncthreads();
    const int k2 = *s_pick;
    if (k2 < 0) {  // exp underflow relative to the global max wiped the picked thread's mass
        if (tid == 0) *tok_out = -1;
    } else if (tid == k2) {
        const double rr = *s_resid;
        int chosen = -1; double run = 0.0;
        for (int c = k2; c < n_cand; c += NT) {
            const int g = pick + c * NT;
            float x[EPV];
            rv.fetch(g, x);
#pragma unroll
            for (int k = 0; k < EPV; ++k) {
                const float w = fast_exp2(fmaf(x[k], SC, ms2));
                if (w > 0.f) {
                    // the first positive element always qualifies; later ones while the running sum has not
                    // passed the residual (rr < 0: keep going to the last positive element)
                    if (chosen < 0 || rr < 0.0 || run <= rr) chosen = g * EPV - rv.phase + k;
                    run += (double)w;
                }
            }
        }
        *tok_out = chosen;
    }
}

template <typename IN_T, int MK, int NT>
__global__ void __launch_bounds__(NT, 1024 / NT) lse_sample_kernel(SampleArgs A) {
    constexpr int EPV = RowView<IN_T, MK>::EPV;
    __shared__ double s_mass[NT];
    __shared__ float s_wmax[NT / 32];
    __shared__ float s_M;
    __shared__ int s_pick;
    __shared__ double s_resid;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int b = blockIdx.x; b < A.n_rows; b += gridDim.x) {
        RowView<IN_T, MK> rv;
        rv.row = static_cast<const IN_T*>(A.logp) + (size_t)b * A.ld_logp;
        rv.phase = (int)((reinterpret_cast<uintptr_t>(rv.row) & 15) / sizeof(IN_T));
        rv.V = (int)A.V; rv.inv_temp = A.inv_temp;
        rv.mrow = nullptr; rv.mask_vec = false;
        if (MK == GT_MASK_ADD_F32) {
            const float* m = static_cast<const float*>(A.mask) + (size_t)b * A.mask_ld;
            rv.mrow = m;
            // group g starts at element g*EPV - phase: its mask address is 16-byte aligned iff the mask row
            // has the same phase (mod 4 floats) as the group grid
            rv.mask_vec = EPV >= 4 && ((((reinterpret_cast<uintptr_t>(m) >> 2) + 4u - (unsigned)(rv.phase & 3)) & 3u) == 0);
        } else if (MK == GT_MASK_BOOL_U8) {
            const uint8_t* m = static_cast<const uint8_t*>(A.mask) + (size_t)b * A.mask_ld;
            rv.mrow = m;
            // group g starts at element g*EPV - phase: its EPV mask bytes are one aligned word iff (m - phase) is
            // aligned to EPV bytes; fp64 rows (EPV = 2) keep the per-element path
            rv.mask_vec = EPV >= 4 && (((reinterpret_cast<uintptr_t>(m) + (uintptr_t)EPV - (uintptr_t)(rv.phase % EPV)) % (uintptr_t)EPV) == 0);
        } else if (MK == GT_MASK_BITS_U32) {
            rv.mrow = static_cast<const uint32_t*>(A.mask) + (size_t)b * A.mask_ld;
        }
        const int ng = rv.n_groups();

        // ---- pass 1: online (max, sum exp) per thread ------------------------------------------------
        // Thread t owns groups t, t + NT, ...  Its interior groups are streamed in rounds of U with no per-group
        // checks: the 16-byte loads (+ mask words) of the next round are requested while the current round is reduced,
        // so every thread keeps 64 bytes of the row in flight.  What is left (fewer than U interior groups, and the
        // one or two edge groups of an unaligned row) is handled group by group afterwards.
        const float SC = rv.scale();
        float m = -INFINITY, s = 0.f;
        // groups in flight per thread: 64 bytes of row (+ mask words); one group for 2-byte rows under an additive mask,
        // whose 32 mask bytes per group would otherwise push the loop into spills
#ifndef GT_S_U2B
#define GT_S_U2B 2
#endif
#ifndef GT_S_UH2B
#define GT_S_UH2B GT_S_U2B
#endif
        constexpr int U = (EPV >= 8 && MK == GT_MASK_ADD_F32) ? 1 : EPV >= 8 ? GT_S_U2B : MK == GT_MASK_ADD_F32 ? 2 : 4;
        const int g_lo = rv.phase ? 1 : 0, g_hi = (rv.phase + rv.V) / EPV;  // interior groups: [g_lo, g_hi)
        const int g0 = tid < g_lo ? tid + NT : tid;
        const int cnt = g0 < g_hi ? (g_hi - 1 - g0) / NT + 1 : 0;
        const int rounds = cnt / U;
        auto stream = [&](auto vec_tag) {  // vec_tag: the mask lines up with the row's groups (vector mask loads)
            constexpr bool VEC = decltype(vec_tag)::value;
            typename RowView<IN_T, MK>::Raw raw[U];
            typename RowView<IN_T, MK>::Cursor c = rv.cursor(g0);
            if (rounds > 0) {
#pragma unroll
                for (int u = 0; u < U; ++u) raw[u] = rv.template issue<VEC>(c, u * NT);
            }
            for (int r = 0; r < rounds; ++r) {
                const bool more = r + 1 < rounds;
                // the (max, sum) update runs over UH groups at a time: all of the round's values at once is the
                // cheapest, half a round keeps the byte-mask variant inside the register budget of 2 CTAs per SM
                constexpr int UH = (EPV >= 8 && MK != GT_MASK_ADD_F32) ? (GT_S_UH2B < U ? GT_S_UH2B : U) : (MK == GT_MASK_BOOL_U8 && U == 4) ? 2 : U;
#pragma unroll
                for (int h = 0; h < U; h += UH) {
                    float y[UH * EPV];
#pragma unroll
                    for (int uu = 0; uu < UH; ++uu) {
                        const int u = h + uu;
                        float yu[EPV];
                        rv.template finish<VEC>(c, u * NT, raw[u], yu);
#pragma unroll
                        for (int k = 0; k < EPV; ++k) y[uu * EPV + k] = yu[k];
                        // the register set is free again: request this thread's group of the next round right away
                        if (more) raw[u] = rv.template issue<VEC>(c, (U + u) * NT);
                    }
                    online_update<UH * EPV>(y, SC, m, s);
                }
                rv.advance(c, U * NT);
            }
            for (int i = rounds * U; i < cnt; ++i) {
                float y[EPV];
                rv.template finish<VEC>(c, 0, rv.template issue<VEC>(c, 0), y);
                rv.advance(c, NT);
                online_update<EPV>(y, SC, m, s);
            }
        };
        if (MK == GT_MASK_NONE || MK == GT_MASK_BITS_U32 || rv.mask_vec) stream(std::true_type{});
        else stream(std::false_type{});
        {
            if (g_lo == 1 && tid == 0) {
                float y[EPV];
                rv.fetch_edge(0, y);
                online_update<EPV>(y, SC, m, s);
            }
            if (g_hi < ng && g_hi >= g_lo && tid == g_hi % NT) {
                float y[EPV];
                rv.fetch_edge(g_hi, y);
                online_update<EPV>(y, SC, m, s);
            }
        }
        // A NaN element has made this thread's s (and possibly m) NaN: logZ becomes NaN, tok = -1.

        // ---- block reduction (fp64) ------------------------------------------------------------------
        float wm = m;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) wm = fmaxf(wm, __shfl_xor_sync(0xffffffffu, wm, o));
        if (lane == 0) s_wmax[warp] = wm;
        __syncthreads();
        if (tid == 0) {
            float M0 = s_wmax[0];
            for (int w = 1; w < NT / 32; ++w) M0 = fmaxf(M0, s_wmax[w]);
            s_M = M0;
        }
        __syncthreads();
        const float M = s_M;
        s_mass[tid] = (s != s || m != m) ? (double)NAN : (m > -INFINITY) ? (double)s * exp2((double)(m - M) * (double)SC) : 0.0;
        __syncthreads();

        if (warp == 0) {
            double tot = 0.0;
            for (int i = lane; i < NT; i += 32) tot += s_mass[i];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) tot += __shfl_xor_sync(0xffffffffu, tot, o);
            // 53-bit uniform in [0,1): Philox4x32-10, counter = offset + row, key = seed
            const double u = philox_uniform53(A.seed, A.offset + (uint64_t)b);
            const bool ok = (M > -INFINITY) && (tot > 0.0) && (tot < (double)INFINITY);  // false for NaN
            int pick = -1; double before = 0.0;
            if (ok) warp_find(s_mass, NT, u * tot, pick, before);
            if (lane == 0) {
                s_pick = pick;
                s_resid = before < 0.0 ? -1.0 : u * tot - before;
                A.logZ[b] = (tot != tot) ? NAN : (M == -INFINITY) ? -INFINITY : (float)((double)M * (double)rv.unit() + log(tot));
            }
        }
        __syncthreads();
        const int pick = s_pick;
        const double resid = s_resid;
        __syncthreads();  // s_pick / s_resid / s_mass are reused below
        if (pick < 0) {
            if (M == INFINITY) {
                // A +inf at an allowed position made its thread's sum NaN (inf - inf in the exponent), so logZ was
                // written NaN above.  As torch.logsumexp: +inf unless an allowed value is NaN; a re-scan decides.
                bool nan = false;
                for (int g = tid; g < ng; g += NT) {
                    float y[EPV];
                    rv.fetch(g, y);
#pragma unroll
                    for (int k = 0; k < EPV; ++k) nan |= y[k] != y[k];
                }
                if (__syncthreads_or(nan) == 0 && tid == 0) A.logZ[b] = INFINITY;
            }
            if (tid == 0) A.tok[b] = -1;
            continue;
        }

        // ---- pass 2: re-read the picked thread's groups (L2-hot, a few KB) and locate the element ------
        locate_token<IN_T, MK, NT>(rv, pick, resid, M, SC, ng, s_mass, &s_pick, &s_resid, A.tok + b);
        __syncthreads();
    }
}

template <typename IN_T, int MK> static int launch_sampler_mk(const SampleArgs& A, cudaStream_t st) {
    const int sms = sm_count();
    const int grid = A.n_rows < sms * 8 ? A.n_rows : sms * 8;
    // 2-byte rows under an additive fp32 mask move twice as many mask bytes as row bytes per group and measured faster
    // with two wide CTAs per SM (40 vs 51 us); every other combination prefers four CTAs of kSThreads
    constexpr int NT = (sizeof(IN_T) == 2 && MK == GT_MASK_ADD_F32) ? 2 * kSThreads : kSThreads;
    gt::NvtxRange nv("gt:lse_sample");
    lse_sample_kernel<IN_T, MK, NT><<<grid, NT, 0, st>>>(A);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { set_error("lse_sample launch failed: %s", cudaGetErrorString(e)); return GT_ERR_CUDA; }
    return GT_OK;
}
template <typename IN_T> static int launch_sampler(const SampleArgs& A, cudaStream_t st) {
    switch (A.mask_kind) {
        case GT_MASK_NONE: return launch_sampler_mk<IN_T, GT_MASK_NONE>(A, st);
        case GT_MASK_ADD_F32: return launch_sampler_mk<IN_T, GT_MASK_ADD_F32>(A, st);
        case GT_MASK_BOOL_U8: return launch_sampler_mk<IN_T, GT_MASK_BOOL_U8>(A, st);
        default: return launch_sampler_mk<IN_T, GT_MASK_BITS_U32>(A, st);
    }
}

}  // namespace gt

extern "C" int gt_lse_sample(const void* logp, int in_type, int64_t n_rows, int64_t n_vocab, int64_t ld_logp,
                             const void* mask, int mask_kind, int64_t mask_ld, float temperature, uint64_t seed,
                             uint64_t offset, float* logZ_out, int32_t* tok_out, gt_stream stream) {
    if (n_rows < 0 || n_vocab <= 0 || n_vocab >= (int64_t)1 << 30 || ld_logp < n_vocab || !logp || !logZ_out || !tok_out) {
        gt::set_error("gt_lse_sample: bad argument"); return GT_ERR_ARG;
    }
    if (mask_kind != GT_MASK_NONE && !mask) { gt::set_error("gt_lse_sample: mask kind %d needs a mask pointer", mask_kind); return GT_ERR_ARG; }
    if (mask_kind < GT_MASK_NONE || mask_kind > GT_MASK_BITS_U32) { gt::set_error("gt_lse_sample: unknown mask kind %d", mask_kind); return GT_ERR_ARG; }
    if (!(temperature > 0.f)) { gt::set_error("gt_lse_sample: temperature must be > 0"); return GT_ERR_ARG; }
    if (n_rows == 0) return GT_OK;
    if (n_rows > INT32_MAX) { gt::set_error("gt_lse_sample: too many rows"); return GT_ERR_LIMIT; }
    gt::SampleArgs A;
    A.logp = logp; A.ld_logp = ld_logp; A.V = n_vocab; A.n_rows = (int)n_rows;
    A.mask = mask; A.mask_kind = mask_kind; A.mask_ld = mask_ld;
    A.inv_temp = 1.0f / temperature; A.seed = seed; A.offset = offset; A.logZ = logZ_out; A.tok = tok_out;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    switch (in_type) {
        case GT_F32: return gt::launch_sampler<float>(A, st);
        case GT_F64: return gt::launch_sampler<double>(A, st);
        case GT_F16: return gt::launch_sampler<__half>(A, st);
        case GT_BF16: return gt::launch_sampler<__nv_bfloat16>(A, st);
        default: gt::set_error("gt_lse_sample: unknown input type %d", in_type); return GT_ERR_ARG;
    }
}
