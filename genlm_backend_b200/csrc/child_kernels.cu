// sm_100a kernels for the next-symbol read-outs of the trie.
#include <climits>
#include <cmath>
#include <cstring>
#include <algorithm>

#include "trie_device.cuh"
#include "philox.cuh"

namespace gt {

// ---- next-symbol read-outs: masses of the children of one node per row, by child or by symbol, and the draw ---------
// (gt_child_masses / gt_child_sample / gt_symbol_masses / gt_symbol_sample, and their *_masked twins, which restrict
// the rows to the items a per-row keep-bitmask allows: only the block kernel differs, by a compile-time parameter)
//
// The children of a node n tile its DFS leaf range [lo(n), hi(n)) with consecutive ranges (post-order numbering, DESIGN
// section 2), so the job is a segmented reduction over one contiguous range of DFS ranks per row, with at most D segments.
// The range is cut into *blocks* of kChildBlock ranks aligned to lo(n), and a block is one warp's work: a batch of root
// rows (251 blocks each at 128k tokens) spreads over every SM, while a deep node's row is a single block.
//   child_scan_kernel    one CTA: blocks per row and their exclusive scan (the chunk's work list)
//   child_block_kernel   persistent warps take blocks u = warp, warp + warps, ...; block k of row b writes the fp64 partial
//                        sum (and the max) of each child segment j it overlaps to slot j + k of the row.  Children are
//                        consecutive, so k_first(j + 1) >= k_last(j) and (j, k) -> j + k is injective: no atomics
//   finish kernels       one warp per row, all starting from finish_row (a child's slots added in k order, the lanes'
//                        sums scanned in a fixed order); one per job:
//     child_masses_kernel   ids / sums / maxes by child (normalised, logs)
//     symbol_masses_kernel  sums / maxes by symbol
//     child_draw_kernel     the next child, optionally under per-row symbol log-weights
// Every sum is a fixed function of (node, child): lane l of a block adds the block's ranks 4l + 128q + i (q < 4, i < 4)
// in that order, the warp combines its lanes by a fixed butterfly, and the finish kernel adds a child's blocks in order.
// The batch, the row's position in it, the chunking, the input order and the grid size change nothing.
constexpr int kChildBlock = 512;  // DFS ranks per block: 16 per lane, as four quads of 4 consecutive ranks
constexpr int kChildQuads = kChildBlock / 128;
constexpr int64_t kMaxChildRows = 1024;  // rows per chunk (the chunk's work list is staged in shared memory)
constexpr int kChildThreads = 256;

struct ChildArgs {
    const void* ws; int in_type; int log_input; int dfs_order; int64_t ld_ws;
    const int32_t* nodes; int n_rows;   // the chunk's rows
    int32_t* blk_off;                   // [n_rows + 1] exclusive scan of the blocks per row
    double* part_sum; float* part_max;  // [n_rows][slots]
    int64_t slots; int need_max;
    // child_masses_kernel (child_ids, D) and symbol_masses_kernel
    int32_t* child_ids; float* out_sum; float* out_max; int64_t ld_out; int D; int normalize, log_out;
    // child_draw_kernel
    int32_t* child_out; float* logp_out; float* logZ_out; uint64_t seed, ctr0;  // ctr0 = offset + first row of the chunk
    // ... optional: per-row symbol log-weights (row stride ld_w, 0 = shared), the drawn symbol and the node's log-mass
    const float* sym_logw; int64_t ld_w; int32_t* symbol_out; float* logM_out;
    // the *_masked calls: keep-bitmask in item order (GT_MASK_BITS_U32), row stride mask_ld words (0 = shared)
    const uint32_t* mask; int64_t mask_ld;
};

// Children CSR range and DFS leaf range of node n; false for an id outside [0, N) and for a leaf.
__device__ __forceinline__ bool child_node(const PlanView& P, int n, int& cp0, int& deg, int& lo, int& hi) {
    if (n < 0 || n >= P.N) return false;
    cp0 = __ldg(P.child_ptr + n);
    deg = __ldg(P.child_ptr + n + 1) - cp0;
    if (deg <= 0) return false;
    lo = __ldg(P.node_lo + n); hi = __ldg(P.node_hi + n);
    return true;
}

__global__ void __launch_bounds__(1024) child_scan_kernel(PlanView P, ChildArgs A) {
    __shared__ int s_warp[32];
    pdl_wait();  // the node ids may come from the previous kernel; the work list may still be read by the last chunk
    pdl_trigger();
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int carry = 0;
    for (int base = 0; base < A.n_rows; base += 1024) {
        const int i = base + tid;
        int x = 0, cp0, deg, lo, hi;
        if (i < A.n_rows && child_node(P, __ldg(A.nodes + i), cp0, deg, lo, hi)) x = (hi - lo + kChildBlock - 1) / kChildBlock;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int y = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= o) x += y;
        }
        if (lane == 31) s_warp[warp] = x;
        __syncthreads();
        if (warp == 0) {
            int w = s_warp[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int y = __shfl_up_sync(0xffffffffu, w, o);
                if (lane >= o) w += y;
            }
            s_warp[lane] = w;
        }
        __syncthreads();
        if (i < A.n_rows) A.blk_off[i + 1] = carry + x + (warp ? s_warp[warp - 1] : 0);
        carry += s_warp[31];
        __syncthreads();  // s_warp is rewritten by the next 1,024 rows
    }
    if (tid == 0) A.blk_off[0] = 0;
}

template <typename IN_T> __device__ __forceinline__ void load_quad(const IN_T* p, IN_T (&x)[4]) {
    if constexpr (sizeof(IN_T) == 4) { const float4 t = __ldg(reinterpret_cast<const float4*>(p)); memcpy(x, &t, 16); }
    else if constexpr (sizeof(IN_T) == 2) { const uint2 t = __ldg(reinterpret_cast<const uint2*>(p)); memcpy(x, &t, 8); }
    else {
        const double2 a = __ldg(reinterpret_cast<const double2*>(p)), c = __ldg(reinterpret_cast<const double2*>(p) + 1);
        memcpy(x, &a, 16); memcpy(x + 2, &c, 16);
    }
}

// Bit i of the keep-bitmask row m (item order, bit i % 32 of word i / 32).
__device__ __forceinline__ bool mask_keeps(const uint32_t* m, int i) { return (__ldg(m + (i >> 5)) >> (i & 31)) & 1u; }

// Block k of row b (one warp).  MASKED: an item whose bit in the row's keep-bitmask is 0 contributes the weight 0.f
// (its weight is not loaded where that is cheap), which is the converted weight of a zeroed row (-inf under
// GT_FLAG_LOG_INPUT): every sum, its order and every max are those of the zeroed row.
template <typename IN_T, bool MASKED>
__device__ __forceinline__ void child_block(const PlanView& P, const ChildArgs& A, int b, int k, int lane) {
    int cp0 = 0, deg = 0, lo = 0, hi = 0;
    child_node(P, __ldg(A.nodes + b), cp0, deg, lo, hi);  // true: the row has blocks
    const int w0 = lo + k * kChildBlock, w1 = min(hi, w0 + kChildBlock);
    const IN_T* row = static_cast<const IN_T*>(A.ws) + (size_t)b * A.ld_ws;
    const bool log_input = A.log_input != 0;
    const uint32_t* mrow = MASKED ? A.mask + (size_t)b * A.mask_ld : nullptr;
    // the weights of this lane's ranks w0 + 4 lane + 128 q + i (0 outside the block; never added)
    float f[kChildQuads][4];
    if (A.dfs_order) {  // contiguous: one vector load per quad where the row allows it
        unsigned keep = 0xffffu;  // MASKED: bit 4 q + i is the mask bit of rank w0 + 4 lane + 128 q + i
        if constexpr (MASKED) {  // the rank's item perm[r], then its mask word
            keep = 0;
#pragma unroll
            for (int q = 0; q < kChildQuads; ++q)
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int r = w0 + 4 * lane + 128 * q + i;
                    if (r < w1 && mask_keeps(mrow, __ldg(P.perm + r))) keep |= 1u << (4 * q + i);
                }
        }
        const bool vec = (reinterpret_cast<uintptr_t>(row + w0) & (sizeof(IN_T) == 2 ? 7 : 15)) == 0;
#pragma unroll
        for (int q = 0; q < kChildQuads; ++q) {
            const int r0 = w0 + 4 * lane + 128 * q;
            if (vec && r0 + 4 <= w1) {
                if (!MASKED || ((keep >> (4 * q)) & 15u)) {
                    IN_T x[4];
                    load_quad<IN_T>(row + r0, x);
#pragma unroll
                    for (int i = 0; i < 4; ++i) f[q][i] = convert_in<float, IN_T>(x[i], log_input);
                } else {
#pragma unroll
                    for (int i = 0; i < 4; ++i) f[q][i] = 0.f;
                }
            } else {
#pragma unroll
                for (int i = 0; i < 4; ++i) f[q][i] = r0 + i < w1 ? convert_in<float, IN_T>(__ldg(row + r0 + i), log_input) : 0.f;
            }
            if constexpr (MASKED) {  // the cleared bits of a quad loaded as a whole, and of a block's edge
#pragma unroll
                for (int i = 0; i < 4; ++i) f[q][i] = (keep >> (4 * q + i)) & 1u ? f[q][i] : 0.f;
            }
        }
    } else {  // vocabulary order: ws[b, perm[r]], perm read coalesced (L2-resident metadata)
        const bool vec = (w0 & 3) == 0;
        int pi[kChildQuads][4];
#pragma unroll
        for (int q = 0; q < kChildQuads; ++q) {
            const int r0 = w0 + 4 * lane + 128 * q;
            if (vec && r0 + 4 <= w1) {
                const int4 t = __ldg(reinterpret_cast<const int4*>(P.perm + r0));
                pi[q][0] = t.x; pi[q][1] = t.y; pi[q][2] = t.z; pi[q][3] = t.w;
            } else {
#pragma unroll
                for (int i = 0; i < 4; ++i) pi[q][i] = r0 + i < w1 ? __ldg(P.perm + r0 + i) : -1;
            }
        }
#pragma unroll
        for (int q = 0; q < kChildQuads; ++q)
#pragma unroll
            for (int i = 0; i < 4; ++i)
                f[q][i] = pi[q][i] >= 0 && (!MASKED || mask_keeps(mrow, pi[q][i]))
                              ? convert_in<float, IN_T>(__ldg(row + pi[q][i]), log_input) : 0.f;
    }

    // first child whose range ends past w0: narrow [a, z] about 31-fold per round (hi(c_z) > w0 holds throughout).  The
    // probes a, a + s, ..., min(a + 31 s, z) reach z (31 s >= z - a), so some lane always passes
    const int32_t* ch = P.child_idx + cp0;
    int a = 0, z = deg - 1;
    while (z - a >= 32) {
        const int s = (z - a + 30) / 31;
        const int j = min(a + lane * s, z);
        const int l = __ffs(__ballot_sync(0xffffffffu, __ldg(P.node_hi + __ldg(ch + j)) > w0)) - 1;
        const int na = l == 0 ? a : a + (l - 1) * s + 1;
        z = min(z, a + l * s);
        a = na;
    }
    const bool first = a + lane <= z && __ldg(P.node_hi + __ldg(ch + a + lane)) > w0;
    const int jf = a + __ffs(__ballot_sync(0xffffffffu, first)) - 1;

    double* psum = A.part_sum + (size_t)b * A.slots + k;
    float* pmax = A.part_max + (size_t)b * A.slots + k;
    for (int j0 = jf; j0 < deg; j0 += 32) {
        int clo = INT_MAX, chi = INT_MAX;  // the ranges of the next 32 children, one per lane
        if (j0 + lane < deg) {
            const int c = __ldg(ch + j0 + lane);
            clo = __ldg(P.node_lo + c); chi = __ldg(P.node_hi + c);
        }
        const int cnt = min(32, deg - j0);
        for (int t = 0; t < cnt; ++t) {
            const int sa = max(__shfl_sync(0xffffffffu, clo, t), w0), sb = min(__shfl_sync(0xffffffffu, chi, t), w1);
            if (sa >= w1) return;  // warp-uniform: this child and the later ones start past the block
            double s = 0.0;
            float m = -INFINITY;
#pragma unroll
            for (int q = 0; q < kChildQuads; ++q)
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int r = w0 + 4 * lane + 128 * q + i;
                    if (r >= sa && r < sb) { s += (double)f[q][i]; m = fmaxf(m, f[q][i]); }
                }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                s += __shfl_xor_sync(0xffffffffu, s, o);
                m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
            }
            if (lane == 0) {
                psum[j0 + t] = s;
                if (A.need_max) pmax[j0 + t] = m;
            }
        }
    }
}

// Three CTAs per SM: 70 registers without spills (the default budget for these parameters was 64, which spilled).
// MASKED (the *_masked calls) is a separate instantiation, so the unmasked kernel is the code it was without masks.
template <bool MASKED>
__global__ void __launch_bounds__(kChildThreads, 3) child_block_kernel(PlanView P, ChildArgs A) {
    __shared__ int s_off[kMaxChildRows + 1];
    pdl_wait();  // rows, node ids and the work list come from earlier kernels; the slots may still be read by the last chunk
    pdl_trigger();
    for (int i = threadIdx.x; i <= A.n_rows; i += kChildThreads) s_off[i] = A.blk_off[i];
    __syncthreads();
    const int total = s_off[A.n_rows];
    const int lane = threadIdx.x & 31;
    const int warps = (int)gridDim.x * (kChildThreads / 32);
    for (int u = (int)blockIdx.x * (kChildThreads / 32) + (int)(threadIdx.x >> 5); u < total; u += warps) {
        int lo = 0, hi = A.n_rows - 1;  // the row of block u: the last b with s_off[b] <= u
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (s_off[mid] <= u) lo = mid; else hi = mid - 1;
        }
        GT_IN_TYPE_SWITCH(A.in_type, (child_block<IN_T, MASKED>(P, A, lo, u - s_off[lo], lane)));
    }
}

// The slots of row b seen from a finish kernel: child j's sum (its blocks' fp64 partials added in k order) and max.
struct ChildSlots {
    const PlanView& P; const int32_t* ch; const double* psum; const float* pmax; int lo;
    __device__ __forceinline__ void blocks(int c, int& k0, int& k1) const {  // the blocks child c overlaps
        k0 = (__ldg(P.node_lo + c) - lo) / kChildBlock;
        k1 = (__ldg(P.node_hi + c) - 1 - lo) / kChildBlock;
    }
    __device__ __forceinline__ double sum(int j) const {
        int k0, k1;
        blocks(__ldg(ch + j), k0, k1);
        double s = 0.0;
        for (int k = k0; k <= k1; ++k) s += psum[j + k];
        return s;
    }
    __device__ __forceinline__ float max(int j) const {
        int k0, k1;
        blocks(__ldg(ch + j), k0, k1);
        float m = -INFINITY;
        for (int k = k0; k <= k1; ++k) m = fmaxf(m, pmax[j + k]);
        return m;
    }
};

// The draw of a finish kernel: the first child whose running sum of terms q(j) exceeds target (= u * total, total > 0
// and finite), else -- rounding pushed the target past the running sums -- the last child with q(j) > 0.  Lane l owns
// the children [j_lo, j_hi); local is the sum of their terms, incl its inclusive scan over the lanes.  Returns the
// child's position j and its term in `term`.
template <typename Q>
__device__ __forceinline__ int pick_child(const Q& q, int j_lo, int j_hi, double local, double incl, double target, int lane,
                                          double& term) {
    int pick = -1;
    double mass = 0.0;
    const unsigned hit = __ballot_sync(0xffffffffu, incl > target && local > 0.0);
    if (hit) {
        const int src = __ffs(hit) - 1;
        if (lane == src) {
            double run = incl - local;
            for (int j = j_lo; j < j_hi; ++j) {
                const double s = q(j);
                if (s > 0.0) { pick = j; mass = s; if (run + s > target) break; }
                run += s;
            }
        }
        pick = __shfl_sync(0xffffffffu, pick, src);
        mass = __shfl_sync(0xffffffffu, mass, src);
    } else {
        int last = -1;
        if (local > 0.0)
            for (int j = j_hi - 1; j >= j_lo; --j)
                if (q(j) > 0.0) { last = j; break; }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) last = max(last, __shfl_xor_sync(0xffffffffu, last, o));
        pick = last;
        mass = q(pick);  // last >= 0: total > 0
    }
    term = mass;
    return pick;
}

__device__ __forceinline__ double warp_inclusive_scan(double x, int lane) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const double y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
    }
    return x;
}

// Where every finish kernel starts (one warp per row b): the row's node (no children for an invalid id or a leaf), its
// slots, and the children [j_lo, j_hi) lane l owns.  local adds their sums in order and an inclusive scan over the lanes
// gives the running sums incl and the node's mass total: one fixed order, so normalisation, draw and every finish kernel
// see the same sums.
struct FinishRow {
    ChildSlots cs; const int32_t* sy; int deg, j_lo, j_hi; double local, incl, total;
};
__device__ __forceinline__ FinishRow finish_row(const PlanView& P, const ChildArgs& A, int b, int lane) {
    int cp0 = 0, deg = 0, lo = 0, hi = 0;
    if (!child_node(P, __ldg(A.nodes + b), cp0, deg, lo, hi)) deg = 0;
    const ChildSlots cs{P, P.child_idx + cp0, A.part_sum + (size_t)b * A.slots, A.part_max + (size_t)b * A.slots, lo};
    const int per = (deg + 31) / 32;
    const int j_lo = min(deg, lane * per), j_hi = min(deg, j_lo + per);
    double local = 0.0;
    for (int j = j_lo; j < j_hi; ++j) local += cs.sum(j);
    const double incl = warp_inclusive_scan(local, lane);
    return {cs, P.child_sym + cp0, deg, j_lo, j_hi, local, incl, __shfl_sync(0xffffffffu, incl, 31)};
}

// A child's sum and max as the masses read-outs write them: the sum divided by the node's mass (GT_CHILD_NORMALIZE),
// both as logs (GT_CHILD_LOG), rounded to fp32 once.
__device__ __forceinline__ float sum_out(const ChildArgs& A, double s, double total) {
    if (A.normalize) s /= total;
    return (float)(A.log_out ? log(s) : s);
}
__device__ __forceinline__ float max_out(const ChildArgs& A, float m) { return A.log_out ? (float)log((double)m) : m; }

__global__ void __launch_bounds__(kChildThreads) child_masses_kernel(PlanView P, ChildArgs A) {
    pdl_wait();  // the slots come from child_block_kernel
    pdl_trigger();
    const int lane = threadIdx.x & 31;
    const int b = (int)blockIdx.x * (kChildThreads / 32) + (int)(threadIdx.x >> 5);
    if (b >= A.n_rows) return;
    const FinishRow r = finish_row(P, A, b, lane);
    int32_t* ids = A.child_ids + (size_t)b * A.ld_out;
    float* os = A.out_sum ? A.out_sum + (size_t)b * A.ld_out : nullptr;
    float* om = A.out_max ? A.out_max + (size_t)b * A.ld_out : nullptr;
    for (int j = r.j_lo; j < r.j_hi; ++j) {
        ids[j] = __ldg(r.cs.ch + j);
        if (os) os[j] = sum_out(A, r.cs.sum(j), r.total);
        if (om) om[j] = max_out(A, r.cs.max(j));
    }
    const float pad = A.log_out ? -INFINITY : 0.f;
    for (int j = r.deg + lane; j < A.D; j += 32) {
        ids[j] = -1;
        if (os) os[j] = pad;
        if (om) om[j] = pad;
    }
}

// Indexed by symbol: child j goes to column child_sym[j] (S for a leaf child), so every value is bit-equal to that of
// child_masses_kernel.  The row is first filled with padding, then each non-leaf child writes its own column (a node
// has one child per symbol), and column S gets the leaf children's sums added in child order.
__global__ void __launch_bounds__(kChildThreads) symbol_masses_kernel(PlanView P, ChildArgs A) {
    pdl_wait();  // the slots come from child_block_kernel
    pdl_trigger();
    const int lane = threadIdx.x & 31;
    const int b = (int)blockIdx.x * (kChildThreads / 32) + (int)(threadIdx.x >> 5);
    if (b >= A.n_rows) return;
    const FinishRow r = finish_row(P, A, b, lane);
    const int S = P.S;
    float* os = A.out_sum ? A.out_sum + (size_t)b * A.ld_out : nullptr;
    float* om = A.out_max ? A.out_max + (size_t)b * A.ld_out : nullptr;
    const float pad = A.log_out ? -INFINITY : 0.f;
    for (int s = lane; s <= S; s += 32) {
        if (os) os[s] = pad;
        if (om) om[s] = pad;
    }
    __syncwarp();  // the children's columns overwrite the padding
    bool has_end = false;
    for (int j = r.j_lo; j < r.j_hi; ++j) {
        const int sym = __ldg(r.sy + j);
        if (sym == S) { has_end = true; continue; }
        if (os) os[sym] = sum_out(A, r.cs.sum(j), r.total);
        if (om) om[sym] = max_out(A, r.cs.max(j));
    }
    // end of token: the leaf children, lane by lane in child order (usually one lane, one child)
    const unsigned ends = __ballot_sync(0xffffffffu, has_end);
    double es = 0.0;
    float em = -INFINITY;
    for (unsigned e = ends; e; e &= e - 1) {
        const int src = __ffs(e) - 1;
        if (lane == src)
            for (int j = r.j_lo; j < r.j_hi; ++j)
                if (__ldg(r.sy + j) == S) {
                    if (os) es += r.cs.sum(j);
                    if (om) em = fmaxf(em, r.cs.max(j));
                }
        es = __shfl_sync(0xffffffffu, es, src);
        em = __shfl_sync(0xffffffffu, em, src);
    }
    if (ends && lane == 0) {
        if (os) os[S] = sum_out(A, es, r.total);
        if (om) om[S] = max_out(A, em);
    }
}

// The next-symbol draw: the first child whose running sum of terms q_j exceeds u * Z, Z the sum of all q_j.  Without
// log-weights q_j is the child's mass m_j and Z the node's mass.  With them (gt_symbol_sample) q_j = m_j * exp(logw[sym_j])
// in fp64, scanned like the m_j: no mass stays 0 whatever the weight, and a NaN weight poisons the row.  With all
// log-weights 0 the two give the same bits.  symbol_out and logM_out are optional.
__global__ void __launch_bounds__(kChildThreads) child_draw_kernel(PlanView P, ChildArgs A) {
    pdl_wait();  // the slots come from child_block_kernel
    pdl_trigger();
    const int lane = threadIdx.x & 31;
    const int b = (int)blockIdx.x * (kChildThreads / 32) + (int)(threadIdx.x >> 5);
    if (b >= A.n_rows) return;
    const FinishRow r = finish_row(P, A, b, lane);
    const float* lw = A.sym_logw ? A.sym_logw + (size_t)b * A.ld_w : nullptr;
    auto term = [&](int j) {
        if (!lw) return r.cs.sum(j);
        const float w = __ldg(lw + __ldg(r.sy + j));
        if (isnan(w)) return (double)NAN;
        const double m = r.cs.sum(j);
        return m == 0.0 ? 0.0 : m * exp((double)w);
    };
    double local = r.local, incl = r.incl, total = r.total;
    if (lw) {
        local = 0.0;
        for (int j = r.j_lo; j < r.j_hi; ++j) local += term(j);
        incl = warp_inclusive_scan(local, lane);
        total = __shfl_sync(0xffffffffu, incl, 31);
    }
    const bool ok = total > 0.0 && total < (double)INFINITY;  // false for NaN
    int pick = -1;
    double mass = 0.0;
    if (ok) pick = pick_child(term, r.j_lo, r.j_hi, local, incl, philox_uniform53(A.seed, A.ctr0 + (uint64_t)b) * total, lane, mass);
    if (lane == 0) {
        A.child_out[b] = ok ? __ldg(r.cs.ch + pick) : -1;
        if (A.symbol_out) A.symbol_out[b] = ok ? __ldg(r.sy + pick) : -1;
        A.logZ_out[b] = (float)log(total);  // -inf for no mass, NaN for a NaN weight, +inf for an infinite total
        A.logp_out[b] = ok ? (float)(log(mass) - log(total)) : (total == 0.0 ? -INFINITY : NAN);
        if (A.logM_out) A.logM_out[b] = (float)log(r.total);
    }
}

// Scratch of the child-mass calls for a chunk of `rows` rows:
//   blk_off [rows + 1] int32 | part_sum [rows][slots] fp64 | part_max [rows][slots] fp32
// slots = D + ceil(V / kChildBlock): block k of a row writes child j's partials to slot j + k, j < D, k < ceil(V / kChildBlock).
struct ChildScratch {
    int32_t* blk_off; double* part_sum; float* part_max;
    int64_t rows;  // capacity (0: not even one row)
    static size_t pad(size_t b) { return (b + 255) & ~size_t(255); }
    static int64_t slots(const Layout& L) { return L.max_children + (L.V + kChildBlock - 1) / kChildBlock; }
    static size_t total(int64_t rows, int64_t slots) {
        return pad((size_t)(rows + 1) * 4) + pad((size_t)rows * slots * 8) + pad((size_t)rows * slots * 4);
    }
    ChildScratch(void* base, size_t bytes, int64_t slots) {
        int64_t lo = 0, hi = kMaxChildRows;
        while (lo < hi) {  // total() is monotone in the row count
            const int64_t mid = (lo + hi + 1) / 2;
            if (total(mid, slots) <= bytes) lo = mid; else hi = mid - 1;
        }
        rows = lo;
        char* p = static_cast<char*>(base);
        blk_off = reinterpret_cast<int32_t*>(p);
        p += pad((size_t)(rows + 1) * 4);
        part_sum = reinterpret_cast<double*>(p);
        p += pad((size_t)rows * slots * 8);
        part_max = reinterpret_cast<float*>(p);
    }
};

// Shared by gt_child_masses, gt_child_sample, gt_symbol_masses and gt_symbol_sample and their *_masked twins: arguments
// are checked by the callers (before any CUDA call); this selects the device plan and launches scan -> blocks -> finish
// per chunk of rows, chained with programmatic dependent launch on the caller's stream.  A.nodes / A.ws / A.mask /
// outputs point at row 0; chunk c advances them.  A mask selects the masked instantiation of the block kernel.
static int launch_child(const gt_trie* t, ChildArgs A, int64_t n_rows, int64_t out_ld_rows, uint64_t offset, void* workspace,
                        size_t workspace_bytes, cudaStream_t st, const char* what, void (*finish)(PlanView, ChildArgs)) {
    const int64_t slots = ChildScratch::slots(t->layout);
    const ChildScratch sc(workspace, workspace_bytes, slots);
    if (sc.rows < 1) {
        set_error("%s: workspace too small: %zu bytes given, one row needs %zu", what, workspace_bytes, ChildScratch::total(1, slots));
        return GT_ERR_STATE;
    }
    const PlanView* pv = nullptr;
    if (const int rc = resident_plan(t, pv); rc != GT_OK) return rc;
    const PlanView& v = *pv;
    const size_t in_size = in_type_size(A.in_type);
    const int64_t max_blocks = (t->layout.V + kChildBlock - 1) / kChildBlock;
    void (*block)(PlanView, ChildArgs) = A.mask ? child_block_kernel<true> : child_block_kernel<false>;
    const int resident = sm_count() * resident_ctas(reinterpret_cast<const void*>(block), kChildThreads, 0);
    A.blk_off = sc.blk_off; A.part_sum = sc.part_sum; A.part_max = sc.part_max; A.slots = slots;
    const char* ws0 = static_cast<const char*>(A.ws);
    const int32_t* nodes0 = A.nodes;
    ChildArgs C = A;
    NvtxRange nv("gt:child");
    for (int64_t r0 = 0; r0 < n_rows; r0 += sc.rows) {
        const int rows = (int)std::min<int64_t>(sc.rows, n_rows - r0);
        C.n_rows = rows;
        C.ws = ws0 + (size_t)r0 * A.ld_ws * in_size;
        C.nodes = nodes0 + r0;
        const size_t o = (size_t)r0 * out_ld_rows;
        if (A.child_ids) C.child_ids = A.child_ids + o;
        if (A.out_sum) C.out_sum = A.out_sum + o;
        if (A.out_max) C.out_max = A.out_max + o;
        if (A.child_out) { C.child_out = A.child_out + r0; C.logp_out = A.logp_out + r0; C.logZ_out = A.logZ_out + r0; }
        if (A.symbol_out) C.symbol_out = A.symbol_out + r0;
        if (A.logM_out) C.logM_out = A.logM_out + r0;
        if (A.sym_logw) C.sym_logw = A.sym_logw + (size_t)r0 * A.ld_w;
        if (A.mask) C.mask = A.mask + (size_t)r0 * A.mask_ld;
        C.ctr0 = offset + (uint64_t)r0;
        const int64_t blocks_ub = (int64_t)rows * max_blocks;  // every row at the root
        const unsigned grid = (unsigned)std::max<int64_t>(1, std::min<int64_t>(resident, (blocks_ub + kChildThreads / 32 - 1) / (kChildThreads / 32)));
        GT_CUDA(launch_pdl(child_scan_kernel, dim3(1), dim3(1024), 0, st, v, C));
        GT_CUDA(launch_pdl(block, dim3(grid), dim3(kChildThreads), 0, st, v, C));
        GT_CUDA(launch_pdl(finish, dim3((unsigned)((rows + kChildThreads / 32 - 1) / (kChildThreads / 32))),
                           dim3(kChildThreads), 0, st, v, C));
    }
    return GT_OK;
}
}  // namespace gt

extern "C" {

size_t gt_child_workspace_bytes(const gt_trie* t, int64_t max_rows) {
    if (!t || max_rows <= 0) return 0;
    return gt::ChildScratch::total(std::min<int64_t>(max_rows, gt::kMaxChildRows), gt::ChildScratch::slots(t->layout)) + 256;
}

// Checks shared by the next-symbol read-outs.  Each of the four calls and its *_masked twin share one implementation
// (the unmasked call passes no mask), which makes its checks in one order: the scalars and strides
// (child_check_scalars, then its own), the early return for no rows, the data pointers (its own outputs, then
// child_check_pointers) and last the workspace, so that a call without rows accepts null pointers.
// child_check_scalars fills the input half of A.
static int child_check_scalars(const gt_trie* t, const void* ws, int in_type, int64_t n_rows, int64_t ld_ws,
                               const int32_t* nodes, const uint32_t* mask, int64_t mask_ld, unsigned flags, unsigned known,
                               const char* what, gt::ChildArgs& A) {
    if (!t) { gt::set_error("%s: null trie", what); return GT_ERR_ARG; }
    if (n_rows < 0 || (flags & ~known) || !gt::in_type_size(in_type)) {
        gt::set_error("%s: bad n_rows / flags / input type", what); return GT_ERR_ARG;
    }
    if (ld_ws < t->layout.V) {
        gt::set_error("%s: row stride %lld smaller than V = %lld", what, (long long)ld_ws, (long long)t->layout.V); return GT_ERR_ARG;
    }
    const int64_t words = (t->layout.V + 31) / 32;
    if (mask_ld < 0 || (mask_ld > 0 && mask_ld < words)) {
        gt::set_error("%s: mask row stride %lld is neither 0 (shared) nor >= ceil(V/32) = %lld", what, (long long)mask_ld,
                      (long long)words);
        return GT_ERR_ARG;
    }
    A.ws = ws; A.in_type = in_type; A.ld_ws = ld_ws; A.nodes = nodes; A.mask = mask; A.mask_ld = mask_ld;
    A.log_input = (flags & GT_FLAG_LOG_INPUT) ? 1 : 0; A.dfs_order = (flags & GT_FLAG_DFS_ORDER) ? 1 : 0;
    A.normalize = (flags & GT_CHILD_NORMALIZE) ? 1 : 0; A.log_out = (flags & GT_CHILD_LOG) ? 1 : 0;
    return GT_OK;
}

// masked: the *_masked twin, which needs its mask.
static int child_check_pointers(const gt_trie* t, const void* ws, const int32_t* nodes, bool masked, const uint32_t* mask,
                                const void* workspace, const char* what) {
    if ((t->layout.V > 0 && !ws) || !nodes || (masked && !mask)) { gt::set_error("%s: null data pointer", what); return GT_ERR_ARG; }
    if (!workspace || (reinterpret_cast<uintptr_t>(workspace) & 255)) {
        gt::set_error("%s: workspace must be a 256-byte aligned device pointer", what); return GT_ERR_ARG;
    }
    return GT_OK;
}

static const unsigned kMassesFlags = GT_FLAG_LOG_INPUT | GT_FLAG_DFS_ORDER | GT_CHILD_NORMALIZE | GT_CHILD_LOG;
static const unsigned kSampleFlags = GT_FLAG_LOG_INPUT | GT_FLAG_DFS_ORDER;

static int child_masses_impl(const gt_trie* t, const void* ws, int in_type, int64_t n_rows, int64_t ld_ws, const int32_t* nodes,
                             bool masked, const uint32_t* mask_bits, int64_t mask_ld, int32_t* child_ids, float* out_sum,
                             float* out_max, int64_t ld_out, unsigned ops, unsigned flags, void* workspace,
                             size_t workspace_bytes, gt_stream stream, const char* what) {
    gt::ChildArgs A{};
    int rc = child_check_scalars(t, ws, in_type, n_rows, ld_ws, nodes, mask_bits, mask_ld, flags, kMassesFlags, what, A);
    if (rc != GT_OK) return rc;
    const int64_t D = t->layout.max_children;
    if (!gt::ops_ok(ops) || ld_out < D) {
        gt::set_error("%s: bad ops, or output row stride %lld smaller than D = %lld", what, (long long)ld_out, (long long)D);
        return GT_ERR_ARG;
    }
    if (n_rows == 0 || D == 0) return GT_OK;
    if (!child_ids || ((ops & GT_OP_SUM) && !out_sum) || ((ops & GT_OP_MAX) && !out_max)) {
        gt::set_error("%s: null data pointer", what); return GT_ERR_ARG;
    }
    if ((rc = child_check_pointers(t, ws, nodes, masked, mask_bits, workspace, what)) != GT_OK) return rc;
    A.need_max = (ops & GT_OP_MAX) ? 1 : 0;
    A.child_ids = child_ids; A.out_sum = (ops & GT_OP_SUM) ? out_sum : nullptr; A.out_max = (ops & GT_OP_MAX) ? out_max : nullptr;
    A.ld_out = ld_out; A.D = (int)D;
    return gt::launch_child(t, A, n_rows, ld_out, 0, workspace, workspace_bytes, static_cast<cudaStream_t>(stream), what,
                            gt::child_masses_kernel);
}

int gt_child_masses(const gt_trie* t, const void* ws, int in_type, int64_t n_rows, int64_t ld_ws, const int32_t* nodes,
                    int32_t* child_ids, float* out_sum, float* out_max, int64_t ld_out, unsigned ops, unsigned flags,
                    void* workspace, size_t workspace_bytes, gt_stream stream) {
    return child_masses_impl(t, ws, in_type, n_rows, ld_ws, nodes, false, nullptr, 0, child_ids, out_sum, out_max, ld_out, ops,
                             flags, workspace, workspace_bytes, stream, __func__);
}

int gt_child_masses_masked(const gt_trie* t, const void* ws, int in_type, int64_t n_rows, int64_t ld_ws, const int32_t* nodes,
                           const uint32_t* mask_bits, int64_t mask_ld, int32_t* child_ids, float* out_sum, float* out_max,
                           int64_t ld_out, unsigned ops, unsigned flags, void* workspace, size_t workspace_bytes,
                           gt_stream stream) {
    return child_masses_impl(t, ws, in_type, n_rows, ld_ws, nodes, true, mask_bits, mask_ld, child_ids, out_sum, out_max,
                             ld_out, ops, flags, workspace, workspace_bytes, stream, __func__);
}

static int child_sample_impl(const gt_trie* t, const void* ws, int in_type, int64_t n_rows, int64_t ld_ws, const int32_t* nodes,
                             bool masked, const uint32_t* mask_bits, int64_t mask_ld, unsigned flags, uint64_t seed,
                             uint64_t offset, int32_t* child_out, float* logp_out, float* logZ_out, void* workspace,
                             size_t workspace_bytes, gt_stream stream, const char* what) {
    gt::ChildArgs A{};
    int rc = child_check_scalars(t, ws, in_type, n_rows, ld_ws, nodes, mask_bits, mask_ld, flags, kSampleFlags, what, A);
    if (rc != GT_OK) return rc;
    if (n_rows == 0) return GT_OK;
    if (!child_out || !logp_out || !logZ_out) { gt::set_error("%s: null data pointer", what); return GT_ERR_ARG; }
    if ((rc = child_check_pointers(t, ws, nodes, masked, mask_bits, workspace, what)) != GT_OK) return rc;
    A.seed = seed; A.child_out = child_out; A.logp_out = logp_out; A.logZ_out = logZ_out;
    return gt::launch_child(t, A, n_rows, 0, offset, workspace, workspace_bytes, static_cast<cudaStream_t>(stream), what,
                            gt::child_draw_kernel);
}

int gt_child_sample(const gt_trie* t, const void* ws, int in_type, int64_t n_rows, int64_t ld_ws, const int32_t* nodes,
                    unsigned flags, uint64_t seed, uint64_t offset, int32_t* child_out, float* logp_out, float* logZ_out,
                    void* workspace, size_t workspace_bytes, gt_stream stream) {
    return child_sample_impl(t, ws, in_type, n_rows, ld_ws, nodes, false, nullptr, 0, flags, seed, offset, child_out, logp_out,
                             logZ_out, workspace, workspace_bytes, stream, __func__);
}

int gt_child_sample_masked(const gt_trie* t, const void* ws, int in_type, int64_t n_rows, int64_t ld_ws, const int32_t* nodes,
                           const uint32_t* mask_bits, int64_t mask_ld, unsigned flags, uint64_t seed, uint64_t offset,
                           int32_t* child_out, float* logp_out, float* logZ_out, void* workspace, size_t workspace_bytes,
                           gt_stream stream) {
    return child_sample_impl(t, ws, in_type, n_rows, ld_ws, nodes, true, mask_bits, mask_ld, flags, seed, offset, child_out,
                             logp_out, logZ_out, workspace, workspace_bytes, stream, __func__);
}

static int symbol_masses_impl(const gt_trie* t, const void* ws, int in_type, int64_t n_rows, int64_t ld_ws, const int32_t* nodes,
                              bool masked, const uint32_t* mask_bits, int64_t mask_ld, float* out_sum, float* out_max,
                              int64_t ld_out, unsigned ops, unsigned flags, void* workspace, size_t workspace_bytes,
                              gt_stream stream, const char* what) {
    gt::ChildArgs A{};
    int rc = child_check_scalars(t, ws, in_type, n_rows, ld_ws, nodes, mask_bits, mask_ld, flags, kMassesFlags, what, A);
    if (rc != GT_OK) return rc;
    const int64_t S = t->layout.num_symbols;
    if (!gt::ops_ok(ops) || ld_out < S + 1) {
        gt::set_error("%s: bad ops, or output row stride %lld smaller than S + 1 = %lld", what, (long long)ld_out,
                      (long long)(S + 1));
        return GT_ERR_ARG;
    }
    if (n_rows == 0) return GT_OK;
    if (((ops & GT_OP_SUM) && !out_sum) || ((ops & GT_OP_MAX) && !out_max)) {
        gt::set_error("%s: null data pointer", what); return GT_ERR_ARG;
    }
    if ((rc = child_check_pointers(t, ws, nodes, masked, mask_bits, workspace, what)) != GT_OK) return rc;
    A.need_max = (ops & GT_OP_MAX) ? 1 : 0;
    A.out_sum = (ops & GT_OP_SUM) ? out_sum : nullptr; A.out_max = (ops & GT_OP_MAX) ? out_max : nullptr; A.ld_out = ld_out;
    return gt::launch_child(t, A, n_rows, ld_out, 0, workspace, workspace_bytes, static_cast<cudaStream_t>(stream), what,
                            gt::symbol_masses_kernel);
}

int gt_symbol_masses(const gt_trie* t, const void* ws, int in_type, int64_t n_rows, int64_t ld_ws, const int32_t* nodes,
                     float* out_sum, float* out_max, int64_t ld_out, unsigned ops, unsigned flags,
                     void* workspace, size_t workspace_bytes, gt_stream stream) {
    return symbol_masses_impl(t, ws, in_type, n_rows, ld_ws, nodes, false, nullptr, 0, out_sum, out_max, ld_out, ops, flags,
                              workspace, workspace_bytes, stream, __func__);
}

int gt_symbol_masses_masked(const gt_trie* t, const void* ws, int in_type, int64_t n_rows, int64_t ld_ws, const int32_t* nodes,
                            const uint32_t* mask_bits, int64_t mask_ld, float* out_sum, float* out_max, int64_t ld_out,
                            unsigned ops, unsigned flags, void* workspace, size_t workspace_bytes, gt_stream stream) {
    return symbol_masses_impl(t, ws, in_type, n_rows, ld_ws, nodes, true, mask_bits, mask_ld, out_sum, out_max, ld_out, ops,
                              flags, workspace, workspace_bytes, stream, __func__);
}

static int symbol_sample_impl(const gt_trie* t, const void* ws, int in_type, int64_t n_rows, int64_t ld_ws, const int32_t* nodes,
                              bool masked, const uint32_t* mask_bits, int64_t mask_ld, const float* sym_logw, int64_t ld_w,
                              unsigned flags, uint64_t seed, uint64_t offset, int32_t* child_out, int32_t* symbol_out,
                              float* logp_out, float* logZ_out, float* logM_out, void* workspace, size_t workspace_bytes,
                              gt_stream stream, const char* what) {
    gt::ChildArgs A{};
    int rc = child_check_scalars(t, ws, in_type, n_rows, ld_ws, nodes, mask_bits, mask_ld, flags, kSampleFlags, what, A);
    if (rc != GT_OK) return rc;
    const int64_t S = t->layout.num_symbols;
    if (ld_w < 0 || (ld_w > 0 && ld_w < S + 1)) {
        gt::set_error("%s: log-weight row stride %lld is neither 0 (shared) nor >= S + 1 = %lld", what, (long long)ld_w,
                      (long long)(S + 1));
        return GT_ERR_ARG;
    }
    if (n_rows == 0) return GT_OK;
    if (!sym_logw || !child_out || !symbol_out || !logp_out || !logZ_out) {
        gt::set_error("%s: null data pointer", what); return GT_ERR_ARG;
    }
    if ((rc = child_check_pointers(t, ws, nodes, masked, mask_bits, workspace, what)) != GT_OK) return rc;
    A.seed = seed; A.child_out = child_out; A.logp_out = logp_out; A.logZ_out = logZ_out;
    A.sym_logw = sym_logw; A.ld_w = ld_w; A.symbol_out = symbol_out; A.logM_out = logM_out;
    return gt::launch_child(t, A, n_rows, 0, offset, workspace, workspace_bytes, static_cast<cudaStream_t>(stream), what,
                            gt::child_draw_kernel);
}

int gt_symbol_sample(const gt_trie* t, const void* ws, int in_type, int64_t n_rows, int64_t ld_ws, const int32_t* nodes,
                     const float* sym_logw, int64_t ld_w, unsigned flags, uint64_t seed, uint64_t offset,
                     int32_t* child_out, int32_t* symbol_out, float* logp_out, float* logZ_out, float* logM_out,
                     void* workspace, size_t workspace_bytes, gt_stream stream) {
    return symbol_sample_impl(t, ws, in_type, n_rows, ld_ws, nodes, false, nullptr, 0, sym_logw, ld_w, flags, seed, offset,
                              child_out, symbol_out, logp_out, logZ_out, logM_out, workspace, workspace_bytes, stream, __func__);
}

int gt_symbol_sample_masked(const gt_trie* t, const void* ws, int in_type, int64_t n_rows, int64_t ld_ws, const int32_t* nodes,
                            const uint32_t* mask_bits, int64_t mask_ld, const float* sym_logw, int64_t ld_w, unsigned flags,
                            uint64_t seed, uint64_t offset, int32_t* child_out, int32_t* symbol_out, float* logp_out,
                            float* logZ_out, float* logM_out, void* workspace, size_t workspace_bytes, gt_stream stream) {
    return symbol_sample_impl(t, ws, in_type, n_rows, ld_ws, nodes, true, mask_bits, mask_ld, sym_logw, ld_w, flags, seed,
                              offset, child_out, symbol_out, logp_out, logZ_out, logM_out, workspace, workspace_bytes, stream,
                              __func__);
}

}  // extern "C"
