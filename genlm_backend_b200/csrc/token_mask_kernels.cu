// sm_100a kernels for per-row token masks over the trie: the items under a node (gt_subtree_token_mask), the items a
// byte DFA accepts from there (gt_dfa_token_mask), their log-weights under a weighted byte DFA (gt_dfa_token_logw), and
// the DFA state after a drawn token (gt_dfa_advance).
#include <climits>
#include <algorithm>
#include <type_traits>

#include "trie_device.cuh"

namespace gt {

// token mask: bit i of row b is set iff item i's leaf lies in the subtree of nodes[b], i.e. iff the reference's
// reachability matrix has M[i, nodes[b]] = 1 (parallel.py:33-64).  With leaves in DFS order that is one range test
// on the leaf's DFS rank, so a warp produces one mask word per ballot; kMaskRows rows share every rank load.
constexpr int kMaskThreads = 512, kMaskRows = 16;
__global__ void __launch_bounds__(kMaskThreads) subtree_mask_kernel(PlanView P, const int32_t* __restrict__ nodes, int n_rows,
                                                                    uint32_t* __restrict__ bits, int64_t ld_bits) {
    __shared__ int s_lo[kMaskRows];
    __shared__ unsigned s_len[kMaskRows];
    const int b0 = blockIdx.y * kMaskRows;
    if (threadIdx.x < kMaskRows) {
        const int b = b0 + threadIdx.x;
        int lo = 0; unsigned len = 0;
        if (b < n_rows) {
            const int n = __ldg(nodes + b);
            if (n >= 0 && n < P.N) { lo = __ldg(P.node_lo + n); len = (unsigned)(__ldg(P.node_hi + n) - lo); }
        }
        s_lo[threadIdx.x] = lo; s_len[threadIdx.x] = len;
    }
    const int64_t i = (int64_t)blockIdx.x * kMaskThreads + threadIdx.x;
    const int r = i < P.V ? __ldg(P.leaf_rank + i) : -1;  // -1: fails every range test
    __syncthreads();
    const int64_t w = i >> 5;
    const int rows = min(kMaskRows, n_rows - b0);
    for (int q = 0; q < rows; ++q) {
        const unsigned word = __ballot_sync(0xffffffffu, r >= 0 && (unsigned)(r - s_lo[q]) < s_len[q]);
        if ((threadIdx.x & 31) == 0 && w < ld_bits) bits[(size_t)(b0 + q) * ld_bits + w] = word;
    }
}

// ---- token masks under a byte DFA (gt_dfa_token_mask / gt_dfa_token_logw / gt_dfa_advance) ----------------------------
//
// Row b stands at node n = nodes[b] (the root without nodes) in DFA state q = states[b].  Item i is allowed iff its leaf
// lies under n, q is live (in [0, Q)) and delta walked from q over the item's symbols depth(n) .. len(i)-1 never leaves
// [0, Q).  dfa_mask_kernel: one thread per item, so that a warp's ballot is one mask word (as in subtree_mask_kernel), and
// kDfaRows rows per CTA.  The loop runs over the item's symbols outside and the rows inside: symbol k is loaded once and
// steps the state of every row of the group, which gives each thread kDfaRows independent chains of dependent table loads
// instead of one long chain.  A row outside the subtree, or with a dead start state, starts dead; a thread stops once every
// row of its group is dead.  The table is read through the read-only path (__ldg): a hot table stays in L1 / L2.
// Rows per CTA.  Measured on B200 at 64 rows (DESIGN section 5.10): 8 is 9 % faster than 4 for root rows under a 256-state
// table and 10-29 % slower for depth-1 rows, which have few items each.
#ifndef GT_DFA_ROWS
#define GT_DFA_ROWS 8
#endif
constexpr int kDfaThreads = 256, kDfaRows = GT_DFA_ROWS;

struct DfaArgs {
    const int32_t* delta; int32_t Q, ld;  // [Q][ld] next state; Q * ld < 2^31 (checked by the entry points)
    const int32_t* states; const int32_t* nodes;  // nodes == null: every row at the root
    int n_rows;
};

// Start of row b: its state, the DFS leaf range and the depth of its node; false for an invalid node or a dead state.
__device__ __forceinline__ bool dfa_row(const PlanView& P, const DfaArgs& A, int b, int& q, int& lo, unsigned& len, int& d) {
    const int n = A.nodes ? __ldg(A.nodes + b) : (int)P.N - 1;
    q = __ldg(A.states + b);
    if (n < 0 || n >= P.N || q < 0 || q >= A.Q) return false;
    lo = __ldg(P.node_lo + n);
    len = (unsigned)(__ldg(P.node_hi + n) - lo);
    d = __ldg(P.node_depth + n);
    return true;
}

// One transition; every value outside [0, Q) is a reject, so a malformed table never leads to a read outside it.
__device__ __forceinline__ int dfa_step(const DfaArgs& A, int q, int s) {
    const int nq = __ldg(A.delta + q * A.ld + s);
    return (unsigned)nq < (unsigned)A.Q ? nq : -1;
}

// kLogw = false (gt_dfa_token_mask): out holds keep-bitmask words, ld_out words per row, words of them written.
// kLogw = true (gt_dfa_token_logw): out[b, i] is the fp64 sum of logw[q_k, s_k] over the walked transitions, in
// increasing k and rounded once to fp32, where the bit would be set, else -inf; ld_out floats per row, the first V
// written, words unused.  logw has delta's shape and is loaded at delta's index, as an independent load, so the chain
// of dependent table loads does not grow.  A -inf accumulator does not stop the walk: only the states decide it.
template <bool kLogw>
__global__ void __launch_bounds__(kDfaThreads) dfa_mask_kernel(PlanView P, DfaArgs A, std::conditional_t<kLogw, float, uint32_t>* __restrict__ out,
                                                               int64_t ld_out, int64_t words, const float* __restrict__ logw) {
    __shared__ int s_q[kDfaRows], s_lo[kDfaRows], s_d[kDfaRows];
    __shared__ unsigned s_len[kDfaRows];
    const int b0 = blockIdx.y * kDfaRows;
    if (threadIdx.x < kDfaRows) {
        const int b = b0 + threadIdx.x;
        int q = -1, lo = 0, d = 0;
        unsigned len = 0;
        if (b >= A.n_rows || !dfa_row(P, A, b, q, lo, len, d)) { q = -1; len = 0; }
        s_q[threadIdx.x] = q; s_lo[threadIdx.x] = lo; s_len[threadIdx.x] = len; s_d[threadIdx.x] = d;
    }
    const int64_t i = (int64_t)blockIdx.x * kDfaThreads + threadIdx.x;
    int r = -1, p0 = 0, L = 0;
    if (i < P.V) {
        r = __ldg(P.leaf_rank + i);
        p0 = __ldg(P.item_sym_ptr + i);
        L = __ldg(P.item_sym_ptr + i + 1) - p0;
    }
    __syncthreads();
    int st[kDfaRows], dk[kDfaRows];
    double acc[kDfaRows] = {};
    int k0 = INT_MAX;
#pragma unroll
    for (int g = 0; g < kDfaRows; ++g) {
        const bool in = r >= 0 && s_q[g] >= 0 && (unsigned)(r - s_lo[g]) < s_len[g];
        st[g] = in ? s_q[g] : -1;
        dk[g] = s_d[g];
        if (in) k0 = min(k0, dk[g]);
    }
    const int32_t* sy = P.item_sym + p0;
    for (int k = k0; k < L; ++k) {
        const int s = __ldg(sy + k);
        bool any = false;
#pragma unroll
        for (int g = 0; g < kDfaRows; ++g) {
            if (st[g] >= 0 && k >= dk[g]) {
                if constexpr (kLogw) acc[g] += (double)__ldg(logw + st[g] * A.ld + s);
                st[g] = dfa_step(A, st[g], s);
            }
            any |= st[g] >= 0;
        }
        if (!any) break;
    }
    const int rows = min(kDfaRows, A.n_rows - b0);
    if constexpr (kLogw) {
        if (i >= P.V) return;
#pragma unroll
        for (int g = 0; g < kDfaRows; ++g) {  // consecutive threads store consecutive items: one coalesced store per warp
            if (g >= rows) break;
            out[(size_t)(b0 + g) * ld_out + i] = st[g] >= 0 ? (float)acc[g] : -INFINITY;
        }
    } else {
        const int64_t w = i >> 5;
#pragma unroll
        for (int g = 0; g < kDfaRows; ++g) {
            if (g >= rows) break;
            const unsigned word = __ballot_sync(0xffffffffu, st[g] >= 0);
            if ((threadIdx.x & 31) == 0 && w < words) out[(size_t)(b0 + g) * ld_out + w] = word;
        }
    }
}

// One thread per row walks the drawn item's remaining symbols: the state the particle stands in after the token.
constexpr int kDfaAdvanceThreads = 256;
__global__ void __launch_bounds__(kDfaAdvanceThreads) dfa_advance_kernel(PlanView P, DfaArgs A, const int32_t* __restrict__ tokens,
                                                                         int32_t* __restrict__ out) {
    const int b = blockIdx.x * kDfaAdvanceThreads + threadIdx.x;
    if (b >= A.n_rows) return;
    const int t = __ldg(tokens + b);
    int q, lo, d, res = -1;
    unsigned len;
    if (t >= 0 && t < P.V && dfa_row(P, A, b, q, lo, len, d) && (unsigned)(__ldg(P.leaf_rank + t) - lo) < len) {
        const int p1 = __ldg(P.item_sym_ptr + t + 1);
        for (int p = __ldg(P.item_sym_ptr + t) + d; p < p1 && q >= 0; ++p) q = dfa_step(A, q, __ldg(P.item_sym + p));
        res = q;
    }
    out[b] = res;
}

}  // namespace gt

extern "C" {

int gt_subtree_token_mask(const gt_trie* t, const int32_t* nodes, int64_t n_rows, uint32_t* mask_bits, int64_t mask_ld,
                          gt_stream stream) {
    if (!t) { gt::set_error("gt_subtree_token_mask: null trie"); return GT_ERR_ARG; }
    const int64_t words = (t->layout.V + 31) / 32;
    if (n_rows < 0 || mask_ld < words) { gt::set_error("gt_subtree_token_mask: bad n_rows / mask_ld (need >= %lld words)", (long long)words); return GT_ERR_ARG; }
    if (n_rows == 0 || words == 0) return GT_OK;
    if (!nodes || !mask_bits) { gt::set_error("gt_subtree_token_mask: null data pointer"); return GT_ERR_ARG; }
    if (n_rows > (int64_t)65535 * gt::kMaskRows) { gt::set_error("gt_subtree_token_mask: too many rows"); return GT_ERR_LIMIT; }
    const gt::PlanView* v = nullptr;
    if (const int rc = gt::resident_plan(t, v); rc != GT_OK) return rc;
    // the grid covers whole mask words: ceil(V/32) of them, kMaskThreads/32 per CTA
    dim3 grid((unsigned)((words * 32 + gt::kMaskThreads - 1) / gt::kMaskThreads), (unsigned)((n_rows + gt::kMaskRows - 1) / gt::kMaskRows));
    gt::subtree_mask_kernel<<<grid, gt::kMaskThreads, 0, static_cast<cudaStream_t>(stream)>>>(*v, nodes, (int)n_rows, mask_bits, mask_ld);
    GT_CUDA(cudaGetLastError());
    return GT_OK;
}

// Checks shared by the two DFA entry points (host only, before any CUDA call); fills the kernels' table / row arguments.
static int dfa_args(const gt_trie* t, const int32_t* delta, int64_t n_states, int64_t ld_delta, const int32_t* states,
                    const int32_t* nodes, int64_t n_rows, const char* what, gt::DfaArgs& A) {
    const int64_t S = t->layout.num_symbols;
    if (n_states < 1 || ld_delta < S || n_rows < 0) {
        gt::set_error("%s: bad n_states / ld_delta / n_rows (n_states=%lld >= 1, ld_delta=%lld >= S=%lld, n_rows=%lld >= 0)", what,
                      (long long)n_states, (long long)ld_delta, (long long)S, (long long)n_rows);
        return GT_ERR_ARG;
    }
    if (n_states > (int64_t)INT32_MAX / ld_delta) {  // the kernels index the table with 32-bit offsets
        gt::set_error("%s: table of %lld x %lld entries reaches 2^31", what, (long long)n_states, (long long)ld_delta);
        return GT_ERR_LIMIT;
    }
    A.delta = delta; A.Q = (int32_t)n_states; A.ld = (int32_t)ld_delta;
    A.states = states; A.nodes = nodes; A.n_rows = (int)std::min<int64_t>(n_rows, INT32_MAX);
    return GT_OK;
}

int gt_dfa_token_mask(const gt_trie* t, const int32_t* delta, int64_t n_states, int64_t ld_delta, const int32_t* states,
                      const int32_t* nodes, int64_t n_rows, uint32_t* mask_bits, int64_t mask_ld, gt_stream stream) {
    if (!t) { gt::set_error("gt_dfa_token_mask: null trie"); return GT_ERR_ARG; }
    if (!delta || !states || !mask_bits) { gt::set_error("gt_dfa_token_mask: null data pointer"); return GT_ERR_ARG; }
    const int64_t words = (t->layout.V + 31) / 32;
    if (mask_ld < words) { gt::set_error("gt_dfa_token_mask: mask_ld %lld < %lld words", (long long)mask_ld, (long long)words); return GT_ERR_ARG; }
    gt::DfaArgs A{};
    const int rc = dfa_args(t, delta, n_states, ld_delta, states, nodes, n_rows, "gt_dfa_token_mask", A);
    if (rc != GT_OK) return rc;
    if (n_rows == 0 || words == 0) return GT_OK;
    if (n_rows > (int64_t)65535 * gt::kDfaRows) { gt::set_error("gt_dfa_token_mask: too many rows"); return GT_ERR_LIMIT; }
    const gt::PlanView* v = nullptr;
    if (const int rc = gt::resident_plan(t, v); rc != GT_OK) return rc;
    // the grid covers whole mask words: ceil(V/32) of them, kDfaThreads/32 per CTA
    dim3 grid((unsigned)((words * 32 + gt::kDfaThreads - 1) / gt::kDfaThreads), (unsigned)((n_rows + gt::kDfaRows - 1) / gt::kDfaRows));
    gt::NvtxRange nv("gt:dfa_mask");
    gt::dfa_mask_kernel<false><<<grid, gt::kDfaThreads, 0, static_cast<cudaStream_t>(stream)>>>(*v, A, mask_bits, mask_ld, words, nullptr);
    GT_CUDA(cudaGetLastError());
    return GT_OK;
}

int gt_dfa_token_logw(const gt_trie* t, const int32_t* delta, const float* logw, int64_t n_states, int64_t ld_delta,
                      const int32_t* states, const int32_t* nodes, int64_t n_rows, float* out, int64_t ld_out, gt_stream stream) {
    if (!t) { gt::set_error("gt_dfa_token_logw: null trie"); return GT_ERR_ARG; }
    if (!delta || !logw || !states || !out) { gt::set_error("gt_dfa_token_logw: null data pointer"); return GT_ERR_ARG; }
    const int64_t V = t->layout.V;
    if (ld_out < V) { gt::set_error("gt_dfa_token_logw: ld_out %lld < V = %lld", (long long)ld_out, (long long)V); return GT_ERR_ARG; }
    gt::DfaArgs A{};
    const int rc = dfa_args(t, delta, n_states, ld_delta, states, nodes, n_rows, "gt_dfa_token_logw", A);
    if (rc != GT_OK) return rc;
    if (n_rows == 0 || V == 0) return GT_OK;
    if (n_rows > (int64_t)65535 * gt::kDfaRows) { gt::set_error("gt_dfa_token_logw: too many rows"); return GT_ERR_LIMIT; }
    const gt::PlanView* v = nullptr;
    if (const int rc = gt::resident_plan(t, v); rc != GT_OK) return rc;
    // the same grid as gt_dfa_token_mask's: ceil(ceil(V/32) * 32 / kDfaThreads) = ceil(V / kDfaThreads)
    dim3 grid((unsigned)((V + gt::kDfaThreads - 1) / gt::kDfaThreads), (unsigned)((n_rows + gt::kDfaRows - 1) / gt::kDfaRows));
    gt::NvtxRange nv("gt:dfa_logw");
    gt::dfa_mask_kernel<true><<<grid, gt::kDfaThreads, 0, static_cast<cudaStream_t>(stream)>>>(*v, A, out, ld_out, 0, logw);
    GT_CUDA(cudaGetLastError());
    return GT_OK;
}

int gt_dfa_advance(const gt_trie* t, const int32_t* delta, int64_t n_states, int64_t ld_delta, const int32_t* states,
                   const int32_t* nodes, const int32_t* tokens, int64_t n_rows, int32_t* states_out, gt_stream stream) {
    if (!t) { gt::set_error("gt_dfa_advance: null trie"); return GT_ERR_ARG; }
    if (!delta || !states || !tokens || !states_out) { gt::set_error("gt_dfa_advance: null data pointer"); return GT_ERR_ARG; }
    gt::DfaArgs A{};
    const int rc = dfa_args(t, delta, n_states, ld_delta, states, nodes, n_rows, "gt_dfa_advance", A);
    if (rc != GT_OK) return rc;
    if (n_rows == 0) return GT_OK;
    if (n_rows > INT32_MAX) { gt::set_error("gt_dfa_advance: too many rows"); return GT_ERR_LIMIT; }
    const gt::PlanView* v = nullptr;
    if (const int rc = gt::resident_plan(t, v); rc != GT_OK) return rc;
    const unsigned grid = (unsigned)((n_rows + gt::kDfaAdvanceThreads - 1) / gt::kDfaAdvanceThreads);
    gt::dfa_advance_kernel<<<grid, gt::kDfaAdvanceThreads, 0, static_cast<cudaStream_t>(stream)>>>(*v, A, tokens, states_out);
    GT_CUDA(cudaGetLastError());
    return GT_OK;
}

}  // extern "C"
