// sm_100a kernels for per-row token masks over the trie: the items under a node (gt_subtree_token_mask), the items a
// byte DFA accepts from there (gt_dfa_token_mask), their log-weights under a weighted byte DFA (gt_dfa_token_logw), and
// the DFA state after a drawn token (gt_dfa_advance); the items a byte pushdown automaton accepts from a row's
// configuration at the root (gt_pda_token_mask), their log-weights under a weighted one (gt_pda_token_logw), and the
// configuration after a drawn token (gt_pda_advance).
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

// ---- token masks under a byte-level pushdown automaton (gt_pda_token_mask / gt_pda_token_logw / gt_pda_advance) --------
//
// Row b stands at the root in configuration (states[b], stack[b, 0 .. depth[b]-1]).  A walk over an item's symbols pushes
// onto a private overlay and pops from it first; only once the overlay is empty does a pop read the row's stack, below a
// read cursor that starts at depth[b].  The walk therefore never writes the row's stack, and the configuration after
// the item is row stack[0 .. cursor) followed by the overlay.  A push past stack_ld rejects, so the overlay never holds
// more than stack_ld - depth[b] <= GT_PDA_MAX_DEPTH entries, whatever the item's length.
constexpr int kPdaMaxDepth = GT_PDA_MAX_DEPTH;

struct PdaArgs {
    DfaArgs A;  // delta, Q, ld, states, n_rows (nodes is null: every row at the root)
    const int32_t* push;  // push[q * ld + s], read where delta[q, s] is a move
    int cap;  // stack_ld: the row stride of the stacks and every row's capacity
};

// A row is valid iff its state lies in [0, Q) and its depth in [0, cap].
__device__ __forceinline__ bool pda_row_valid(const PdaArgs& A, int q, int d) {
    return q >= 0 && q < A.A.Q && d >= 0 && d <= A.cap;
}

// One symbol of a walk from q: a move (with an optional push onto the overlay ov[0 .. n)) or a pop (from the overlay,
// else from row_stack below the cursor rd).  Returns the next state, or -1 on any reject.
__device__ __forceinline__ int pda_step(const PdaArgs& A, int q, int s, int* ov, int& n, const int32_t* row_stack, int& rd) {
    const int nq = dfa_step(A.A, q, s);
    if (nq >= 0) {
        const int pu = __ldg(A.push + q * A.A.ld + s);
        if (pu < 0) return nq;
        if (pu >= A.A.Q || rd + n >= A.cap) return -1;
        ov[n++] = pu;
        return nq;
    }
    if (__ldg(A.A.delta + q * A.A.ld + s) != GT_PDA_POP) return -1;
    const int v = n > 0 ? ov[--n] : rd > 0 ? row_stack[--rd] : -1;
    return (unsigned)v < (unsigned)A.A.Q ? v : -1;
}

// One thread per item, kPdaRows rows per CTA, so that a warp's ballot is one mask word as in dfa_mask_kernel.  As there,
// the loop runs over the item's symbols outside and the rows inside, which gives each thread kPdaRows independent chains
// of dependent table loads; each row has its own overlay of GT_PDA_MAX_DEPTH words in local memory (L1-resident, touched
// only by pushes and pops).  The rows' stacks are staged in shared memory, where every item of the CTA reads them.
// Rows per CTA, measured on B200 (DESIGN section 5.14): at 128k tokens 4 interleaved rows take 1-18 % less time than 8
// and 3-17 % less than 2; walking 8 rows one after another with a single overlay took 10-19 % more.
#ifndef GT_PDA_ROWS
#define GT_PDA_ROWS 4
#endif
constexpr int kPdaThreads = 256, kPdaRows = GT_PDA_ROWS;

// kLogw = false (gt_pda_token_mask): out holds keep-bitmask words, ld_out words per row, words of them written.
// kLogw = true (gt_pda_token_logw): out[b, i] is the fp64 sum of logw[q_k, s_k] over the walked transitions (moves,
// pushes and pops alike), in increasing k and rounded once to fp32, where the bit would be set, else -inf; ld_out floats
// per row, the first V written, words unused.  As in dfa_mask_kernel, logw is loaded at delta's index as an independent
// load, and a -inf accumulator does not stop the walk.  logw is a trailing parameter, so the bits instantiation keeps
// its parameter offsets.
template <bool kLogw>
__global__ void __launch_bounds__(kPdaThreads) pda_mask_kernel(PlanView P, PdaArgs A, const int32_t* __restrict__ stack,
                                                               const int32_t* __restrict__ depth,
                                                               std::conditional_t<kLogw, float, uint32_t>* __restrict__ out,
                                                               int64_t ld_out, int64_t words, const float* __restrict__ logw) {
    __shared__ int s_q[kPdaRows], s_d[kPdaRows];
    __shared__ int32_t s_stack[kPdaRows][kPdaMaxDepth];
    const int b0 = blockIdx.y * kPdaRows;
    const int rows = min(kPdaRows, A.A.n_rows - b0);
    if (threadIdx.x < kPdaRows) {
        int q = -1, d = 0;
        if (threadIdx.x < rows) { q = __ldg(A.A.states + b0 + threadIdx.x); d = __ldg(depth + b0 + threadIdx.x); }
        if (!pda_row_valid(A, q, d)) { q = -1; d = 0; }
        s_q[threadIdx.x] = q; s_d[threadIdx.x] = d;
    }
    __syncthreads();
    for (int e = threadIdx.x; e < kPdaRows * kPdaMaxDepth; e += kPdaThreads) {
        const int g = e / kPdaMaxDepth, k = e % kPdaMaxDepth;
        if (k < s_d[g]) s_stack[g][k] = __ldg(stack + (size_t)(b0 + g) * A.cap + k);
    }
    const int64_t i = (int64_t)blockIdx.x * kPdaThreads + threadIdx.x;
    int p0 = 0, L = 0;
    if (i < P.V) {
        p0 = __ldg(P.item_sym_ptr + i);
        L = __ldg(P.item_sym_ptr + i + 1) - p0;
    }
    __syncthreads();
    int st[kPdaRows], n[kPdaRows], rd[kPdaRows];
    int ov[kPdaRows][kPdaMaxDepth];
    double acc[kPdaRows] = {};
#pragma unroll
    for (int g = 0; g < kPdaRows; ++g) {
        st[g] = i < P.V ? s_q[g] : -1;
        n[g] = 0;
        rd[g] = s_d[g];
    }
    const int32_t* sy = P.item_sym + p0;
    for (int k = 0; k < L; ++k) {
        const int s = __ldg(sy + k);
        bool any = false;
#pragma unroll
        for (int g = 0; g < kPdaRows; ++g) {
            if (st[g] >= 0) {
                if constexpr (kLogw) acc[g] += (double)__ldg(logw + st[g] * A.A.ld + s);
                st[g] = pda_step(A, st[g], s, ov[g], n[g], s_stack[g], rd[g]);
            }
            any |= st[g] >= 0;
        }
        if (!any) break;
    }
    if constexpr (kLogw) {
        if (i >= P.V) return;
#pragma unroll
        for (int g = 0; g < kPdaRows; ++g) {  // consecutive threads store consecutive items: one coalesced store per warp
            if (g >= rows) break;
            out[(size_t)(b0 + g) * ld_out + i] = st[g] >= 0 ? (float)acc[g] : -INFINITY;
        }
    } else {
        const int64_t w = i >> 5;
#pragma unroll
        for (int g = 0; g < kPdaRows; ++g) {
            if (g >= rows) break;
            const unsigned word = __ballot_sync(0xffffffffu, st[g] >= 0);
            if ((threadIdx.x & 31) == 0 && w < words) out[(size_t)(b0 + g) * ld_out + w] = word;
        }
    }
}

// One thread per row walks the drawn item from the row's configuration, then writes the overlay over the row's stack
// above the read cursor.  Nothing is written on a reject, so a rejected row keeps its stack and depth.  states and depth
// are read with plain loads: out may alias states, and depth is written in place.
constexpr int kPdaAdvanceThreads = 128;
__global__ void __launch_bounds__(kPdaAdvanceThreads) pda_advance_kernel(PlanView P, PdaArgs A, int32_t* __restrict__ stack,
                                                                         int32_t* __restrict__ depth,
                                                                         const int32_t* __restrict__ tokens,
                                                                         int32_t* out) {
    const int b = blockIdx.x * kPdaAdvanceThreads + threadIdx.x;
    if (b >= A.A.n_rows) return;
    const int t = __ldg(tokens + b);
    int q = A.A.states[b], res = -1;
    const int d = depth[b];
    if (t >= 0 && t < P.V && pda_row_valid(A, q, d)) {
        int32_t* row_stack = stack + (size_t)b * A.cap;
        int ov[kPdaMaxDepth], n = 0, rd = d;
        const int p1 = __ldg(P.item_sym_ptr + t + 1);
        for (int p = __ldg(P.item_sym_ptr + t); p < p1 && q >= 0; ++p) q = pda_step(A, q, __ldg(P.item_sym + p), ov, n, row_stack, rd);
        if (q >= 0) {
            for (int k = 0; k < n; ++k) row_stack[rd + k] = ov[k];
            depth[b] = rd + n;
        }
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

// Checks shared by the three PDA entry points after their null-pointer checks: dfa_args, then the stack capacity.
static int pda_args(const gt_trie* t, const int32_t* delta, const int32_t* push, int64_t n_states, int64_t ld_delta,
                    const int32_t* states, int64_t stack_ld, int64_t n_rows, const char* what, gt::PdaArgs& A) {
    if (const int rc = dfa_args(t, delta, n_states, ld_delta, states, nullptr, n_rows, what, A.A); rc != GT_OK) return rc;
    if (stack_ld < 1) { gt::set_error("%s: stack_ld %lld < 1", what, (long long)stack_ld); return GT_ERR_ARG; }
    if (stack_ld > GT_PDA_MAX_DEPTH) {
        gt::set_error("%s: stack_ld %lld > GT_PDA_MAX_DEPTH = %d", what, (long long)stack_ld, GT_PDA_MAX_DEPTH);
        return GT_ERR_LIMIT;
    }
    A.push = push; A.cap = (int)stack_ld;
    return GT_OK;
}

int gt_pda_token_mask(const gt_trie* t, const int32_t* delta, const int32_t* push, int64_t n_states, int64_t ld_delta,
                      const int32_t* states, const int32_t* stack, int64_t stack_ld, const int32_t* depth, int64_t n_rows,
                      uint32_t* mask_bits, int64_t mask_ld, gt_stream stream) {
    if (!t) { gt::set_error("gt_pda_token_mask: null trie"); return GT_ERR_ARG; }
    if (!delta || !push || !states || !stack || !depth || !mask_bits) { gt::set_error("gt_pda_token_mask: null data pointer"); return GT_ERR_ARG; }
    const int64_t words = (t->layout.V + 31) / 32;
    if (mask_ld < words) { gt::set_error("gt_pda_token_mask: mask_ld %lld < %lld words", (long long)mask_ld, (long long)words); return GT_ERR_ARG; }
    gt::PdaArgs A{};
    const int rc = pda_args(t, delta, push, n_states, ld_delta, states, stack_ld, n_rows, "gt_pda_token_mask", A);
    if (rc != GT_OK) return rc;
    if (n_rows == 0 || words == 0) return GT_OK;
    if (n_rows > (int64_t)65535 * gt::kPdaRows) { gt::set_error("gt_pda_token_mask: too many rows"); return GT_ERR_LIMIT; }
    const gt::PlanView* v = nullptr;
    if (const int rc = gt::resident_plan(t, v); rc != GT_OK) return rc;
    dim3 grid((unsigned)((words * 32 + gt::kPdaThreads - 1) / gt::kPdaThreads), (unsigned)((n_rows + gt::kPdaRows - 1) / gt::kPdaRows));
    gt::NvtxRange nv("gt:pda_mask");
    gt::pda_mask_kernel<false><<<grid, gt::kPdaThreads, 0, static_cast<cudaStream_t>(stream)>>>(*v, A, stack, depth, mask_bits, mask_ld,
                                                                                               words, nullptr);
    GT_CUDA(cudaGetLastError());
    return GT_OK;
}

int gt_pda_token_logw(const gt_trie* t, const int32_t* delta, const int32_t* push, const float* logw, int64_t n_states,
                      int64_t ld_delta, const int32_t* states, const int32_t* stack, int64_t stack_ld, const int32_t* depth,
                      int64_t n_rows, float* out, int64_t ld_out, gt_stream stream) {
    if (!t) { gt::set_error("gt_pda_token_logw: null trie"); return GT_ERR_ARG; }
    if (!delta || !push || !logw || !states || !stack || !depth || !out) { gt::set_error("gt_pda_token_logw: null data pointer"); return GT_ERR_ARG; }
    const int64_t V = t->layout.V;
    if (ld_out < V) { gt::set_error("gt_pda_token_logw: ld_out %lld < V = %lld", (long long)ld_out, (long long)V); return GT_ERR_ARG; }
    gt::PdaArgs A{};
    const int rc = pda_args(t, delta, push, n_states, ld_delta, states, stack_ld, n_rows, "gt_pda_token_logw", A);
    if (rc != GT_OK) return rc;
    if (n_rows == 0 || V == 0) return GT_OK;
    if (n_rows > (int64_t)65535 * gt::kPdaRows) { gt::set_error("gt_pda_token_logw: too many rows"); return GT_ERR_LIMIT; }
    const gt::PlanView* v = nullptr;
    if (const int rc = gt::resident_plan(t, v); rc != GT_OK) return rc;
    // the same grid as gt_pda_token_mask's: ceil(ceil(V/32) * 32 / kPdaThreads) = ceil(V / kPdaThreads)
    dim3 grid((unsigned)((V + gt::kPdaThreads - 1) / gt::kPdaThreads), (unsigned)((n_rows + gt::kPdaRows - 1) / gt::kPdaRows));
    gt::NvtxRange nv("gt:pda_logw");
    gt::pda_mask_kernel<true><<<grid, gt::kPdaThreads, 0, static_cast<cudaStream_t>(stream)>>>(*v, A, stack, depth, out, ld_out, 0, logw);
    GT_CUDA(cudaGetLastError());
    return GT_OK;
}

int gt_pda_advance(const gt_trie* t, const int32_t* delta, const int32_t* push, int64_t n_states, int64_t ld_delta,
                   const int32_t* states, int32_t* stack, int64_t stack_ld, int32_t* depth, const int32_t* tokens,
                   int64_t n_rows, int32_t* states_out, gt_stream stream) {
    if (!t) { gt::set_error("gt_pda_advance: null trie"); return GT_ERR_ARG; }
    if (!delta || !push || !states || !stack || !depth || !tokens || !states_out) { gt::set_error("gt_pda_advance: null data pointer"); return GT_ERR_ARG; }
    gt::PdaArgs A{};
    const int rc = pda_args(t, delta, push, n_states, ld_delta, states, stack_ld, n_rows, "gt_pda_advance", A);
    if (rc != GT_OK) return rc;
    if (n_rows == 0) return GT_OK;
    if (n_rows > INT32_MAX) { gt::set_error("gt_pda_advance: too many rows"); return GT_ERR_LIMIT; }
    const gt::PlanView* v = nullptr;
    if (const int rc = gt::resident_plan(t, v); rc != GT_OK) return rc;
    const unsigned grid = (unsigned)((n_rows + gt::kPdaAdvanceThreads - 1) / gt::kPdaAdvanceThreads);
    gt::NvtxRange nv("gt:pda_advance");
    gt::pda_advance_kernel<<<grid, gt::kPdaAdvanceThreads, 0, static_cast<cudaStream_t>(stream)>>>(*v, A, stack, depth, tokens, states_out);
    GT_CUDA(cudaGetLastError());
    return GT_OK;
}

}  // extern "C"
