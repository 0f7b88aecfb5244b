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

// kLogw = false: the outputs of a mask kernel are keep-bitmask words; kLogw = true: one float per item and row.
template <bool kLogw>
using MaskOut = std::conditional_t<kLogw, float, uint32_t>;

// The walk of the mask kernels over one item: symbols sy[k0 .. L) outside and the kRows interleaved rows inside, so that
// symbol k is loaded once and steps the state st[g] of every row of the group, which gives each thread kRows
// independent chains of dependent table loads instead of one long chain.  takes(g, k) says whether live row g walks
// symbol k, step(g, q, s) is its transition from state q (-1 on a reject).  kLogw adds (double) logw[q, s] to acc[g]
// before the step, loaded at delta's index ld as an independent load, so the chain of dependent loads does not grow;
// a -inf sum does not stop the walk, only the states decide it.  The thread stops once every row is dead.
template <bool kLogw, int kRows, class Takes, class Step>
__device__ __forceinline__ void walk_item(const int32_t* sy, int k0, int L, int (&st)[kRows], double (&acc)[kRows],
                                          const float* __restrict__ logw, int ld, Takes takes, Step step) {
    for (int k = k0; k < L; ++k) {
        const int s = __ldg(sy + k);
        bool any = false;
#pragma unroll
        for (int g = 0; g < kRows; ++g) {
            if (st[g] >= 0 && takes(g, k)) {
                if constexpr (kLogw) acc[g] += (double)__ldg(logw + st[g] * ld + s);
                st[g] = step(g, st[g], s);
            }
            any |= st[g] >= 0;
        }
        if (!any) break;
    }
}

// The stores of the mask kernels for item i and rows b0 .. b0 + rows - 1 (rows <= kRows).  kLogw = false: one ballot
// word per row, the bit set where st[g] >= 0, words of them written of ld_out per row.  kLogw = true: the first V of
// ld_out floats per row, acc[g] rounded once where st[g] >= 0, else -inf; consecutive threads store consecutive items,
// one coalesced store per warp.  The storing lane is told by i (the CTAs are whole warps): a read of threadIdx.x here
// would merge with the kernel's and lose the range its launch bounds give, which changes the kernels' code.
template <bool kLogw, int kRows>
__device__ __forceinline__ void store_rows(MaskOut<kLogw>* __restrict__ out, int64_t ld_out, int64_t words, int64_t V,
                                           int64_t i, int b0, int rows, const int (&st)[kRows], const double (&acc)[kRows]) {
    if constexpr (kLogw) {
        if (i >= V) return;
#pragma unroll
        for (int g = 0; g < kRows; ++g) {
            if (g >= rows) break;
            out[(size_t)(b0 + g) * ld_out + i] = st[g] >= 0 ? (float)acc[g] : -INFINITY;
        }
    } else {
        const int64_t w = i >> 5;
#pragma unroll
        for (int g = 0; g < kRows; ++g) {
            if (g >= rows) break;
            const unsigned word = __ballot_sync(0xffffffffu, st[g] >= 0);
            if ((i & 31) == 0 && w < words) out[(size_t)(b0 + g) * ld_out + w] = word;
        }
    }
}

// ---- token masks under a byte DFA (gt_dfa_token_mask / gt_dfa_token_logw / gt_dfa_advance) ----------------------------
//
// Row b stands at node n = nodes[b] (the root without nodes) in DFA state q = states[b].  Item i is allowed iff its leaf
// lies under n, q is live (in [0, Q)) and delta walked from q over the item's symbols depth(n) .. len(i)-1 never leaves
// [0, Q).  dfa_mask_kernel: one thread per item, so that a warp's ballot is one mask word (as in subtree_mask_kernel), and
// kDfaRows rows per CTA, interleaved in walk_item.  A row outside the subtree, or with a dead start state, starts dead,
// and row g walks the item from its node's depth on.  The table is read through the read-only path (__ldg): a hot table
// stays in L1 / L2.
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
// written, words unused.  logw has delta's shape.
template <bool kLogw>
__global__ void __launch_bounds__(kDfaThreads) dfa_mask_kernel(PlanView P, DfaArgs A, MaskOut<kLogw>* __restrict__ out, int64_t ld_out,
                                                               int64_t words, const float* __restrict__ logw) {
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
    walk_item<kLogw>(P.item_sym + p0, k0, L, st, acc, logw, A.ld, [&](int g, int k) { return k >= dk[g]; },
                     [&](int, int q, int s) { return dfa_step(A, q, s); });
    store_rows<kLogw>(out, ld_out, words, P.V, i, b0, min(kDfaRows, A.n_rows - b0), st, acc);
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
    int32_t* stack; int32_t* depth;  // [n_rows][cap] and [n_rows]; only the advance writes them
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

// One thread per item, so that a warp's ballot is one mask word as in dfa_mask_kernel, and kPdaRows rows per CTA,
// interleaved in walk_item; each row has its own overlay of GT_PDA_MAX_DEPTH words in local memory (L1-resident, touched
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
// per row, the first V written, words unused.  The parameters are dfa_mask_kernel's, with PdaArgs for DfaArgs.
template <bool kLogw>
__global__ void __launch_bounds__(kPdaThreads) pda_mask_kernel(PlanView P, PdaArgs A, MaskOut<kLogw>* __restrict__ out, int64_t ld_out,
                                                               int64_t words, const float* __restrict__ logw) {
    __shared__ int s_q[kPdaRows], s_d[kPdaRows];
    __shared__ int32_t s_stack[kPdaRows][kPdaMaxDepth];
    const int b0 = blockIdx.y * kPdaRows;
    const int rows = min(kPdaRows, A.A.n_rows - b0);
    if (threadIdx.x < kPdaRows) {
        int q = -1, d = 0;
        if (threadIdx.x < rows) { q = __ldg(A.A.states + b0 + threadIdx.x); d = __ldg(A.depth + b0 + threadIdx.x); }
        if (!pda_row_valid(A, q, d)) { q = -1; d = 0; }
        s_q[threadIdx.x] = q; s_d[threadIdx.x] = d;
    }
    __syncthreads();
    for (int e = threadIdx.x; e < kPdaRows * kPdaMaxDepth; e += kPdaThreads) {
        const int g = e / kPdaMaxDepth, k = e % kPdaMaxDepth;
        if (k < s_d[g]) s_stack[g][k] = __ldg(A.stack + (size_t)(b0 + g) * A.cap + k);
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
    walk_item<kLogw>(P.item_sym + p0, 0, L, st, acc, logw, A.A.ld, [](int, int) { return true; },
                     [&](int g, int q, int s) { return pda_step(A, q, s, ov[g], n[g], s_stack[g], rd[g]); });
    store_rows<kLogw>(out, ld_out, words, P.V, i, b0, rows, st, acc);
}

// One thread per row walks the drawn item from the row's configuration, then writes the overlay over the row's stack
// above the read cursor.  Nothing is written on a reject, so a rejected row keeps its stack and depth.  states and depth
// are read with plain loads: out may alias states, and depth is written in place.
constexpr int kPdaAdvanceThreads = 128;
__global__ void __launch_bounds__(kPdaAdvanceThreads) pda_advance_kernel(PlanView P, PdaArgs A, const int32_t* __restrict__ tokens,
                                                                         int32_t* out) {
    const int b = blockIdx.x * kPdaAdvanceThreads + threadIdx.x;
    if (b >= A.A.n_rows) return;
    const int t = __ldg(tokens + b);
    int q = A.A.states[b], res = -1;
    const int d = A.depth[b];
    if (t >= 0 && t < P.V && pda_row_valid(A, q, d)) {
        int32_t* row_stack = A.stack + (size_t)b * A.cap;
        int ov[kPdaMaxDepth], n = 0, rd = d;
        const int p1 = __ldg(P.item_sym_ptr + t + 1);
        for (int p = __ldg(P.item_sym_ptr + t); p < p1 && q >= 0; ++p) q = pda_step(A, q, __ldg(P.item_sym + p), ov, n, row_stack, rd);
        if (q >= 0) {
            for (int k = 0; k < n; ++k) row_stack[rd + k] = ov[k];
            A.depth[b] = rd + n;
        }
        res = q;
    }
    out[b] = res;
}

}  // namespace gt

// Checks shared by the automaton entry points (host only, before any CUDA call); fills the kernels' table / row arguments.
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

// Checks shared by the three PDA entry points: dfa_args, then the stack capacity.
static int pda_args(const gt_trie* t, const int32_t* delta, const int32_t* push, int64_t n_states, int64_t ld_delta,
                    const int32_t* states, const int32_t* stack, int64_t stack_ld, const int32_t* depth, int64_t n_rows,
                    const char* what, gt::PdaArgs& A) {
    if (const int rc = dfa_args(t, delta, n_states, ld_delta, states, nullptr, n_rows, what, A.A); rc != GT_OK) return rc;
    if (stack_ld < 1) { gt::set_error("%s: stack_ld %lld < 1", what, (long long)stack_ld); return GT_ERR_ARG; }
    if (stack_ld > GT_PDA_MAX_DEPTH) {
        gt::set_error("%s: stack_ld %lld > GT_PDA_MAX_DEPTH = %d", what, (long long)stack_ld, GT_PDA_MAX_DEPTH);
        return GT_ERR_LIMIT;
    }
    A.push = push; A.cap = (int)stack_ld;
    A.stack = const_cast<int32_t*>(stack); A.depth = const_cast<int32_t*>(depth);  // the mask kernels only read them
    return GT_OK;
}

// The first checks of every automaton entry point: a null trie, then a null data pointer.
static int null_checks(const char* what, const gt_trie* t, bool null_ptr) {
    if (!t) { gt::set_error("%s: null trie", what); return GT_ERR_ARG; }
    if (null_ptr) { gt::set_error("%s: null data pointer", what); return GT_ERR_ARG; }
    return GT_OK;
}

// The last checks of every automaton entry point before its launch: more than max_rows rows, then the resident plan.
static int plan_for_rows(const char* what, const gt_trie* t, int64_t n_rows, int64_t max_rows, const gt::PlanView*& v) {
    if (n_rows > max_rows) { gt::set_error("%s: too many rows", what); return GT_ERR_LIMIT; }
    return gt::resident_plan(t, v);
}

// The four mask and log-weight calls.  The checks, in order: null trie, null data pointers, the output row width
// (ld_out >= ceil(V/32) words of a keep-bitmask, or >= V floats), args (dfa_args or pda_args, which fill the kernel's
// arguments), no rows or no items, rows beyond the grid's 65535 x rows_per_cta, the resident plan.  Then kernel, under
// the NVTX range `range`, with one thread per item: ceil(V / threads) CTAs per row group, which cover the ceil(V/32)
// mask words as threads is a multiple of 32.
template <class Args, class Out, class ArgsFn>
static int mask_call(const char* what, const char* range, void (*kernel)(gt::PlanView, Args, Out*, int64_t, int64_t, const float*),
                     int threads, int rows_per_cta, const gt_trie* t, bool null_ptr, int64_t n_rows, Out* out, int64_t ld_out,
                     const float* logw, gt_stream stream, ArgsFn args) {
    constexpr bool kLogw = std::is_same_v<Out, float>;
    if (const int rc = null_checks(what, t, null_ptr); rc != GT_OK) return rc;
    const int64_t V = t->layout.V, words = (V + 31) / 32;
    if (kLogw && ld_out < V) { gt::set_error("%s: ld_out %lld < V = %lld", what, (long long)ld_out, (long long)V); return GT_ERR_ARG; }
    if (!kLogw && ld_out < words) { gt::set_error("%s: mask_ld %lld < %lld words", what, (long long)ld_out, (long long)words); return GT_ERR_ARG; }
    Args A{};
    if (const int rc = args(A); rc != GT_OK) return rc;
    if (n_rows == 0 || V == 0) return GT_OK;
    const gt::PlanView* v = nullptr;
    if (const int rc = plan_for_rows(what, t, n_rows, (int64_t)65535 * rows_per_cta, v); rc != GT_OK) return rc;
    const dim3 grid((unsigned)((V + threads - 1) / threads), (unsigned)((n_rows + rows_per_cta - 1) / rows_per_cta));
    gt::NvtxRange nv(range);
    kernel<<<grid, threads, 0, static_cast<cudaStream_t>(stream)>>>(*v, A, out, ld_out, kLogw ? 0 : words, logw);
    GT_CUDA(cudaGetLastError());
    return GT_OK;
}

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

int gt_dfa_token_mask(const gt_trie* t, const int32_t* delta, int64_t n_states, int64_t ld_delta, const int32_t* states,
                      const int32_t* nodes, int64_t n_rows, uint32_t* mask_bits, int64_t mask_ld, gt_stream stream) {
    return mask_call("gt_dfa_token_mask", "gt:dfa_mask", gt::dfa_mask_kernel<false>, gt::kDfaThreads, gt::kDfaRows, t,
                     !delta || !states || !mask_bits, n_rows, mask_bits, mask_ld, nullptr, stream, [&](gt::DfaArgs& A) {
        return dfa_args(t, delta, n_states, ld_delta, states, nodes, n_rows, "gt_dfa_token_mask", A);
    });
}

int gt_dfa_token_logw(const gt_trie* t, const int32_t* delta, const float* logw, int64_t n_states, int64_t ld_delta,
                      const int32_t* states, const int32_t* nodes, int64_t n_rows, float* out, int64_t ld_out, gt_stream stream) {
    return mask_call("gt_dfa_token_logw", "gt:dfa_logw", gt::dfa_mask_kernel<true>, gt::kDfaThreads, gt::kDfaRows, t,
                     !delta || !logw || !states || !out, n_rows, out, ld_out, logw, stream, [&](gt::DfaArgs& A) {
        return dfa_args(t, delta, n_states, ld_delta, states, nodes, n_rows, "gt_dfa_token_logw", A);
    });
}

int gt_dfa_advance(const gt_trie* t, const int32_t* delta, int64_t n_states, int64_t ld_delta, const int32_t* states,
                   const int32_t* nodes, const int32_t* tokens, int64_t n_rows, int32_t* states_out, gt_stream stream) {
    const char* what = "gt_dfa_advance";
    if (const int rc = null_checks(what, t, !delta || !states || !tokens || !states_out); rc != GT_OK) return rc;
    gt::DfaArgs A{};
    if (const int rc = dfa_args(t, delta, n_states, ld_delta, states, nodes, n_rows, what, A); rc != GT_OK || n_rows == 0) return rc;
    const gt::PlanView* v = nullptr;
    if (const int rc = plan_for_rows(what, t, n_rows, INT32_MAX, v); rc != GT_OK) return rc;
    const unsigned grid = (unsigned)((n_rows + gt::kDfaAdvanceThreads - 1) / gt::kDfaAdvanceThreads);
    gt::dfa_advance_kernel<<<grid, gt::kDfaAdvanceThreads, 0, static_cast<cudaStream_t>(stream)>>>(*v, A, tokens, states_out);
    GT_CUDA(cudaGetLastError());
    return GT_OK;
}

int gt_pda_token_mask(const gt_trie* t, const int32_t* delta, const int32_t* push, int64_t n_states, int64_t ld_delta,
                      const int32_t* states, const int32_t* stack, int64_t stack_ld, const int32_t* depth, int64_t n_rows,
                      uint32_t* mask_bits, int64_t mask_ld, gt_stream stream) {
    return mask_call("gt_pda_token_mask", "gt:pda_mask", gt::pda_mask_kernel<false>, gt::kPdaThreads, gt::kPdaRows, t,
                     !delta || !push || !states || !stack || !depth || !mask_bits, n_rows, mask_bits, mask_ld, nullptr, stream,
                     [&](gt::PdaArgs& A) {
        return pda_args(t, delta, push, n_states, ld_delta, states, stack, stack_ld, depth, n_rows, "gt_pda_token_mask", A);
    });
}

int gt_pda_token_logw(const gt_trie* t, const int32_t* delta, const int32_t* push, const float* logw, int64_t n_states,
                      int64_t ld_delta, const int32_t* states, const int32_t* stack, int64_t stack_ld, const int32_t* depth,
                      int64_t n_rows, float* out, int64_t ld_out, gt_stream stream) {
    return mask_call("gt_pda_token_logw", "gt:pda_logw", gt::pda_mask_kernel<true>, gt::kPdaThreads, gt::kPdaRows, t,
                     !delta || !push || !logw || !states || !stack || !depth || !out, n_rows, out, ld_out, logw, stream,
                     [&](gt::PdaArgs& A) {
        return pda_args(t, delta, push, n_states, ld_delta, states, stack, stack_ld, depth, n_rows, "gt_pda_token_logw", A);
    });
}

int gt_pda_advance(const gt_trie* t, const int32_t* delta, const int32_t* push, int64_t n_states, int64_t ld_delta,
                   const int32_t* states, int32_t* stack, int64_t stack_ld, int32_t* depth, const int32_t* tokens,
                   int64_t n_rows, int32_t* states_out, gt_stream stream) {
    const char* what = "gt_pda_advance";
    if (const int rc = null_checks(what, t, !delta || !push || !states || !stack || !depth || !tokens || !states_out); rc != GT_OK) return rc;
    gt::PdaArgs A{};
    const int rc = pda_args(t, delta, push, n_states, ld_delta, states, stack, stack_ld, depth, n_rows, what, A);
    if (rc != GT_OK || n_rows == 0) return rc;
    const gt::PlanView* v = nullptr;
    if (const int rc = plan_for_rows(what, t, n_rows, INT32_MAX, v); rc != GT_OK) return rc;
    const unsigned grid = (unsigned)((n_rows + gt::kPdaAdvanceThreads - 1) / gt::kPdaAdvanceThreads);
    gt::NvtxRange nv("gt:pda_advance");
    gt::pda_advance_kernel<<<grid, gt::kPdaAdvanceThreads, 0, static_cast<cudaStream_t>(stream)>>>(*v, A, tokens, states_out);
    GT_CUDA(cudaGetLastError());
    return GT_OK;
}

}  // extern "C"
