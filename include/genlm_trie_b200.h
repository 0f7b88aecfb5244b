/*
 * genlm_trie_b200.h -- C ABI of the B200-native token-character-trie mass path.
 *
 * This is the drop-in boundary for genlm-backend's trie hot path.  The reference
 * has no FFI of its own (it is Python over numba / torch library kernels), so
 * every entry point below names the reference Python code it replaces
 * (paths relative to the genlm-backend repository root):
 *
 *   gt_build / gt_export_*      genlm/backend/trie/base.py:13-122   (TokenCharacterTrie.__init__, _rename,
 *                                                                    _order, _order_full)
 *   gt_export_reachability      genlm/backend/trie/parallel.py:21-64 (_build_parent_map,
 *                                                                    _build_reachability_matrix)
 *   gt_weight_reduce            ops & GT_OP_SUM:  genlm/backend/trie/base.py:346-368   (_update_trie_numba_sum)
 *                                                 genlm/backend/trie/parallel.py:92-103 (batch_weight_sum: sparse.mm)
 *                               ops & GT_OP_MAX:  genlm/backend/trie/base.py:371-393   (_update_trie_numba_max)
 *                                                 genlm/backend/trie/parallel.py:120-145 (batch_weight_max:
 *                                                 scatter_reduce amax)
 *   gt_lse_sample               README.md:82-91 / genlm/backend/llm/base.py:131-146
 *                               (masked logsumexp + multinomial of the SMC particle step)
 *   gt_gather_nodes             genlm/backend/trie/parallel.py:103,145 (the .cpu().numpy() of the whole slab)
 *   gt_subtree_token_mask       genlm/backend/trie/parallel.py:33-64 (a column of the reachability matrix)
 *   gt_child_masses             genlm/backend/trie/parallel.py:92-103 (batch_weight_sum) followed by indexing
 *                               children(node) of the result on the host: the next-symbol masses of a
 *                               character-level sampler, without the [B, N] slab
 *   gt_child_sample             the same, plus one categorical draw of the next symbol per row
 *   gt_symbol_masses            the child masses laid out by symbol (column S = end of token), aligned with the
 *                               per-symbol weight vector of a byte-level potential
 *   gt_symbol_sample            the draw of the next symbol in proportion to mass(child) * weight(symbol), with the
 *                               weighted normaliser (the particle's weight increment)
 *   gt_child_masses_masked, gt_child_sample_masked, gt_symbol_masses_masked, gt_symbol_sample_masked
 *                               the same four over the tokens a keep-bitmask allows: what a caller gets today by
 *                               torch.where(keep, ws, 0) over the whole [B, V] rows before the unmasked call; drawn
 *                               symbol by symbol from the root, the masked token draw of README.md:82-91
 *   gt_dfa_token_mask           the host-side walk of every token's bytes through a constraint's automaton that a
 *                               constrained token sampler does to build the mask of README.md:82-91's masked draw
 *   gt_dfa_token_logw           the same walk through a weighted automaton, summing each token's transition
 *                               log-weights: the additive mask of a soft byte-level potential
 *   gt_dfa_advance              the host-side tracking of each particle's automaton state over the drawn token
 *   gt_pda_token_mask           the host-side walk of every token's bytes through a parser (a pushdown automaton
 *                               with a stack per particle) for a nested constraint such as JSON
 *   gt_pda_token_logw           the same walk through a weighted pushdown automaton (a probabilistic grammar, a
 *                               nesting penalty), summing each token's transition log-weights: an additive mask
 *   gt_pda_advance             the host-side tracking of each particle's parser state and stack over the drawn token
 *   gt_resample                 the effective sample size of each particle group and, below a threshold, the
 *                               multinomial, stratified or systematic ancestors an SMC driver draws on the host
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on failure; gt_last_error() returns a
 *     thread-local message for the last failure on the calling thread;
 *   - plain pointers and sizes only, no torch / numpy types;
 *   - all device pointers are caller-owned; nothing is allocated per call; every launch goes to the
 *     caller-supplied stream (a cudaStream_t passed as void*); no hidden synchronisation (gt_upload, which
 *     runs once per trie and device, is the exception: it returns when the metadata is resident);
 *   - node ids, leaf ids and row layout are exactly the reference's (post-order ids, root = N-1).
 */
#ifndef GENLM_TRIE_B200_H
#define GENLM_TRIE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct gt_trie gt_trie; /* opaque: host layout + per-device resident metadata */
typedef void* gt_stream;        /* cudaStream_t */

/* ---- status ------------------------------------------------------------------------------- */
#define GT_OK 0
#define GT_ERR_ARG 1     /* bad argument (null pointer, negative size, row stride too small ...) */
#define GT_ERR_CUDA 2    /* a CUDA runtime call failed; message has the cudaError string */
#define GT_ERR_STATE 3   /* trie not uploaded to the current device, workspace too small ... */
#define GT_ERR_LIMIT 4   /* vocabulary exceeds a compiled-in limit */

const char* gt_last_error(void);
int gt_version(void);

/* ---- builder (host only; works without a GPU) --------------------------------------------- */

/* Build the trie over n_tokens items.  Item i spells symbols[offsets[i] .. offsets[i+1]).
 * Symbols 0..255 are bytes; symbols >= 256 stand for non-byte edge labels (the reference iterates
 * arbitrary iterables, base.py:45-48).  Each item gets its own leaf (base.py:55-61), so duplicate
 * byte strings are legal here; the (bytes, token_id) duplicate check of base.py:63-64 is the
 * caller's job.  Node ids are the reference's post-order numbering (base.py:80-83, 236-247). */
int gt_build(const int32_t* symbols, const int64_t* offsets, int64_t n_tokens, gt_trie** out);
void gt_free(gt_trie* t);

int64_t gt_num_tokens(const gt_trie* t); /* V = len(decode)                      */
int64_t gt_num_nodes(const gt_trie* t);  /* N = len(children)                    */
int64_t gt_root(const gt_trie* t);       /* == N-1                               */
int64_t gt_num_reach(const gt_trie* t);  /* nnz of the leaf x node reachability  */
int64_t gt_max_depth(const gt_trie* t);

/* Copy layout arrays out (any pointer may be NULL to skip it).
 *   leaf_node[V]     node id of the leaf of item i            (idx_to_leaf[:,1], base.py:115-117)
 *   parent[N]        parent node id, -1 for the root          (parallel.py:21-31)
 *   edge_label[N]    label of the edge into the node: symbol >= 0, or -1-i for the leaf of item i,
 *                    INT32_MIN for the root                   (keys of children[..], base.py:50-58)
 *   child_ptr[N+1], child_idx[N-1]   children CSR in insertion order (== ascending id order, which
 *                    is what jump[] holds, base.py:120-122)
 *   perm[V]          DFS leaf rank -> item position
 *   lo[N], hi[N]     every node's leaves are DFS ranks [lo, hi) */
int gt_export_layout(const gt_trie* t, int32_t* leaf_node, int32_t* parent, int32_t* edge_label,
                     int32_t* child_ptr, int32_t* child_idx, int32_t* perm, int32_t* lo, int32_t* hi);

/* (row, col) pairs of the reachability matrix in the reference's order: for item i its leaf, then
 * each ancestor up to the root (parallel.py:42-54).  Arrays of gt_num_reach() entries. */
int gt_export_reachability(const gt_trie* t, int64_t* rows, int64_t* cols);

/* ---- device plan -------------------------------------------------------------------------- */

/* Build the tile plan (once) and make its metadata resident on `device`.  Idempotent per device. */
int gt_upload(gt_trie* t, int device);

typedef struct gt_plan_info {
    int64_t n_tokens, n_nodes;
    int32_t tile_leaves;     /* T: DFS-ordered leaves per tile                       */
    int32_t n_tiles;
    int32_t rows_per_item;   /* R: fp32 rows that share a work item (16-byte value slots; fp64: R/2) */
    int32_t permute_unit;    /* vocabulary positions per permute work unit           */
    int32_t n_span;          /* nodes whose leaf range crosses a tile boundary       */
    int32_t max_levels;      /* levels of the per-tile aligned-block pyramid         */
    int64_t span_terms;      /* per-tile pieces the spanning nodes are reduced from  */
    int32_t max_tile_values; /* largest per-tile value array (leaf + pyramid + range slots) */
    int32_t reserved;
    int64_t staged_slots;    /* value slots per row group of the staging buffer (n_tiles * tile_leaves) */
    int64_t meta_bytes;      /* device-resident metadata                              */
} gt_plan_info;
int gt_get_plan_info(const gt_trie* t, gt_plan_info* info);

/* Host-only: build the tile plan without touching a device (gt_upload calls this with its default when
 * no plan exists yet).  tile_leaves: 1024 or 2048, 0 for the default.  Fails if a plan already exists with a
 * different tile size. */
int gt_plan(gt_trie* t, int32_t tile_leaves);

/* Host-only introspection of the plan arrays, used by the CPU tests that emulate the kernels' data flow.
 * `name` is one of: leaf_dest ell_chunk_ptr ell_desc ell_terms ell_row_ptr tile_node_lo
 * node_slot piece_ptr piece_slot piece_idx span_node span_pp.  Returns the element count (or -1), and copies
 * min(count, capacity) elements into dst when dst != NULL.  elem_size receives 2 or 4. */
int64_t gt_export_plan_array(const gt_trie* t, const char* name, void* dst, int64_t capacity, int32_t* elem_size);

/* Profiling aid.  With GT_TRACE=1 in the environment at gt_upload() time, the tile kernel stamps the SM clock at
 * its pipeline events per (CTA, item); this copies the stamps out (dims = {ctas, items, events}) and clears them.
 * Returns the element count, or -1 when no trace buffer exists.  tools/trace_tile.py prints the phase durations. */
int64_t gt_debug_read_trace(const gt_trie* t, int device, long long* dst, int64_t capacity, int32_t dims[3]);

/* Caller-owned scratch for batches of up to max_rows rows: the staging buffer of one chunk (at most 64 rows: it
 * should stay L2-resident between the permute and the tile kernel) plus the spanning-node pieces of min(max_rows, 1024)
 * rows, so that the span kernel runs once per 1,024 rows.  Larger batches, or a smaller workspace, are processed in
 * as many chunks / span groups as it takes (any size that holds one row works).  One call at a time may use a
 * workspace: calls that share one must be ordered (same stream).  The pointer must be 256-byte aligned. */
size_t gt_workspace_bytes(const gt_trie* t, int64_t max_rows);

/* ---- trie mass kernels -------------------------------------------------------------------- */

#define GT_FLAG_LOG_INPUT 1u /* rows hold log-weights: exp() is fused into the load (-inf -> 0) */
/* The rows are given in DFS leaf order: element r of a row is the weight of item perm[r] (gt_export_layout), e.g. because
 * the producer of the rows -- an LM head whose output rows were permuted once at load time -- emits them that way.  The
 * permute kernel then has nothing to scatter: it interleaves row groups with coalesced stores (4.2 us instead of
 * 15.3 us for 64 rows x 128k tokens).  Results are identical to those for the same weights in vocabulary order. */
#define GT_FLAG_DFS_ORDER 2u
/* Profiling aids: restrict a call to some phases (default: all).  Used by bench.py to time one kernel in
 * isolation with CUDA events; results are only complete when all phases have run in order. */
#define GT_FLAG_PHASE_PERMUTE 0x100u /* permute kernel */
#define GT_FLAG_PHASE_TILE 0x200u    /* tile kernel (the staging buffer of an earlier call is reused) */
#define GT_FLAG_PHASE_SPAN 0x400u    /* the small spanning-node kernel that follows it */
#define GT_FLAG_PHASE_MASK 0x700u

/* Input / output element types. */
#define GT_F32 0
#define GT_F64 1
#define GT_F16 2
#define GT_BF16 3

#define GT_OP_SUM 1
#define GT_OP_MAX 2

/* out[b, n] = sum (or max) over the leaves under node n of ws[b, item(leaf)],  b < n_rows, n < N.
 *   ws       device pointer, row b starts at ws + b*ld_ws elements, V elements per row, type in_type
 *   out_sum / out_max   device pointers (one may be NULL when the op is not requested), row stride
 *            ld_out elements, type out_type (GT_F32 or GT_F64)
 *   ops      GT_OP_SUM | GT_OP_MAX
 *   workspace  device scratch, see gt_workspace_bytes
 * Numerics: every node is a sum of non-negative terms (aligned leaf blocks; no prefix differences).  With
 * out_type GT_F32 the terms inside a tile of 1024 leaves are added pairwise in fp32 and the per-tile pieces of a
 * node that spans tiles in fp64, rounded once (measured <= 2e-7 relative to the fp64 reference); with GT_F64
 * everything is fp64.  max is exact. */
int gt_weight_reduce(const gt_trie* t, const void* ws, int in_type, int64_t n_rows, int64_t ld_ws,
                     void* out_sum, void* out_max, int out_type, int64_t ld_out, unsigned ops,
                     unsigned flags, void* workspace, size_t workspace_bytes, gt_stream stream);

/* ---- SMC row op: masked logsumexp + one categorical draw per row ------------------------- */

#define GT_MASK_NONE 0
#define GT_MASK_ADD_F32 1 /* additive float mask ({0,-inf} in the reference idiom, README.md:59-70) */
#define GT_MASK_BOOL_U8 2 /* one byte per token, 0 = masked out                                   */
#define GT_MASK_BITS_U32 3/* bit i%32 of word i/32, 0 = masked out                                */

/* For each row b: masked = logp[b]/temperature + mask;  logZ[b] = logsumexp(masked);
 * tok[b] ~ Categorical(exp(masked - logZ[b])) by inverse CDF with one Philox uniform per row,
 * counter = (seed, offset + b).  Rows with no mass get logZ = -inf, tok = -1.  As torch.logsumexp, an allowed NaN
 * gives logZ = NaN, else an allowed +inf gives logZ = +inf; both give tok = -1.  A masked-out value is dropped by a
 * GT_MASK_BOOL_U8 or GT_MASK_BITS_U32 mask whatever it is (NaN and +inf included), while an additive mask adds -inf to
 * it: a masked-out +inf (or NaN) then makes logZ NaN, as in torch.
 *   mask_ld   elements (floats / bytes / words) between consecutive rows' masks; 0 = shared mask */
int gt_lse_sample(const void* logp, int in_type, int64_t n_rows, int64_t n_vocab, int64_t ld_logp,
                  const void* mask, int mask_kind, int64_t mask_ld, float temperature,
                  uint64_t seed, uint64_t offset, float* logZ_out, int32_t* tok_out, gt_stream stream);

/* ---- read-outs that keep the [B, N] slab on the GPU ------------------------------------------ */

#define GT_GATHER_LOG 1u /* return log-masses */

/* out[b, k] = mass[b, node_ids[b * ids_ld + k]]  (ids_ld = 0: one id list shared by all rows; id < 0 or >= n_nodes
 * reads as mass 0).  With norm_node != NULL the value is divided by mass[b, norm_node[b]] (with GT_GATHER_LOG:
 * log mass - log normaliser) -- the conditional next-symbol distribution a caller of weight_sum forms from
 * mass[children(node)] / mass[node].  Replaces the D2H copy of the whole slab in parallel.py:103,145 when only a few
 * nodes per row are read.  mass / out: device, type GT_F32 or GT_F64; node_ids / norm_node: device int32. */
int gt_gather_nodes(const void* mass, int type, int64_t n_rows, int64_t n_nodes, int64_t ld_mass,
                    const int32_t* node_ids, int64_t n_ids, int64_t ids_ld, const int32_t* norm_node,
                    unsigned flags, void* out, int64_t ld_out, gt_stream stream);

/* The copy the reference ends on (parallel.py:103,145: masses.cpu().numpy()): n_rows rows of width_bytes each from a
 * device slab whose rows are src_pitch bytes apart (the engine pads rows to whole 128-byte lines) into host memory
 * whose rows are dst_pitch bytes apart -- a C-contiguous [n_rows, N] array when dst_pitch == width_bytes.  One pitched
 * DMA on `stream` (cudaMemcpy2DAsync); dst_host should be page-locked for the copy to be asynchronous. */
int gt_download_rows(void* dst_host, size_t dst_pitch, const void* src_dev, size_t src_pitch, size_t width_bytes,
                     int64_t n_rows, gt_stream stream);

/* mask_bits[b, i/32] bit i%32 = 1 iff item i's leaf lies in the subtree of node nodes[b] -- column nodes[b] of the
 * reference's reachability matrix M (parallel.py:33-64) as a keep-bitmask in gt_lse_sample's GT_MASK_BITS_U32 layout
 * (tokens whose spelling extends the prefix of that node).  nodes[b] < 0 or >= N gives an all-zero row.
 * nodes / mask_bits: device; mask_ld >= ceil(V/32) words per row, every word of the first ceil(V/32) is written. */
int gt_subtree_token_mask(const gt_trie* t, const int32_t* nodes, int64_t n_rows, uint32_t* mask_bits,
                          int64_t mask_ld, gt_stream stream);

/* ---- child masses of one node per row, straight from the rows ------------------------------ */

/* D: the largest child count of any node (host only, no GPU needed); -1 for a null trie. */
int64_t gt_max_children(const gt_trie* t);

/* Caller-owned scratch of gt_child_masses / gt_child_sample for batches of up to max_rows rows (capped at 1,024: larger
 * batches, or a smaller workspace, are processed in chunks; any size that holds one row works).  Host only.  One call at
 * a time may use a workspace; the pointer must be 256-byte aligned. */
size_t gt_child_workspace_bytes(const gt_trie* t, int64_t max_rows);

#define GT_CHILD_NORMALIZE 0x10u /* divide each child's sum by the node's mass (the fp64 sum over its children) */
#define GT_CHILD_LOG 0x20u       /* return log-masses (sum and max) */

/* For each row b and the node n = nodes[b] (device int32), with the children c_0 < c_1 < ... of n in jump[n] order:
 *   child_ids[b, j] = c_j
 *   out_sum[b, j]   = sum of the row's weights over the leaves under c_j
 *   out_max[b, j]   = max of the row's weights over the same leaves
 * for j < deg(n); columns deg(n) <= j < D (D = gt_max_children) are padding: child id -1 and the value of no mass,
 * 0 (-inf with GT_CHILD_LOG).  A node id < 0 or >= N, or a leaf, gives an all-padding row.
 *   ws, in_type, ld_ws, GT_FLAG_LOG_INPUT, GT_FLAG_DFS_ORDER   as for gt_weight_reduce
 *   child_ids / out_sum / out_max   device, row stride ld_out >= D elements; out_sum / out_max may be NULL when the
 *                                   op is not in `ops` (GT_OP_SUM | GT_OP_MAX)
 *   flags    GT_FLAG_LOG_INPUT | GT_FLAG_DFS_ORDER | GT_CHILD_NORMALIZE | GT_CHILD_LOG
 * Numerics: each weight is converted exactly as gt_weight_reduce converts it (so out_max is bit-equal to its fp32 max
 * slab at child_ids); sums are accumulated in fp64 in an order that depends only on (node, child) -- not on the batch,
 * the row order, the workspace or the input order -- and rounded once.  Only the leaves under nodes[b] are read. */
int gt_child_masses(const gt_trie* t, const void* ws, int in_type, int64_t n_rows, int64_t ld_ws, const int32_t* nodes,
                    int32_t* child_ids, float* out_sum, float* out_max, int64_t ld_out, unsigned ops, unsigned flags,
                    void* workspace, size_t workspace_bytes, gt_stream stream);

/* One draw of the next symbol per row: u = 53-bit Philox4x32-10 uniform (counter offset + b, key seed, as
 * gt_lse_sample), m_j = the fp64 child sums of gt_child_masses, total = sum_j m_j; the chosen child is the first j whose
 * running sum exceeds u * total (a child without mass is never chosen).
 *   child_out[b] = c_j,  logp_out[b] = log m_j - log total,  logZ_out[b] = log total (the node's mass)
 * A row without mass (also a leaf or an invalid node id) gives child -1 and logp = logZ = -inf; a NaN weight under the
 * node gives child -1 and logp = logZ = NaN.  flags: GT_FLAG_LOG_INPUT | GT_FLAG_DFS_ORDER. */
int gt_child_sample(const gt_trie* t, const void* ws, int in_type, int64_t n_rows, int64_t ld_ws, const int32_t* nodes,
                    unsigned flags, uint64_t seed, uint64_t offset, int32_t* child_out, float* logp_out, float* logZ_out,
                    void* workspace, size_t workspace_bytes, gt_stream stream);

/* ---- next-symbol masses indexed by symbol, and a draw under per-row symbol log-weights ---------- */

/* S = max(256, 1 + the largest symbol passed to gt_build); -1 for a null trie.  Host only.  The symbol read-outs are
 * S + 1 wide: column s < S is the child whose edge symbol is s, column S is "the token ends here" (the leaf children). */
int64_t gt_num_symbols(const gt_trie* t);

/* For each row b and the node n = nodes[b], with the per-child fp64 sums and fp32 maxes of gt_child_masses:
 *   out_sum[b, s] / out_max[b, s]   (s < S) the sum / max over the leaves under the child of n with edge symbol s;
 *                                   0 (-inf with GT_CHILD_LOG) when n has no such child
 *   out_sum[b, S]                   the fp64 sum of the sums of all leaf children of n, added in child order, rounded once
 *   out_max[b, S]                   the max over the maxes of the leaf children of n
 * A node id < 0 or >= N, or a leaf, gives an all-padding row.  ws, in_type, ld_ws, ops, flags (GT_FLAG_LOG_INPUT |
 * GT_FLAG_DFS_ORDER | GT_CHILD_NORMALIZE | GT_CHILD_LOG) and the workspace (gt_child_workspace_bytes) are those of
 * gt_child_masses; out_sum / out_max are device, row stride ld_out >= S + 1.  out_sum[b, sym(c_j)] is bit-equal to
 * gt_child_masses' out_sum[b, j] under the same flags (column S too when n has one leaf child); maxes likewise. */
int gt_symbol_masses(const gt_trie* t, const void* ws, int in_type, int64_t n_rows, int64_t ld_ws, const int32_t* nodes,
                     float* out_sum, float* out_max, int64_t ld_out, unsigned ops, unsigned flags,
                     void* workspace, size_t workspace_bytes, gt_stream stream);

/* One draw of the next symbol per row in proportion to q_j = m_j * exp(sym_logw[b, sym(c_j)]) (fp64; q_j = 0 when
 * m_j = 0, whatever the log-weight), with m_j the child sums of gt_child_masses and sym(c) the edge symbol of child c,
 * S for a leaf child.  Z = sum_j q_j in the order gt_child_sample adds the m_j; u as in gt_child_sample (counter
 * offset + b, key seed); the pick is the first child whose running sum exceeds u * Z (else the last with q_j > 0).
 *   child_out[b] = c_j, symbol_out[b] = sym(c_j), logp_out[b] = log q_j - log Z, logZ_out[b] = log Z,
 *   logM_out[b] = log sum_j m_j (gt_child_sample's logZ; logM_out may be NULL)
 * sym_logw: device fp32 log-weights, [rows][S + 1]; ld_w = 0 shares row 0 between all rows, else ld_w >= S + 1.
 * With every log-weight 0, child / logp / logZ are bit-identical to gt_child_sample.  A row without a draw gives
 * child = symbol = -1: Z = 0 (also a leaf or an invalid id) gives logp = logZ = -inf; a NaN weight under the node, or
 * a NaN log-weight at a symbol the node has, gives logp = logZ = NaN; Z = +inf gives logZ = +inf, logp = NaN.
 * flags: GT_FLAG_LOG_INPUT | GT_FLAG_DFS_ORDER. */
int gt_symbol_sample(const gt_trie* t, const void* ws, int in_type, int64_t n_rows, int64_t ld_ws, const int32_t* nodes,
                     const float* sym_logw, int64_t ld_w, unsigned flags, uint64_t seed, uint64_t offset,
                     int32_t* child_out, int32_t* symbol_out, float* logp_out, float* logZ_out, float* logM_out,
                     void* workspace, size_t workspace_bytes, gt_stream stream);

/* ---- the next-symbol read-outs restricted to the items a per-row keep-bitmask allows -------------------------------- */

/* gt_child_masses / gt_child_sample / gt_symbol_masses / gt_symbol_sample over the allowed items only.  mask_bits: device
 * keep-bitmask in GT_MASK_BITS_U32 layout and item order (bit i % 32 of word i / 32 = 1: item i is kept) -- what
 * gt_dfa_token_mask and gt_subtree_token_mask write; row b's mask starts at mask_bits + b * mask_ld words, mask_ld = 0
 * shares one mask between all rows, else mask_ld >= ceil(V/32).  Bits at or above V are ignored.
 * Every result -- ids, sums, maxes, normalised and log outputs, and the child, symbol, logp, logZ and logM of the draws
 * under the same seed and offset -- is bit for bit that of the unmasked call on rows whose masked-out weights are 0
 * (-inf with GT_FLAG_LOG_INPUT): a masked-out weight never contributes, NaN and inf included; a child without an
 * allowed item has sum and max 0 (-inf with GT_CHILD_LOG) and is never drawn; a row without allowed mass under its node
 * gives child -1 and logZ = -inf; an all-ones mask gives the unmasked results.  For a byte-level DFA, the mask of
 * gt_dfa_token_mask at the root in the particle's state stays valid for every symbol of the token: drawing symbol by
 * symbol from the root under it draws exactly from the masked token distribution of gt_lse_sample, and the root's
 * logZ is that call's logZ.  Only the leaves under nodes[b] and their mask words are read; a weight whose bit is 0 is
 * not read where its load can be skipped.  Argument checks, in order: the unmasked call's scalars and mask_ld (< 0, or
 * between 0 and ceil(V/32): GT_ERR_ARG); no rows returns GT_OK, null pointers accepted; the data pointers (a null
 * mask_bits: GT_ERR_ARG); the workspace.  No allocation, no synchronisation, graph-capturable. */
int gt_child_masses_masked(const gt_trie* t, const void* ws, int in_type, int64_t n_rows, int64_t ld_ws, const int32_t* nodes,
                           const uint32_t* mask_bits, int64_t mask_ld, int32_t* child_ids, float* out_sum, float* out_max,
                           int64_t ld_out, unsigned ops, unsigned flags, void* workspace, size_t workspace_bytes,
                           gt_stream stream);
int gt_child_sample_masked(const gt_trie* t, const void* ws, int in_type, int64_t n_rows, int64_t ld_ws, const int32_t* nodes,
                           const uint32_t* mask_bits, int64_t mask_ld, unsigned flags, uint64_t seed, uint64_t offset,
                           int32_t* child_out, float* logp_out, float* logZ_out, void* workspace, size_t workspace_bytes,
                           gt_stream stream);
int gt_symbol_masses_masked(const gt_trie* t, const void* ws, int in_type, int64_t n_rows, int64_t ld_ws, const int32_t* nodes,
                            const uint32_t* mask_bits, int64_t mask_ld, float* out_sum, float* out_max, int64_t ld_out,
                            unsigned ops, unsigned flags, void* workspace, size_t workspace_bytes, gt_stream stream);
int gt_symbol_sample_masked(const gt_trie* t, const void* ws, int in_type, int64_t n_rows, int64_t ld_ws, const int32_t* nodes,
                            const uint32_t* mask_bits, int64_t mask_ld, const float* sym_logw, int64_t ld_w, unsigned flags,
                            uint64_t seed, uint64_t offset, int32_t* child_out, int32_t* symbol_out, float* logp_out,
                            float* logZ_out, float* logM_out, void* workspace, size_t workspace_bytes, gt_stream stream);

/* ---- token masks under a byte-level DFA, and the DFA advance over drawn tokens ------------------------------------ */

/* delta: device int32 [n_states][ld_delta], ld_delta >= S (gt_num_symbols): delta[q * ld_delta + s] is the state after
 * symbol s from state q; -1 (any value outside [0, n_states)) rejects.  A state is live iff it lies in [0, n_states).  The
 * table is meant to be trimmed (every state a non-reject transition reaches can still reach an accepting state), so that
 * "live" means "the prefix can still be completed"; the kernels only follow the table.  depth(n) is the number of symbols
 * on the path root -> n (a leaf edge consumes none: a leaf's depth is its item's length).  For row b, n = nodes[b] (the
 * root when nodes == NULL) and q = states[b], the state after the symbols of the path to n; item i is allowed iff its leaf
 * lies under n (gt_subtree_token_mask), q is live, and delta walked from q over item i's symbols depth(n) .. len(i)-1 never
 * leaves the live states (an item with no remaining symbols: iff q is live).  A node id < 0 or >= N, or a state outside
 * [0, n_states), gives an all-zero row.  End of sequence needs no special case: an EOS item spells a non-byte symbol, whose
 * column decides it (delta[q, eos] = q for accepting q, -1 otherwise).  Several constraints in one call: stack their tables
 * with disjoint state ranges (offset each table's states) and give each row its own start state.
 * Argument checks (GT_ERR_ARG, before any device work): null t / delta / states / outputs (tokens for the advance),
 * n_states < 1, ld_delta < S, n_rows < 0, mask_ld < ceil(V/32); n_states * ld_delta >= 2^31 gives GT_ERR_LIMIT.  No
 * allocation, no synchronisation, launches on `stream`, graph-capturable. */

/* keep-bitmask (GT_MASK_BITS_U32 layout, item order) of the items allowed under a byte DFA, per row.  Every word of the
 * first ceil(V/32) words of each row is written (bits >= V of the last word are 0); words beyond them are not touched. */
int gt_dfa_token_mask(const gt_trie* t, const int32_t* delta, int64_t n_states, int64_t ld_delta,
                      const int32_t* states, const int32_t* nodes /* NULL = root */, int64_t n_rows,
                      uint32_t* mask_bits, int64_t mask_ld, gt_stream stream);

/* Per-row token log-weights under a deterministic weighted byte automaton: delta as above, and logw: device fp32, the
 * same shape and row stride, logw[q * ld_delta + s] the log-weight of the transition from q on symbol s.  For row b, with
 * n and q as above, out[b * ld_out + i] is
 *   - for an item gt_dfa_token_mask allows: the sum of (double) logw[q_k, s_k] over k = depth(n) .. len(i)-1, with q_k
 *     the state before symbol s_k, added in increasing k in fp64 from 0.0 and rounded once to fp32 (0.0f for an item
 *     with no remaining symbols);
 *   - -inf for every other item (outside the subtree, an invalid node, a dead or invalid state, a reject on the way).
 * IEEE arithmetic decides special values: a -inf transition weight makes the token -inf, a NaN weight on the walk or
 * -inf + +inf gives NaN; the walk does not stop on a -inf sum, only on a reject.  With logw = 0 everywhere, out is the
 * additive {0, -inf} form of gt_dfa_token_mask's bits, and isfinite(out) is that mask for any finite table whose sums
 * stay inside the fp32 range.  End of sequence: the EOS column of logw holds the final weight.  The result is
 * gt_lse_sample's GT_MASK_ADD_F32 mask (mask_ld = ld_out): its logZ is log sum_i p_i w_i, the particle's weight
 * increment, and its draw is from p w / Z; gt_dfa_advance takes the same delta.  For a prefix weight phi given by a
 * deterministic weighted automaton, the weight-pushed table makes the row log phi(x t) - log phi(x), the exact
 * token-level factor.  Writes the first V floats of each row, nothing beyond them; ld_out >= V.  Argument checks, in
 * order: null t; null delta / logw / states / out; ld_out < V (GT_ERR_ARG); n_states, ld_delta and n_rows as above (a
 * table of 2^31 entries or more: GT_ERR_LIMIT); no rows returns GT_OK; more rows than the grid takes: GT_ERR_LIMIT. */
int gt_dfa_token_logw(const gt_trie* t, const int32_t* delta, const float* logw, int64_t n_states, int64_t ld_delta,
                      const int32_t* states, const int32_t* nodes /* NULL = root */, int64_t n_rows,
                      float* out, int64_t ld_out, gt_stream stream);

/* states_out[b] = state after item tokens[b]'s symbols depth(nodes[b]) .. end, walked from states[b]; -1 for a token < 0 or
 * >= V (the sampler's "no draw"), a token not under nodes[b], an invalid node, a dead or invalid start state, or any reject
 * on the way.  states_out[b] >= 0 exactly when gt_dfa_token_mask sets the token's bit for that row. */
int gt_dfa_advance(const gt_trie* t, const int32_t* delta, int64_t n_states, int64_t ld_delta,
                   const int32_t* states, const int32_t* nodes /* NULL = root */, const int32_t* tokens,
                   int64_t n_rows, int32_t* states_out, gt_stream stream);

/* ---- token masks under a byte-level pushdown automaton, and the PDA advance over drawn tokens ---------------------- */

#define GT_PDA_POP (-2)
#define GT_PDA_MAX_DEPTH 64

/* A deterministic byte-level pushdown automaton in return-state form (a push saves the state to return to, a pop goes
 * there), as a grammar compiles into a recursive transition network.  delta and push: device int32 [n_states][ld_delta],
 * ld_delta >= S (gt_num_symbols), the same shape and row stride.  From state q on symbol s:
 *   - delta[q, s] in [0, n_states): if push[q, s] >= 0, push it (push[q, s] >= n_states, or a stack already holding
 *     stack_ld entries, rejects), then go to delta[q, s];
 *   - delta[q, s] == GT_PDA_POP: pop the top of the stack and go to the popped state (an empty stack, or a popped value
 *     outside [0, n_states), rejects);
 *   - any other value rejects.  push[q, s] is read only for a move.
 * Row b's configuration is its state states[b], its depth depth[b] and its stack stack[b * stack_ld + 0 .. depth[b]-1],
 * bottom first; stack_ld is both the row stride and every row's capacity, 1 <= stack_ld <= GT_PDA_MAX_DEPTH.  A state
 * outside [0, n_states) or a depth outside [0, stack_ld] makes the row invalid.  Rows stand at the root: item i is
 * allowed iff the row is valid and the walk over all of item i's symbols never rejects (an item with no symbols: iff the
 * row is valid).  End of sequence needs no special case: the EOS item's symbol column decides it.  A table with push
 * -1 everywhere and no GT_PDA_POP entry is a DFA: both calls then give what gt_dfa_token_mask and gt_dfa_advance give at
 * the root, and leave stack and depth untouched.
 * Argument checks, in order: null t or data pointers, mask_ld < ceil(V/32) (GT_ERR_ARG); n_states, ld_delta and n_rows as
 * for the DFA calls (a table of 2^31 entries or more: GT_ERR_LIMIT); stack_ld < 1 (GT_ERR_ARG) or > GT_PDA_MAX_DEPTH
 * (GT_ERR_LIMIT); no rows returns GT_OK; more rows than the grid takes: GT_ERR_LIMIT.  No allocation, no
 * synchronisation, launches on `stream`, graph-capturable. */

/* keep-bitmask of the items allowed under the PDA from each row's configuration, in gt_dfa_token_mask's layout: every word
 * of the first ceil(V/32) words of each row is written (bits >= V of the last word are 0), words beyond them are not
 * touched.  An invalid row gives an all-zero row.  stack and depth are only read. */
int gt_pda_token_mask(const gt_trie* t, const int32_t* delta, const int32_t* push, int64_t n_states, int64_t ld_delta,
                      const int32_t* states, const int32_t* stack, int64_t stack_ld, const int32_t* depth,
                      int64_t n_rows, uint32_t* mask_bits, int64_t mask_ld, gt_stream stream);

/* Per-row token log-weights under a deterministic weighted pushdown automaton: delta, push and the rows as above, and
 * logw: device fp32, the same shape and row stride, logw[q * ld_delta + s] the log-weight of the transition from q on
 * symbol s, be it a move, a move with a push or a pop.  A pop's weight is read at (q, s) and does not depend on the
 * popped state: a weight that should depend on the state returned to belongs on the push that saved it.  For row b,
 * out[b * ld_out + i] is
 *   - for an item gt_pda_token_mask allows: the sum of (double) logw[q_k, s_k] over all of item i's symbols, with q_k
 *     the state before symbol s_k, added in increasing k in fp64 from 0.0 and rounded once to fp32 (0.0f for an item
 *     with no symbols);
 *   - -inf for every other item (an invalid row, any reject on the way: a push past stack_ld, a pop from an empty stack,
 *     a popped value outside [0, n_states)), whatever the weights.
 * IEEE arithmetic decides special values: a -inf transition weight makes the token -inf, a NaN weight on the walk or
 * -inf followed by +inf gives NaN; the walk does not stop on a -inf sum, only on a reject.  With logw = 0 everywhere,
 * out is the additive {0, -inf} form of gt_pda_token_mask's bits; on a table with no push and no pop and empty stacks,
 * out is gt_dfa_token_logw's at the root.  End of sequence: the EOS column of logw holds the final weights.  The
 * result is gt_lse_sample's GT_MASK_ADD_F32 mask (mask_ld = ld_out): its logZ is log sum_i p_i w_i, the particle's
 * weight increment; gt_pda_advance takes the same delta and push.  Writes the first V floats of each row, nothing
 * beyond them; ld_out >= V.  Argument checks, in order: null t; null delta / push / logw / states / stack / depth / out;
 * ld_out < V (GT_ERR_ARG); the table, row and capacity checks of gt_pda_token_mask; no rows returns GT_OK; more rows than
 * the grid takes: GT_ERR_LIMIT.  No allocation, no synchronisation, launches on `stream`, graph-capturable. */
int gt_pda_token_logw(const gt_trie* t, const int32_t* delta, const int32_t* push, const float* logw, int64_t n_states,
                      int64_t ld_delta, const int32_t* states, const int32_t* stack, int64_t stack_ld,
                      const int32_t* depth, int64_t n_rows, float* out, int64_t ld_out, gt_stream stream);

/* states_out[b] = the state after all of item tokens[b]'s symbols from row b's configuration, or -1 for a token < 0 or
 * >= V (the sampler's "no draw"), an invalid row or any reject on the way; states_out[b] >= 0 exactly where
 * gt_pda_token_mask sets the token's bit.  Where states_out[b] >= 0, stack and depth[b] hold the new configuration, in
 * place (entries at or above the new depth are unspecified); elsewhere the row's stack and depth[b] are unchanged.
 * states_out may equal states. */
int gt_pda_advance(const gt_trie* t, const int32_t* delta, const int32_t* push, int64_t n_states, int64_t ld_delta,
                   const int32_t* states, int32_t* stack, int64_t stack_ld, int32_t* depth,
                   const int32_t* tokens, int64_t n_rows, int32_t* states_out, gt_stream stream);

/* ---- particle resampling: per-group effective sample size and ancestors ----------------------------------------- */

#define GT_RESAMPLE_MULTINOMIAL 0
#define GT_RESAMPLE_STRATIFIED 1
#define GT_RESAMPLE_SYSTEMATIC 2
#define GT_RESAMPLE_MAX_GROUP 16384

/* Particles lie contiguously in n_groups groups of P = group_size: particle b = g * P + j is particle j of group g.  For
 * group g, with lw_j = logw[g * P + j] and m = max_j lw_j:
 *   - any NaN: ess = NaN, log_mean_w = NaN; else any +inf: ess = NaN, log_mean_w = +inf; else all -inf: ess = 0,
 *     log_mean_w = -inf.  None of these resamples.
 *   - otherwise, in fp64: w_j = exp((double) lw_j - m), S = sum_j w_j, Q = sum_j w_j^2; ess = (float)(S^2 / Q),
 *     log_mean_w = (float)(m + log S - log P).  The group resamples iff S^2 / Q < ess_threshold * P (fp64): a threshold of
 *     0 never resamples, +inf always does, and uniform weights (ess exactly P) do not at a threshold of 1.
 *   - a group that does not resample: ancestors[b] = b, logw_out[b] = logw[b].
 *   - a group that resamples: with c_i = w_0 + ... + w_i (an fp64 inclusive scan in a fixed order), particle j gets
 *     ancestors[b] = g * P + i for the first i with c_i > t_j, else the last i with w_i > 0 (a particle with w_i = 0 is
 *     never an ancestor); logw_out[b] = log_mean_w, which keeps the running marginal-likelihood estimate.  The points are
 *       multinomial  t_j = u_b * S;  stratified  t_j = (j + u_b) / P * S;  systematic  t_j = (j + u_{g*P}) / P * S,
 *     so stratified and systematic ancestors are non-decreasing in j and multinomial ones come in draw order.
 *   - u_b: the 53-bit Philox4x32-10 uniform of the samplers under key seed, with counter offset + b in the first two words
 *     and 1 (the samplers: 0) in the third, so one (seed, offset) can drive a sampler and the resampler.
 * ess_out, log_mean_w_out and resampled_out (0 or 1) hold one entry per group.  logw_out may equal logw (in place); any
 * other overlap is undefined.  A group's results depend only on its weights, P, method, threshold, seed and
 * offset + g * P.  Argument checks, in order: n_groups < 0, group_size < 1, an unknown method or a NaN threshold:
 * GT_ERR_ARG; group_size > GT_RESAMPLE_MAX_GROUP or n_groups * P > INT32_MAX: GT_ERR_LIMIT; no groups returns GT_OK, null
 * pointers accepted; a null pointer: GT_ERR_ARG.  No allocation, no synchronisation, graph-capturable. */
int gt_resample(const float* logw, int64_t n_groups, int64_t group_size, int method, float ess_threshold,
                uint64_t seed, uint64_t offset, int32_t* ancestors, float* logw_out, float* ess_out,
                float* log_mean_w_out, uint8_t* resampled_out, gt_stream stream);

#ifdef __cplusplus
}
#endif
#endif /* GENLM_TRIE_B200_H */
