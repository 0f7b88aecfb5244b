// Internal definitions shared by the builder (host C++), the planner and the CUDA side.
#pragma once
#include <cstdint>
#include <cstdarg>
#include <cstdio>
#include <string>
#include <vector>
#include <map>
#include <memory>
#include <mutex>

#include "../../include/genlm_trie_b200.h"

#include <nvtx3/nvToolsExt.h>  // header-only; a no-op unless a profiler injects itself (SURVEY.md section 5: trace ranges)

namespace gt {

void set_error(const char* fmt, ...);

// NVTX range around a host-side launch group: shows up as gt:permute / gt:tile / gt:span / gt:lse_sample in Nsight
// timelines (the kernels themselves are asynchronous; the range marks where they were enqueued).
struct NvtxRange {
    explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
    NvtxRange(const NvtxRange&) = delete;
    NvtxRange& operator=(const NvtxRange&) = delete;
};

// Host layout in the reference's node-id space (post-order, root = N-1).
struct Layout {
    int64_t V = 0, N = 0, nnz = 0, max_depth = 0;
    int64_t max_children = 0;         // D: largest child count of any node
    int64_t num_symbols = 256;        // S = max(256, 1 + largest symbol); column S of the symbol read-outs is end of token
    std::vector<int32_t> leaf_node;   // [V]
    std::vector<int32_t> parent;      // [N]
    std::vector<int32_t> edge_label;  // [N]
    std::vector<int32_t> child_ptr;   // [N+1]
    std::vector<int32_t> child_idx;   // [N-1]
    std::vector<int32_t> perm;        // [V]  DFS rank -> item position
    std::vector<int32_t> lo, hi;      // [N]  DFS leaf range
    std::vector<uint8_t> is_leaf;     // [N]
};

// ---- tile plan (host copy; see trie_plan.cpp for how it is derived) -------------------------
//
// Tiles: DFS leaf ranks [t*T, (t+1)*T).  Staging buffer z (device scratch): one block per row group of R rows,
// [NT][T] value slots of R elements each -- tile t's block is the leaf region of the tile's shared-memory value
// array, byte for byte, so the tile kernel fetches it with one bulk copy.  leaf_dest[i] is the slot (in that
// [NT*T] numbering, swizzled) that item i's weight goes to.
// Shared-memory slot swizzle.  Slots below 2T (leaves + pyramid) are stored at swizzle_slot(s): the 16-byte
// chunk index c is XORed with (c >> 3) & (slot_bytes/2 - 1), a bijection inside every aligned group of 8 chunks.
// It makes "lane u touches slots 8u .. 8u+7" (the in-lane pyramid levels) and its strided level stores
// bank-conflict free.  All slot numbers in the plan tables are already swizzled; only code that computes a
// slot arithmetically applies it.
inline int32_t swizzle_slot(int32_t s, int32_t slot_bytes) {
    const int cs = slot_bytes == 4 ? 2 : (slot_bytes == 8 ? 1 : 0);  // log2(slots per 16-byte chunk)
    const int32_t c = s >> cs;
    const int32_t c2 = c ^ ((c >> 3) & (slot_bytes / 2 - 1));
    return (c2 << cs) | (s & ((1 << cs) - 1));
}

// Aligned blocks of the per-tile pyramid stop at 2^kPyramidTop leaves: a warp builds levels 1..kPyramidTop of its
// 2^kPyramidTop leaves (2^(kPyramidTop-5) per lane, then five shuffle levels), so the pyramid has no cross-warp step.
// 8: 256 leaves per warp.  7 (128 leaves per warp, all eight compute warps of a 1024-leaf tile busy) was measured
// slower on B200 (tile kernel 50.2 vs 48.6 us at 64 rows): the phase is bound by shared-memory bandwidth, not by the
// number of warps that work, and the 256-leaf blocks come back as extra two-term ranges.
constexpr int kPyramidTop = 8;

// Term rows of an ELL chunk are padded (with the identity slot) to a multiple of this.  The kernel adds terms four at a
// time and finishes with a pair and / or a single term.  Measured on B200 (tile kernel, 64 rows, both reductions):
// 4 -> 46.75 us (a third of all term rows were padding: most chunks hold two- and three-term ranges), 2 -> 46.1, 1 -> 45.9.
#ifndef GT_ELL_ROW_PAD
#define GT_ELL_ROW_PAD 1
#endif
constexpr int kEllRowPad = GT_ELL_ROW_PAD;
static_assert(kEllRowPad == 1 || kEllRowPad == 2 || kEllRowPad == 4, "ELL term rows: unpadded, or padded to pairs or quads");

struct Plan {
    int32_t T = 0, NT = 0;
    int32_t R = 0;           // rows per work item of the fp32 pipeline (the fp64 pipeline uses R/2: same slot size)
    int32_t slot_bytes = 0;  // 4 * R
    int32_t max_tile_nodes = 0, max_tile_ell_rows = 0;  // sizes of the shared-memory metadata stages
    int32_t max_tile_chunks = 0;                        // ELL chunks of the largest tile

    // permute: item i's weight is stored at value slot leaf_dest[i] of its row group's staging block
    // (= t * T + swizzled leaf slot inside tile t, t = DFS rank / T)
    std::vector<int32_t> leaf_dest;     // [V]

    // per-tile value array: slots [0,T) leaves in DFS order, [T,2T-1) pyramid of aligned blocks (levels 1..8),
    // 2T-1 the identity element, [2T, ..) multi-term ranges.
    // Multi-term ranges in ELL form: per tile chunks of 32 ranges (sorted by descending term count);
    // chunk c holds ell_k[c] rows of 32 uint16 slots starting at ell_terms[32 * ell_off[c]], padded with
    // the identity slot.  Range j of the tile (j = 32*(c - ell_chunk_ptr[t]) + lane) lands in slot 2T + j.
    std::vector<int32_t> ell_chunk_ptr;  // [NT+1]
    std::vector<int32_t> ell_desc;       // [2 * n_chunks]  (off32, k)
    std::vector<uint16_t> ell_terms;
    std::vector<int32_t> ell_row_ptr;    // [NT+1]  first term row (of 32 slots) of each tile
    int32_t max_levels = 0, max_tile_values = 0;
    int64_t n_multi = 0, n_terms = 0;

    // emit: node ids [tile_node_lo[t], tile_node_lo[t+1]) belong to tile t; node_slot[n] is the
    // tile-local value slot, 0xFFFF for spanning nodes.
    std::vector<int32_t> tile_node_lo;  // [NT+1]
    std::vector<uint16_t> node_slot;    // [N]

    // spanning nodes (leaf range crosses a tile boundary, or is empty): one "piece" per overlapped tile
    // (a leaf range inside that tile, resolved to a value slot like any node).  Tile t writes pieces
    // piece_ptr[t]..piece_ptr[t+1] (slot piece_slot[i] -> part[piece_idx[i]]); node span_node[i] is the
    // reduction of parts span_pp[i] .. span_pp[i+1].
    std::vector<int32_t> piece_ptr;     // [NT+1]
    std::vector<uint16_t> piece_slot;   // [n_piece_emits]
    std::vector<int32_t> piece_idx;     // [n_piece_emits]
    std::vector<int32_t> span_node;     // [n_span]
    std::vector<int32_t> span_pp;       // [n_span+1]
    int32_t n_pieces = 0;
};

struct DevicePlan;  // defined in trie_device.cuh
void free_device_plan(DevicePlan*);

}  // namespace gt

struct gt_trie {
    gt::Layout layout;
    std::unique_ptr<gt::Plan> plan;
    std::map<int, gt::DevicePlan*> dev;  // device ordinal -> resident metadata
    std::mutex mu;                       // guards plan / dev while gt_plan / gt_upload build them (several host threads
                                         // may bring up different devices of one trie; the launch paths only read)
    ~gt_trie();
};

namespace gt {
// trie_plan.cpp
int build_plan(const Layout& L, int32_t T, int32_t R, Plan& P);
}
