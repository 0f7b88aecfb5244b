// Host trie builder: reproduces the node numbering of the reference
// (genlm/backend/trie/base.py:29-93 build, :95-122 rename, :219-247 orderings) with flat arrays
// and an iterative post-order walk, and derives the DFS leaf layout the kernels use.
#include "trie_internal.h"

#include <climits>
#include <cstring>

namespace gt {

static thread_local std::string g_err;

void set_error(const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
}

namespace {

// (parent node, symbol) -> child node, open addressing with linear probing.
struct EdgeTable {
    std::vector<uint64_t> keys;
    std::vector<int32_t> vals;
    uint64_t mask = 0;
    static constexpr uint64_t EMPTY = ~0ull;

    explicit EdgeTable(size_t expected) {
        size_t cap = 64;
        while (cap < expected * 2 + 16) cap <<= 1;
        keys.assign(cap, EMPTY);
        vals.assign(cap, -1);
        mask = cap - 1;
    }
    static uint64_t mix(uint64_t x) {
        x ^= x >> 33; x *= 0xff51afd7ed558ccdull;
        x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ull;
        x ^= x >> 33;
        return x;
    }
    // returns the slot holding `key`, or the empty slot where it would go
    size_t find(uint64_t key) const {
        size_t i = mix(key) & mask;
        while (keys[i] != EMPTY && keys[i] != key) i = (i + 1) & mask;
        return i;
    }
};

}  // namespace

static int build_layout(const int32_t* symbols, const int64_t* offsets, int64_t V, Layout& L) {
    const int64_t total = offsets[V] - offsets[0];
    if (total < 0) { set_error("offsets must be non-decreasing"); return GT_ERR_ARG; }
    const int64_t max_nodes = 1 + total + V;
    if (max_nodes >= INT32_MAX) { set_error("trie too large for int32 node ids"); return GT_ERR_LIMIT; }

    // insertion-ordered child lists as sibling chains (base.py:50-58: dict insertion order)
    std::vector<int32_t> first_child, last_child, next_sib, parent, label;
    first_child.reserve(max_nodes); last_child.reserve(max_nodes); next_sib.reserve(max_nodes);
    parent.reserve(max_nodes); label.reserve(max_nodes);
    auto new_node = [&](int32_t par, int32_t lab) -> int32_t {
        int32_t id = (int32_t)first_child.size();
        first_child.push_back(-1); last_child.push_back(-1); next_sib.push_back(-1);
        parent.push_back(par); label.push_back(lab);
        if (par >= 0) {
            if (last_child[par] < 0) first_child[par] = id; else next_sib[last_child[par]] = id;
            last_child[par] = id;
        }
        return id;
    };
    new_node(-1, INT32_MIN);  // root is node 0 before renumbering (base.py:23-24)

    EdgeTable table((size_t)total);
    std::vector<int32_t> leaf_old((size_t)V);
    int64_t max_depth = 0, num_symbols = 256;
    for (int64_t i = 0; i < V; ++i) {
        if (offsets[i + 1] < offsets[i]) { set_error("offsets must be non-decreasing"); return GT_ERR_ARG; }
        int32_t cur = 0;
        for (int64_t k = offsets[i]; k < offsets[i + 1]; ++k) {
            const int32_t sym = symbols[k];
            if (sym < 0) { set_error("negative symbol at item %lld", (long long)i); return GT_ERR_ARG; }
            if ((int64_t)sym + 1 > num_symbols) num_symbols = (int64_t)sym + 1;
            const uint64_t key = ((uint64_t)(uint32_t)cur << 32) | (uint32_t)sym;
            const size_t slot = table.find(key);
            if (table.keys[slot] == EdgeTable::EMPTY) {
                table.keys[slot] = key;
                table.vals[slot] = new_node(cur, sym);
            }
            cur = table.vals[slot];
        }
        // every item gets its own leaf, keyed (None, i) in the reference (base.py:55-61)
        leaf_old[(size_t)i] = new_node(cur, (int32_t)(-1 - i));
        const int64_t depth = offsets[i + 1] - offsets[i] + 1;
        if (depth > max_depth) max_depth = depth;
    }
    const int64_t N = (int64_t)first_child.size();

    // full post-order with children in insertion order (base.py:236-247) -> new ids
    std::vector<int32_t> newid((size_t)N, -1), lo_old((size_t)N), hi_old((size_t)N);
    {
        std::vector<int32_t> stack_node, stack_next;
        stack_node.reserve((size_t)max_depth + 4); stack_next.reserve((size_t)max_depth + 4);
        stack_node.push_back(0); stack_next.push_back(first_child[0]);
        lo_old[0] = 0;
        int32_t counter = 0, leaf_rank = 0;
        while (!stack_node.empty()) {
            const int32_t u = stack_node.back();
            const int32_t c = stack_next.back();
            if (c >= 0) {
                stack_next.back() = next_sib[c];
                lo_old[c] = leaf_rank;
                stack_node.push_back(c); stack_next.push_back(first_child[c]);
            } else {
                if (first_child[u] < 0) ++leaf_rank;  // a leaf
                hi_old[u] = leaf_rank;
                newid[u] = counter++;
                stack_node.pop_back(); stack_next.pop_back();
            }
        }
    }

    L.V = V; L.N = N; L.max_depth = max_depth; L.num_symbols = num_symbols;
    L.leaf_node.resize((size_t)V);
    L.parent.assign((size_t)N, -1);
    L.edge_label.resize((size_t)N);
    L.child_ptr.assign((size_t)N + 1, 0);
    L.child_idx.resize((size_t)(N > 0 ? N - 1 : 0));
    L.perm.resize((size_t)V);
    L.lo.resize((size_t)N); L.hi.resize((size_t)N);
    L.is_leaf.assign((size_t)N, 0);

    for (int64_t u = 0; u < N; ++u) {
        const int32_t n = newid[u];
        L.parent[n] = parent[u] >= 0 ? newid[parent[u]] : -1;
        L.edge_label[n] = label[u];
        L.lo[n] = lo_old[u]; L.hi[n] = hi_old[u];
        L.is_leaf[n] = first_child[u] < 0;
        int32_t deg = 0;
        for (int32_t c = first_child[u]; c >= 0; c = next_sib[c]) ++deg;
        L.child_ptr[(size_t)n + 1] = deg;
        if (deg > L.max_children) L.max_children = deg;
    }
    for (int64_t n = 0; n < N; ++n) L.child_ptr[(size_t)n + 1] += L.child_ptr[(size_t)n];
    for (int64_t u = 0; u < N; ++u) {
        int32_t at = L.child_ptr[newid[u]];
        for (int32_t c = first_child[u]; c >= 0; c = next_sib[c]) L.child_idx[at++] = newid[c];
    }
    int64_t nnz = 0;
    for (int64_t i = 0; i < V; ++i) {
        const int32_t leaf = newid[leaf_old[(size_t)i]];
        L.leaf_node[(size_t)i] = leaf;
        L.perm[L.lo[leaf]] = (int32_t)i;
        nnz += offsets[i + 1] - offsets[i] + 2;  // leaf + one node per symbol + root
    }
    L.nnz = nnz;
    return GT_OK;
}

}  // namespace gt

gt_trie::~gt_trie() {
    for (auto& kv : dev) gt::free_device_plan(kv.second);
}

extern "C" {

const char* gt_last_error(void) { return gt::g_err.c_str(); }
int gt_version(void) { return 1; }

int gt_build(const int32_t* symbols, const int64_t* offsets, int64_t n_tokens, gt_trie** out) {
    if (!out || !offsets || n_tokens < 0 || (!symbols && offsets[n_tokens] != offsets[0])) {
        gt::set_error("gt_build: bad argument");
        return GT_ERR_ARG;
    }
    std::unique_ptr<gt_trie> t(new gt_trie());
    int rc = gt::build_layout(symbols, offsets, n_tokens, t->layout);
    if (rc != GT_OK) return rc;
    *out = t.release();
    return GT_OK;
}

void gt_free(gt_trie* t) { delete t; }

int64_t gt_num_tokens(const gt_trie* t) { return t ? t->layout.V : -1; }
int64_t gt_num_nodes(const gt_trie* t) { return t ? t->layout.N : -1; }
int64_t gt_root(const gt_trie* t) { return t ? t->layout.N - 1 : -1; }
int64_t gt_num_reach(const gt_trie* t) { return t ? t->layout.nnz : -1; }
int64_t gt_max_depth(const gt_trie* t) { return t ? t->layout.max_depth : -1; }
int64_t gt_max_children(const gt_trie* t) { return t ? t->layout.max_children : -1; }
int64_t gt_num_symbols(const gt_trie* t) { return t ? t->layout.num_symbols : -1; }

int gt_export_layout(const gt_trie* t, int32_t* leaf_node, int32_t* parent, int32_t* edge_label,
                     int32_t* child_ptr, int32_t* child_idx, int32_t* perm, int32_t* lo, int32_t* hi) {
    if (!t) { gt::set_error("gt_export_layout: null trie"); return GT_ERR_ARG; }
    const gt::Layout& L = t->layout;
    auto cp = [](int32_t* dst, const std::vector<int32_t>& src) {
        if (dst && !src.empty()) memcpy(dst, src.data(), src.size() * sizeof(int32_t));
    };
    cp(leaf_node, L.leaf_node); cp(parent, L.parent); cp(edge_label, L.edge_label);
    cp(child_ptr, L.child_ptr); cp(child_idx, L.child_idx); cp(perm, L.perm); cp(lo, L.lo); cp(hi, L.hi);
    return GT_OK;
}

int gt_export_reachability(const gt_trie* t, int64_t* rows, int64_t* cols) {
    if (!t || !rows || !cols) { gt::set_error("gt_export_reachability: bad argument"); return GT_ERR_ARG; }
    const gt::Layout& L = t->layout;
    int64_t k = 0;
    for (int64_t i = 0; i < L.V; ++i) {
        for (int32_t n = L.leaf_node[(size_t)i]; n >= 0; n = L.parent[n]) { rows[k] = i; cols[k] = n; ++k; }
    }
    if (k != L.nnz) { gt::set_error("reachability count mismatch"); return GT_ERR_STATE; }
    return GT_OK;
}

}  // extern "C"
