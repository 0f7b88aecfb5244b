// The trie's plan metadata resident on a device (gt_upload), and the per-process caches the launch paths share:
// shared-memory opt-ins, occupancy and SM count.
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <utility>
#include <vector>

#include "trie_device.cuh"

namespace gt {

void free_device_plan(DevicePlan* d) {
    if (!d) return;
    if (d->blob) {
        int cur = 0;
        cudaGetDevice(&cur);
        cudaSetDevice(d->device);
        cudaFree(d->blob);
        if (d->trace) cudaFree(d->trace);
        cudaSetDevice(cur);
    }
    delete d;
}

static DevicePlan* upload_plan(const Layout& L, const Plan& P, int device) {
    struct Part { const void* src; size_t bytes; size_t off; };
    std::vector<Part> parts;
    size_t total = 0;
    auto add = [&](const void* src, size_t bytes) {
        const size_t off = total;
        parts.push_back({src, bytes, off});
        total += (bytes + 255) & ~size_t(255);
        return off;
    };
#define ADDV(v) add((v).data(), (v).size() * sizeof((v)[0]))
    const size_t o_leaf_dest = ADDV(P.leaf_dest);
    const size_t o_ell_chunk_ptr = ADDV(P.ell_chunk_ptr), o_ell_desc = ADDV(P.ell_desc), o_ell_terms = ADDV(P.ell_terms);
    const size_t o_ell_row_ptr = ADDV(P.ell_row_ptr);
    const size_t o_tile_node_lo = ADDV(P.tile_node_lo), o_node_slot = ADDV(P.node_slot);
    const size_t o_piece_ptr = ADDV(P.piece_ptr), o_piece_slot = ADDV(P.piece_slot), o_piece_idx = ADDV(P.piece_idx);
    const size_t o_span_node = ADDV(P.span_node), o_span_pp = ADDV(P.span_pp);
    std::vector<int32_t> leaf_rank((size_t)L.V);
    for (int64_t r = 0; r < L.V; ++r) leaf_rank[(size_t)L.perm[(size_t)r]] = (int32_t)r;
    const size_t o_leaf_rank = ADDV(leaf_rank), o_node_lo = ADDV(L.lo), o_node_hi = ADDV(L.hi);
    const size_t o_perm = ADDV(L.perm), o_child_ptr = ADDV(L.child_ptr), o_child_idx = ADDV(L.child_idx);
    std::vector<int32_t> child_sym(L.child_idx.size());
    for (size_t e = 0; e < child_sym.size(); ++e) {
        const int32_t lab = L.edge_label[(size_t)L.child_idx[e]];
        child_sym[e] = lab >= 0 ? lab : (int32_t)L.num_symbols;  // leaf child: -1 - item
    }
    const size_t o_child_sym = ADDV(child_sym);
    // post-order ids: a parent's id is larger than its children's, so one descending pass sees every parent first
    std::vector<int32_t> node_depth((size_t)L.N, 0);
    for (int64_t n = L.N - 2; n >= 0; --n)
        node_depth[(size_t)n] = node_depth[(size_t)L.parent[(size_t)n]] + (L.edge_label[(size_t)n] >= 0 ? 1 : 0);
    std::vector<int32_t> item_sym_ptr((size_t)L.V + 1, 0);
    for (int64_t i = 0; i < L.V; ++i) item_sym_ptr[(size_t)i + 1] = item_sym_ptr[(size_t)i] + node_depth[(size_t)L.leaf_node[(size_t)i]];
    std::vector<int32_t> item_sym((size_t)item_sym_ptr[(size_t)L.V]);
    for (int64_t i = 0; i < L.V; ++i) {  // the edge labels from the leaf's parent up to the root, stored back to front
        int32_t at = item_sym_ptr[(size_t)i + 1];
        for (int32_t n = L.parent[(size_t)L.leaf_node[(size_t)i]]; n >= 0 && at > item_sym_ptr[(size_t)i]; n = L.parent[(size_t)n])
            item_sym[(size_t)--at] = L.edge_label[(size_t)n];
    }
    const size_t o_node_depth = ADDV(node_depth), o_item_sym_ptr = ADDV(item_sym_ptr), o_item_sym = ADDV(item_sym);
#undef ADDV
    total += 256;

    int cur = 0;
    if (cudaGetDevice(&cur) != cudaSuccess || cudaSetDevice(device) != cudaSuccess) {
        set_error("cannot select CUDA device %d: %s", device, cudaGetErrorString(cudaGetLastError()));
        return nullptr;
    }
    DevicePlan* d = new DevicePlan();
    d->device = device;
    cudaError_t e = cudaMalloc(&d->blob, total);
    if (e != cudaSuccess) {
        set_error("cudaMalloc(%zu) for trie metadata failed: %s", total, cudaGetErrorString(e));
        d->blob = nullptr;
        cudaSetDevice(cur);
        free_device_plan(d);
        return nullptr;
    }
    d->blob_bytes = total;
    std::vector<unsigned char> host(total, 0);
    for (const Part& p : parts) if (p.bytes) memcpy(host.data() + p.off, p.src, p.bytes);
    e = cudaMemcpy(d->blob, host.data(), total, cudaMemcpyHostToDevice);
    // The source is pageable: the copy may return once the data is staged, before the DMA has finished, and only the
    // legacy stream is ordered after it.  The kernels run on the caller's (possibly non-blocking) streams, so wait for
    // the device here -- once per trie and device.
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    cudaSetDevice(cur);
    if (e != cudaSuccess) {
        set_error("metadata upload failed: %s", cudaGetErrorString(e));
        free_device_plan(d);
        return nullptr;
    }

    unsigned char* base = static_cast<unsigned char*>(d->blob);
    PlanView& v = d->view;
    v.T = P.T; v.logT = 0; while ((1 << (v.logT + 1)) <= P.T) ++v.logT;
    v.NT = P.NT;
    v.SV = (P.max_tile_values + 3) & ~3;
    v.V = L.V; v.N = L.N; v.ZG = (int64_t)P.NT * P.T;
    v.leaf_dest = (const int32_t*)(base + o_leaf_dest);
    v.ell_chunk_ptr = (const int32_t*)(base + o_ell_chunk_ptr); v.ell_desc = (const int2*)(base + o_ell_desc);
    v.ell_terms = (const uint16_t*)(base + o_ell_terms); v.ell_row_ptr = (const int32_t*)(base + o_ell_row_ptr);
    v.R = P.R; v.max_tile_nodes = P.max_tile_nodes; v.max_tile_ell_rows = P.max_tile_ell_rows;
    v.max_tile_chunks = P.max_tile_chunks;
    v.tile_node_lo = (const int32_t*)(base + o_tile_node_lo); v.node_slot = (const uint16_t*)(base + o_node_slot);
    v.piece_ptr = (const int32_t*)(base + o_piece_ptr); v.piece_slot = (const uint16_t*)(base + o_piece_slot);
    v.piece_idx = (const int32_t*)(base + o_piece_idx);
    v.n_span = (int32_t)P.span_node.size(); v.n_pieces = P.n_pieces;
    v.span_node = (const int32_t*)(base + o_span_node); v.span_pp = (const int32_t*)(base + o_span_pp);
    v.leaf_rank = (const int32_t*)(base + o_leaf_rank);
    v.node_lo = (const int32_t*)(base + o_node_lo); v.node_hi = (const int32_t*)(base + o_node_hi);
    v.perm = (const int32_t*)(base + o_perm);
    v.child_ptr = (const int32_t*)(base + o_child_ptr); v.child_idx = (const int32_t*)(base + o_child_idx);
    v.child_sym = (const int32_t*)(base + o_child_sym); v.S = (int32_t)L.num_symbols;
    v.node_depth = (const int32_t*)(base + o_node_depth);
    v.item_sym_ptr = (const int32_t*)(base + o_item_sym_ptr); v.item_sym = (const int32_t*)(base + o_item_sym);
    { const char* e = getenv("GT_DEBUG_STOP"); v.debug_stop = e && *e ? atoi(e) : 0; }
    v.trace = nullptr;
    if (const char* e = getenv("GT_TRACE")) {
        if (*e && atoi(e) != 0) {
            const size_t bytes = (size_t)kTraceCtas * kTraceItems * kTraceEvents * sizeof(long long);
            cudaSetDevice(device);
            if (cudaMalloc(&d->trace, bytes) == cudaSuccess) { cudaMemset(d->trace, 0, bytes); v.trace = d->trace; }
            else { d->trace = nullptr; (void)cudaGetLastError(); }
            cudaSetDevice(cur);
        }
    }
    return d;
}

// Opt in to > 48 KB dynamic shared memory once per (kernel, device, size): the attribute call is kept off the
// steady-state launch path (and out of CUDA graph captures).  Keyed by the kernel's address: instantiations
// with the same signature share a function type.
cudaError_t allow_smem_impl(const void* kernel, size_t bytes) {
    static std::mutex mu;
    static std::map<std::pair<const void*, int>, size_t> granted;
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    std::lock_guard<std::mutex> lock(mu);
    auto key = std::make_pair(kernel, dev);
    auto it = granted.find(key);
    if (it != granted.end() && it->second >= bytes) return cudaSuccess;
    e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e == cudaSuccess) granted[key] = bytes;
    return e;
}

// Resident CTAs per SM of a kernel at a given dynamic shared-memory size (cached: the query is not free).
int resident_ctas(const void* kernel, int threads, size_t smem) {
    static std::mutex mu;
    static std::map<std::pair<const void*, size_t>, int> cache;
    std::lock_guard<std::mutex> lock(mu);
    auto key = std::make_pair(kernel, smem);
    auto it = cache.find(key);
    if (it != cache.end()) return it->second;
    int n = 0;
    // the query honours the kernel's dynamic shared-memory limit: raise it first, or a size above it reports 0
    if (allow_smem_impl(kernel, smem) != cudaSuccess) (void)cudaGetLastError();
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kernel, threads, smem) != cudaSuccess || n < 1) {
        (void)cudaGetLastError();
        n = 1;
    }
    cache[key] = n;
    return n;
}
int sm_count() {
    static std::mutex mu;
    static std::map<int, int> cache;
    int dev = 0;
    cudaGetDevice(&dev);
    std::lock_guard<std::mutex> lock(mu);
    auto it = cache.find(dev);
    if (it != cache.end()) return it->second;
    int n = 148;
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    cache[dev] = n;
    return n;
}

// The plan metadata resident on the current device, for the launches of one call.
int resident_plan(const gt_trie* t, const PlanView*& v) {
    int device = -1;
    GT_CUDA(cudaGetDevice(&device));
    auto it = t->dev.find(device);
    if (it == t->dev.end()) { set_error("trie metadata is not resident on device %d (call gt_upload)", device); return GT_ERR_STATE; }
    v = &it->second->view;
    return GT_OK;
}
}  // namespace gt

extern "C" {

int gt_upload(gt_trie* t, int device) {
    if (!t) { gt::set_error("gt_upload: null trie"); return GT_ERR_ARG; }
    {
        std::lock_guard<std::mutex> lock(t->mu);
        if (t->dev.count(device)) return GT_OK;
    }
    if (!t->plan) {
        const int rc = gt_plan(t, 0);  // takes the lock itself
        if (rc != GT_OK) return rc;
    }
    std::lock_guard<std::mutex> lock(t->mu);
    if (t->dev.count(device)) return GT_OK;  // another thread brought the device up meanwhile
    gt::DevicePlan* d = gt::upload_plan(t->layout, *t->plan, device);
    if (!d) return GT_ERR_CUDA;
    t->dev[device] = d;
    return GT_OK;
}

}  // extern "C"
