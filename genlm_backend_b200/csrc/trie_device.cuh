// Definitions shared by the CUDA translation units of the library (mass_kernels.cu, token_mask_kernels.cu,
// child_kernels.cu, sampler_kernels.cu, device_plan.cu): the resident plan, the launch helpers and the element
// conversions as inline functions and templates, and the host helpers device_plan.cu defines once per process.
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <cuda_bf16.h>

#include <cstddef>

#include "trie_internal.h"

namespace gt {

struct PlanView {
    int32_t T, logT, NT, SV;  // SV = value slots per tile in shared memory (leaves + pyramid + multi-term ranges)
    int32_t R, max_tile_nodes, max_tile_ell_rows, max_tile_chunks;
    int64_t V, N, ZG;         // ZG = NT * T: value slots per row group of the staging buffer
    const int32_t* leaf_dest;  // [V] item position -> value slot of the row group's staging block
    const int32_t* ell_chunk_ptr; const int2* ell_desc; const uint16_t* ell_terms; const int32_t* ell_row_ptr;
    const int32_t* tile_node_lo; const uint16_t* node_slot;
    const int32_t* piece_ptr; const uint16_t* piece_slot; const int32_t* piece_idx;
    int32_t n_span, n_pieces; const int32_t* span_node; const int32_t* span_pp;
    const int32_t* leaf_rank;  // [V] DFS rank of each item's leaf (inverse of Layout::perm)
    const int32_t* node_lo; const int32_t* node_hi;  // [N] DFS leaf range of every node
    const int32_t* perm;       // [V] DFS rank -> item position (Layout::perm)
    const int32_t* child_ptr; const int32_t* child_idx;  // children CSR (ascending ids = jump[] order)
    const int32_t* child_sym;  // [N - 1] beside child_idx: the child's edge symbol, S for a leaf child
    int32_t S;                 // Layout::num_symbols
    const int32_t* node_depth;                             // [N] symbols on the path root -> node (a leaf edge adds none)
    const int32_t* item_sym_ptr; const int32_t* item_sym;  // [V+1] CSR of every item's symbols, in item order
    int32_t debug_stop;  // profiling aid (GT_DEBUG_STOP): 0 = normal; 3 = no emit stores; 9 = emit only
    long long* trace;    // profiling aid (GT_TRACE=1): per (CTA, item) SM-clock stamps of the pipeline events, else null
};

struct DevicePlan {
    int device = -1;
    void* blob = nullptr;  // one allocation holding all metadata
    size_t blob_bytes = 0;
    PlanView view{};
    long long* trace = nullptr;  // GT_TRACE=1 only
};

#define GT_CUDA(call)                                                                     \
    do {                                                                                  \
        cudaError_t e_ = (call);                                                          \
        if (e_ != cudaSuccess) {                                                          \
            gt::set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
            (void)cudaGetLastError(); /* do not leave the error for the next, unrelated call */        \
            return GT_ERR_CUDA;                                                           \
        }                                                                                 \
    } while (0)

// ---- programmatic dependent launch ---------------------------------------------------------------------
// Consecutive kernels of one call (mass -> span -> mass -> span ...) are launched with the programmatic
// stream-serialisation attribute: a kernel's launch set-up and prologue overlap the tail of its predecessor, and
// pdl_wait() -- executed before the first access to memory another kernel of the chain touches -- blocks until the
// predecessor grid has completed and flushed.  pdl_trigger() lets the successor's CTAs start launching.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

template <typename... KArgs, typename... Args>
cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

// ---- element conversion -----------------------------------------------------------------------------------
// in_to_float: an input element as fp32.  convert_in: as the value type VT of a reduction, exponentiated for log-space
// rows (GT_FLAG_LOG_INPUT); fp64 elements skip the fp32 step.

template <typename IN_T> __device__ __forceinline__ float in_to_float(IN_T x);
template <> __device__ __forceinline__ float in_to_float<float>(float x) { return x; }
template <> __device__ __forceinline__ float in_to_float<double>(double x) { return (float)x; }
template <> __device__ __forceinline__ float in_to_float<__half>(__half x) { return __half2float(x); }
template <> __device__ __forceinline__ float in_to_float<__nv_bfloat16>(__nv_bfloat16 x) { return __bfloat162float(x); }

template <typename VT, typename IN_T> __device__ __forceinline__ VT convert_in(IN_T x, bool log_input) {
    if constexpr (sizeof(IN_T) == 8) {
        const double d = log_input ? exp((double)x) : (double)x;
        return (VT)d;
    } else {
        const float f = in_to_float<IN_T>(x);
        if constexpr (sizeof(VT) == 8) return log_input ? exp((double)f) : (double)f;
        else return log_input ? expf(f) : f;
    }
}

// Input-type dispatch (one switch per warp; the loops inside are type-specific).
#define GT_IN_TYPE_SWITCH(in_type, CALL)                          \
    switch (in_type) {                                            \
        case GT_F32: { using IN_T = float; CALL; } break;         \
        case GT_F64: { using IN_T = double; CALL; } break;        \
        case GT_F16: { using IN_T = __half; CALL; } break;        \
        default: { using IN_T = __nv_bfloat16; CALL; } break;     \
    }

// Profiling trace (GT_TRACE=1): [kTraceCtas][kTraceItems][kTraceEvents] SM-clock stamps.  upload_plan sizes the
// buffer, mass_kernel writes it.
constexpr int kTraceCtas = 512, kTraceItems = 32, kTraceEvents = 12;

// ---- host helpers (device_plan.cu) ----------------------------------------------------------------------------
// Hidden: the library exports the C ABI, not these.
#define GT_HIDDEN __attribute__((visibility("hidden")))

// The plan metadata resident on the current device, for the launches of one call.
GT_HIDDEN int resident_plan(const gt_trie* t, const PlanView*& v);
// Opt in to `bytes` of dynamic shared memory for a kernel (once per kernel, device and size).
GT_HIDDEN cudaError_t allow_smem_impl(const void* kernel, size_t bytes);
template <typename K> cudaError_t allow_smem(K kernel, size_t bytes) {
    return allow_smem_impl(reinterpret_cast<const void*>(kernel), bytes);
}
// Resident CTAs per SM of a kernel at a given dynamic shared-memory size.
GT_HIDDEN int resident_ctas(const void* kernel, int threads, size_t smem);
// SMs of the current device.
GT_HIDDEN int sm_count();

inline bool ops_ok(unsigned ops) { return (ops & (GT_OP_SUM | GT_OP_MAX)) && !(ops & ~(unsigned)(GT_OP_SUM | GT_OP_MAX)); }

// Bytes per element of a GT_* input type; 0 for an unknown type.
inline size_t in_type_size(int in_type) {
    switch (in_type) {
        case GT_F64: return 8;
        case GT_F32: return 4;
        case GT_F16: case GT_BF16: return 2;
        default: return 0;
    }
}

}  // namespace gt
