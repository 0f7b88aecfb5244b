// sm_100a kernels for the trie mass path (weight_sum / weight_max over a batch of rows).
//
// Replaces genlm/backend/trie/parallel.py:92-145 (sparse.mm / scatter_reduce amax) and
// genlm/backend/trie/base.py:346-393 (numba loops).  HBM-bound streaming work: no tensor cores; the design rules
// are coalesced global access, shared-memory staging of every irregular access, bulk copies (TMA) for everything
// that is contiguous, and one persistent grid that keeps HBM busy from the first row to the last.
//
// A reduction is three launches, chained with programmatic dependent launch:
//   permute_kernel  reads the rows in vocabulary order (coalesced) and writes every weight to its DFS leaf slot of
//                   the staging buffer z (16-byte scattered stores that stay in L2):
//                   z[row group][tile][leaf slot][row] is, tile by tile, the leaf region of the tile's shared-memory
//                   value array, so the tile kernel needs no scatter phase of its own;
//   mass_kernel     persistent, warp-specialised: a producer thread fetches (row group, tile) pairs -- leaf block +
//                   tile metadata -- by bulk copies (TMA); compute warps build the aligned-block pyramid (warp
//                   shuffles) and the multi-term ranges (ELL-packed term lists); emit warps stream the tile's node-id
//                   interval out with coalesced stores and write the spanning-node pieces;
//   span_kernel     the few nodes whose leaf range crosses tiles, reduced from their pieces (fp64 for sums).
// (Variants that hide the permute inside mass_kernel were built and measured in round 2 and are not here: publishing
// permuted row groups to other SMs of the same launch needs a device-scope fence, which takes ~10 us on an SM saturated
// with output stores; staging the *next* launch's rows from the producer warp works but one warp per CTA is 2.5x too
// slow, and rider code in the other warps costs the tile work 9 us of register allocation; profiles/r02_experiments.md.)
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <cuda_bf16.h>

#include <climits>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <type_traits>
#include <algorithm>
#include <map>
#include <mutex>
#include <utility>

#include "trie_internal.h"
#include "philox.cuh"

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
    bool attrs_set = false;
    long long* trace = nullptr;  // GT_TRACE=1 only
};

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

#define GT_CUDA(call)                                                                     \
    do {                                                                                  \
        cudaError_t e_ = (call);                                                          \
        if (e_ != cudaSuccess) {                                                          \
            gt::set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
            (void)cudaGetLastError(); /* do not leave the error for the next, unrelated call */        \
            return GT_ERR_CUDA;                                                           \
        }                                                                                 \
    } while (0)

constexpr int OP_SUM = 1, OP_MAX = 2;

// ---- programmatic dependent launch ---------------------------------------------------------------------
// Consecutive kernels of one call (mass -> span -> mass -> span ...) are launched with the programmatic
// stream-serialisation attribute: a kernel's launch set-up and prologue overlap the tail of its predecessor, and
// pdl_wait() -- executed before the first access to memory another kernel of the chain touches -- blocks until the
// predecessor grid has completed and flushed.  pdl_trigger() lets the successor's CTAs start launching.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

template <typename... KArgs, typename... Args>
static cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

// ---- small device helpers -----------------------------------------------------------------------

template <int OP, typename VT> __device__ __forceinline__ VT op_apply(VT a, VT b) {
    if constexpr (OP == OP_SUM) return a + b;
    else return fmax(a, b);  // fmaxf/fmax overloads; NaN operands are ignored like numba's max()
}
template <int OP, typename VT> __device__ __forceinline__ VT op_ident() {
    if constexpr (OP == OP_SUM) return VT(0);
    else return -std::numeric_limits<VT>::infinity();
}

__device__ __forceinline__ uint4 ldg_stream(const uint4* p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}

template <typename VT> struct Vec4;
template <> struct Vec4<float> { using type = float4; };
template <> struct Vec4<double> { using type = double4; };

template <typename VT> __device__ __forceinline__ void store4(VT* p, VT a, VT b, VT c, VT d);
template <> __device__ __forceinline__ void store4<float>(float* p, float a, float b, float c, float d) {
    *reinterpret_cast<float4*>(p) = make_float4(a, b, c, d);
}
template <> __device__ __forceinline__ void store4<double>(double* p, double a, double b, double c, double d) {
    reinterpret_cast<double2*>(p)[0] = make_double2(a, b);
    reinterpret_cast<double2*>(p)[1] = make_double2(c, d);
}
template <typename VT> __device__ __forceinline__ void store4_stream(VT* p, VT a, VT b, VT c, VT d);
template <> __device__ __forceinline__ void store4_stream<float>(float* p, float a, float b, float c, float d) {
    __stcs(reinterpret_cast<float4*>(p), make_float4(a, b, c, d));
}
template <> __device__ __forceinline__ void store4_stream<double>(double* p, double a, double b, double c, double d) {
    __stcs(reinterpret_cast<double2*>(p), make_double2(a, b));
    __stcs(reinterpret_cast<double2*>(p) + 1, make_double2(c, d));
}
template <typename VT> __device__ __forceinline__ void load4(const VT* p, VT& a, VT& b, VT& c, VT& d);
template <> __device__ __forceinline__ void load4<float>(const float* p, float& a, float& b, float& c, float& d) {
    const float4 v = *reinterpret_cast<const float4*>(p);
    a = v.x; b = v.y; c = v.z; d = v.w;
}
template <> __device__ __forceinline__ void load4<double>(const double* p, double& a, double& b, double& c, double& d) {
    const double2 u = reinterpret_cast<const double2*>(p)[0], w = reinterpret_cast<const double2*>(p)[1];
    a = u.x; b = u.y; c = w.x; d = w.y;
}

template <typename IN_T> __device__ __forceinline__ float in_to_float(IN_T x);
template <> __device__ __forceinline__ float in_to_float<float>(float x) { return x; }
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


// mbarrier + bulk-copy (TMA) primitives.  One elected thread arms the barrier with the byte count and issues the
// copies; the copy engine signals the barrier when the bytes have landed, so no LSU instruction is spent per 16 bytes.
__device__ __forceinline__ void mbar_init(uint64_t* b, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(b)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* b, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(b)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* b, unsigned parity) {
    const unsigned addr = (unsigned)__cvta_generic_to_shared(b);
    unsigned done;
    for (;;) {  // try_wait suspends the thread in hardware for a bounded time; back off between polls so that
                // waiting warps do not take issue slots from the working ones
        asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}\n"
                     : "=r"(done) : "r"(addr), "r"(parity) : "memory");
        if (done) break;
        __nanosleep(40);
    }
}
// bytes: multiple of 16; both addresses 16-byte aligned
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gsrc, unsigned bytes, uint64_t* b) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     (unsigned)__cvta_generic_to_shared(smem_dst)),
                 "l"(gsrc), "r"(bytes), "r"((unsigned)__cvta_generic_to_shared(b))
                 : "memory");
}

// Device twin of gt::swizzle_slot (trie_internal.h) for slots below 2T; B = bytes per slot.
template <int B> __device__ __forceinline__ int swz(int s) {
    constexpr int cs = B == 4 ? 2 : (B == 8 ? 1 : 0);
    const int c = s >> cs;
    return ((c ^ ((c >> 3) & (B / 2 - 1))) << cs) | (s & ((1 << cs) - 1));
}

// R consecutive rows share a CTA and live interleaved in shared memory: vals[slot * R + r].  One vector
// shared-memory access then serves all R rows of a slot.
template <typename VT, int R> struct RowVec {
    VT v[R];
    __device__ __forceinline__ static RowVec load(const VT* p) {
        RowVec x;
        if constexpr (sizeof(VT) * R == 8) { const float2 t = *reinterpret_cast<const float2*>(p); memcpy(x.v, &t, 8); }
        else if constexpr (sizeof(VT) * R == 16) { const float4 t = *reinterpret_cast<const float4*>(p); memcpy(x.v, &t, 16); }
        else {
#pragma unroll
            for (int r = 0; r < R; ++r) x.v[r] = p[r];
        }
        return x;
    }
    __device__ __forceinline__ void store(VT* p) const {
        if constexpr (sizeof(VT) * R == 8) { float2 t; memcpy(&t, v, 8); *reinterpret_cast<float2*>(p) = t; }
        else if constexpr (sizeof(VT) * R == 16) { float4 t; memcpy(&t, v, 16); *reinterpret_cast<float4*>(p) = t; }
        else {
#pragma unroll
            for (int r = 0; r < R; ++r) p[r] = v[r];
        }
    }
    template <int OP> __device__ __forceinline__ static RowVec combine(const RowVec& a, const RowVec& b) {
        RowVec x;
#pragma unroll
        for (int r = 0; r < R; ++r) x.v[r] = op_apply<OP>(a.v[r], b.v[r]);
        return x;
    }
    template <int OP> __device__ __forceinline__ static RowVec ident() {
        RowVec x;
#pragma unroll
        for (int r = 0; r < R; ++r) x.v[r] = op_ident<OP, VT>();
        return x;
    }
    __device__ __forceinline__ RowVec shfl_down(int delta) const {
        RowVec x;
#pragma unroll
        for (int r = 0; r < R; ++r) x.v[r] = __shfl_down_sync(0xffffffffu, v[r], delta);
        return x;
    }
};

// Streaming stores of one slot's R row values to R row pointers at a compile-time byte offset, all under one
// predicate: address = register + immediate, so a store is one instruction and no pointer is recomputed per store.
template <int OFF, typename VT, int R> struct EmitStore {
    __device__ __forceinline__ static void run(VT* const (&p)[R], const RowVec<VT, R>& x, bool ok) {
        if (ok) {
#pragma unroll
            for (int r = 0; r < R; ++r) __stcs(reinterpret_cast<VT*>(reinterpret_cast<unsigned char*>(p[r]) + OFF), x.v[r]);
        }
    }
};
template <int OFF> struct EmitStore<OFF, float, 4> {
    __device__ __forceinline__ static void run(float* const (&p)[4], const RowVec<float, 4>& x, bool ok) {
        asm volatile(
            "{\n.reg .pred q;\nsetp.ne.u32 q, %8, 0;\n"
            "@q st.global.cs.f32 [%0+%9], %4;\n@q st.global.cs.f32 [%1+%9], %5;\n"
            "@q st.global.cs.f32 [%2+%9], %6;\n@q st.global.cs.f32 [%3+%9], %7;\n}\n" ::"l"(p[0]), "l"(p[1]), "l"(p[2]), "l"(p[3]),
            "f"(x.v[0]), "f"(x.v[1]), "f"(x.v[2]), "f"(x.v[3]), "r"((unsigned)ok), "n"(OFF)
            : "memory");
    }
};
template <int OFF> struct EmitStore<OFF, double, 2> {
    __device__ __forceinline__ static void run(double* const (&p)[2], const RowVec<double, 2>& x, bool ok) {
        asm volatile(
            "{\n.reg .pred q;\nsetp.ne.u32 q, %4, 0;\n"
            "@q st.global.cs.f64 [%0+%5], %2;\n@q st.global.cs.f64 [%1+%5], %3;\n}\n" ::"l"(p[0]), "l"(p[1]), "d"(x.v[0]), "d"(x.v[1]),
            "r"((unsigned)ok), "n"(OFF)
            : "memory");
    }
};


// ---- the tile kernel -----------------------------------------------------------------------------------------------
//
// Work decomposition.  A *pair* is (row group g of R rows, tile t); pairs are numbered g-major (p = g * NT + t) and
// CTA b takes pairs b, b + grid, b + 2 grid, ....  A pair holds one *item* per requested reduction (sum, then max);
// both items read the same leaf block.
//
// Shared memory of a CTA:
//     leaf[2]   leaf blocks of the current and the next pair (T slots of 16 bytes: R rows interleaved per slot)
//     rest[2]   pyramid + multi-term-range slots of the item being built and the item being drained
//     meta[2]   per pair: ELL term rows + chunk descriptors (compute group), node -> slot table (emit group), header
// and eight mbarriers:
//     pairFull[2]   bulk copies of a pair have landed (producer -> both groups)
//     pairEmpty[2]  the emit group has drained the last item of the pair (-> producer)
//     full[2] / empty[2]   hand-over of the rest buffers between compute and emit group, per item
constexpr int kThreads = 512;
#ifndef GT_COMPUTE_WARPS
#define GT_COMPUTE_WARPS 7
#endif
#ifndef GT_EMIT_WARPS
#define GT_EMIT_WARPS 8
#endif
constexpr int kComputeWarps = GT_COMPUTE_WARPS, kEmitWarps = GT_EMIT_WARPS;
constexpr int kProducerWarp = kComputeWarps + kEmitWarps;  // one warp: lane 0 issues every bulk copy
static_assert(kProducerWarp + 1 == kThreads / 32, "compute + emit + producer warps fill the CTA");
constexpr int kComputeThreads = 32 * kComputeWarps, kEmitThreads = 32 * kEmitWarps;
#ifndef GT_PERM_UT
#define GT_PERM_UT 128
#endif
constexpr int kUnitTokens = GT_PERM_UT;  // vocabulary positions per permute unit (half for fp64 rows)

#ifndef GT_ELL_BATCH
#define GT_ELL_BATCH 4
#endif

// trace layout: [kTraceCtas][kTraceItems][kTraceEvents] SM-clock stamps
constexpr int kTraceCtas = 512, kTraceItems = 32, kTraceEvents = 12;
#define GT_TRACE(ev)                                                                                         \
    do {                                                                                                     \
        if (P.trace && gtid == 0 && blockIdx.x < kTraceCtas && k < kTraceItems)                               \
            P.trace[((size_t)blockIdx.x * kTraceItems + k) * kTraceEvents + (ev)] = clock64();               \
    } while (0)
#define GT_PTRACE(cond, kk, ev)                                                                              \
    do {                                                                                                     \
        if (P.trace && (cond) && blockIdx.x < kTraceCtas && (kk) < kTraceItems)                               \
            P.trace[((size_t)blockIdx.x * kTraceItems + (kk)) * kTraceEvents + (ev)] = clock64();            \
    } while (0)

// Shared-memory carve-up of mass_kernel (all sections 128-byte aligned: the bank group of a slot is slot % 8 in
// the leaf blocks and in the rest buffers alike).
struct MassSmem {
    size_t leaf, leaf_bytes, rest, rest_bytes, meta, meta_bytes, terms, desc, slots, hdr, bars, total;
    __host__ __device__ MassSmem(const PlanView& P, int slot_bytes) {
        auto up = [](size_t x) { return (x + 127) & ~size_t(127); };
        size_t o = 0;
        leaf_bytes = up((size_t)P.T * slot_bytes);
        leaf = o; o += 2 * leaf_bytes;
        rest_bytes = up((size_t)(P.SV - P.T) * slot_bytes);
        rest = o; o += 2 * rest_bytes;
        // inside one pair's metadata block
        size_t m = 0;
        terms = m; m += up((size_t)P.max_tile_ell_rows * 64);
        desc = m;  m += up((size_t)(P.max_tile_chunks + 2) * 8);
        slots = m; m += up((size_t)P.max_tile_nodes * 2 + 16);
        hdr = m;   m += 128;
        meta_bytes = m;
        meta = o; o += 2 * meta_bytes;
        bars = o; o += 128;
        total = o;
    }
};

__device__ __forceinline__ void mbar_arrive(uint64_t* b) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"((unsigned)__cvta_generic_to_shared(b)) : "memory");
}
template <int ID, int COUNT> __device__ __forceinline__ void group_sync() {
    asm volatile("bar.sync %0, %1;" ::"n"(ID), "n"(COUNT) : "memory");
}

// What one launch works on.
template <typename VT> struct MassArgs {
    const void* ws; int in_type; int log_input; int64_t ld_ws;
    int dfs_order;  // the rows are already in DFS leaf order (GT_FLAG_DFS_ORDER): destinations are computed, not looked up
    VT* z;
    VT* out_sum; VT* out_max;
    VT* part_sum; VT* part_max;
    int64_t ld_out;
    int n_rows;
    unsigned ops;
};

// ---- permute ---------------------------------------------------------------------------------------------------
// Unit w = (row group g, positions [u * UT, (u + 1) * UT)), UT = 128 (64 for fp64 rows); one warp per unit, a grid
// sized to the job.  Lane l handles positions u * UT + l + 32 j: coalesced loads of the R rows and of leaf_dest, all
// in flight at once, then one 16-byte store per position holding the R rows' weights (exp / conversion fused).  The
// stores are scattered -- every lane its own line of z -- which an SM retires at ~1.6 cycles each when they hit L2
// (tools/scatter_store_probe.cu); that, not HBM, bounds this kernel.  Rows past the end of the batch alias the last
// valid row; nothing outside a row's V elements is read, whatever the alignment.
__device__ __forceinline__ int perm_unit_tokens_rt(int in_type) { return in_type == GT_F64 ? kUnitTokens / 2 : kUnitTokens; }

template <typename VT, typename IN_T, int R>
__device__ __forceinline__ void permute_unit(const PlanView& P, const MassArgs<VT>& A, unsigned w, int n_units, int lane) {
    using RV = RowVec<VT, R>;
    constexpr int UT = sizeof(IN_T) == 8 ? kUnitTokens / 2 : kUnitTokens, TPL = UT / 32;
    const bool log_input = A.log_input != 0;
    const int g = (int)(w / (unsigned)n_units), v0 = (int)(w - (unsigned)g * (unsigned)n_units) * UT;
    const int ntok = min(UT, (int)P.V - v0);
    const IN_T* __restrict__ ws = static_cast<const IN_T*>(A.ws);
    VT* zg = A.z + (size_t)g * P.ZG * R;
    int dst[TPL];
    IN_T x[TPL][R];
    const bool dfs = A.dfs_order != 0;
#pragma unroll
    for (int j = 0; j < TPL; ++j) {
        const int i = min(lane + 32 * j, ntok - 1);
        // position = DFS rank r: slot of leaf r % T in tile r / T (what leaf_dest holds for the item of rank r); consecutive
        // positions then go to consecutive slots and a warp's stores cover whole lines
        const int r = v0 + i;
        dst[j] = dfs ? ((r & ~(P.T - 1)) | swz<(int)sizeof(VT) * R>(r & (P.T - 1))) : __ldg(P.leaf_dest + r);
#pragma unroll
        for (int r = 0; r < R; ++r) x[j][r] = ws[(size_t)min(g * R + r, A.n_rows - 1) * A.ld_ws + v0 + i];
    }
#pragma unroll
    for (int j = 0; j < TPL; ++j) {
        if (lane + 32 * j < ntok) {
            RV y;
#pragma unroll
            for (int r = 0; r < R; ++r) y.v[r] = convert_in<VT, IN_T>(x[j][r], log_input);
            y.store(zg + (size_t)dst[j] * R);
        }
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

#ifndef GT_PERM_THREADS
#define GT_PERM_THREADS 256
#endif
#ifndef GT_PERM_MINB
#define GT_PERM_MINB 1
#endif
constexpr int kPermThreads = GT_PERM_THREADS;
template <typename VT, int R>
__global__ void __launch_bounds__(kPermThreads, GT_PERM_MINB) permute_kernel(PlanView P, MassArgs<VT> A, unsigned total_units) {
    pdl_wait();  // the rows may come from the previous kernel of the stream; z may still be read by the previous call
    pdl_trigger();
    const unsigned w = blockIdx.x * (kPermThreads / 32) + (threadIdx.x >> 5);
    if (w >= total_units) return;
    const int UT = perm_unit_tokens_rt(A.in_type);
    const int n_units = (int)((P.V + UT - 1) / UT);
    GT_IN_TYPE_SWITCH(A.in_type, (permute_unit<VT, IN_T, R>(P, A, w, n_units, (int)(threadIdx.x & 31))));
}

// ---- compute-group phases (OP is a compile-time parameter; the kernel branches once per phase) ----------------------
// Value slot s lives in the pair's leaf block when s < T and in the item's rest buffer otherwise; `restv` is biased
// by -T slots so that both cases are base + s * R.

// 1. pyramid of aligned blocks: level k block i at (swizzled) slot 2T - (T >> (k-1)) + i, levels 1 .. kPyramidTop.
//    Lane u owns 8 consecutive leaves: three levels in registers, five more by warp shuffles, so a warp covers 256
//    leaves and no level needs a cross-warp step (longer aligned blocks are multi-term ranges of the ELL phase).
//    The swizzle makes the 16-byte chunk loads and the strided level stores bank-conflict free.
template <typename VT, int R, int OP, int NWARPS>
__device__ __forceinline__ void phase_pyramid(const VT* leafv, VT* restv, int T, int warp, int lane) {
    using RV = RowVec<VT, R>;
    constexpr int B = (int)sizeof(VT) * R;
    constexpr int SPC = 16 / B;  // slots per 16-byte chunk
    static_assert(kPyramidTop == 8, "the pyramid is written for 8 leaves per lane");
    auto level_slot = [&](int k, int i) { return 2 * T - (T >> (k - 1)) + i; };  // level k >= 1, block i
    for (int ub = warp * 32; ub < (T >> 3); ub += NWARPS * 32) {
        const int u = ub + lane;
        RV x[8];
#pragma unroll
        for (int ch = 0; ch < 8 / SPC; ++ch) {
            const int c = (8 * u) / SPC + ch;
            const int cc = c ^ ((c >> 3) & (B / 2 - 1));
            const float4 raw = *reinterpret_cast<const float4*>(reinterpret_cast<const unsigned char*>(leafv) + (size_t)cc * 16);
            memcpy(&x[ch * SPC], &raw, 16);
        }
        RV a[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            a[e] = RV::template combine<OP>(x[2 * e], x[2 * e + 1]);
            a[e].store(restv + swz<B>(level_slot(1, 4 * u + e)) * R);
        }
        const RV c0 = RV::template combine<OP>(a[0], a[1]), c1 = RV::template combine<OP>(a[2], a[3]);
        c0.store(restv + swz<B>(level_slot(2, 2 * u)) * R);
        c1.store(restv + swz<B>(level_slot(2, 2 * u + 1)) * R);
        RV y = RV::template combine<OP>(c0, c1);
        y.store(restv + swz<B>(level_slot(3, u)) * R);
#pragma unroll
        for (int j = 1; j <= 5; ++j) {
            y = RV::template combine<OP>(y, y.shfl_down(1 << (j - 1)));
            if ((lane & ((1 << j) - 1)) == 0) y.store(restv + swz<B>(level_slot(3 + j, u >> j)) * R);
        }
    }
}

// 2. ranges that need more than one block: ELL chunks of 32 ranges, one warp per chunk, term rows read from shared
//    memory.  Chunks are sorted by descending term count: rounds alternate direction so that the warps that drew the
//    longest chunks of one round draw the shortest of the next.
template <typename VT, int R, int OP, int NWARPS>
__device__ __forceinline__ void phase_ell(const VT* leafv, VT* restv, const uint16_t* s_terms, const int2* dsc, int er0,
                                          int nchunks, int T, int warp, int lane) {
    using RV = RowVec<VT, R>;
    auto val = [&](int sl) { return RV::load((sl < T ? leafv : (const VT*)restv) + sl * R); };
    for (int base = 0, rr = 0; base < nchunks; base += NWARPS, ++rr) {
        const int c = base + ((rr & 1) ? NWARPS - 1 - warp : warp);
        if (c >= nchunks) continue;
        const int2 d = dsc[c];
        const uint16_t* tp = s_terms + (d.x - er0) * 32 + lane;
        RV acc = RV::template ident<OP>();
        int kb = 0;
        for (; kb + 4 <= d.y; kb += 4) {
            int sl[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) sl[e] = tp[(kb + e) * 32];
#pragma unroll
            for (int e = 0; e < 4; ++e) acc = RV::template combine<OP>(acc, val(sl[e]));
        }
        if (kb + 2 <= d.y) {  // no padding rows: a pair, then a single term
            const int s0 = tp[kb * 32], s1 = tp[(kb + 1) * 32];
            acc = RV::template combine<OP>(acc, RV::template combine<OP>(val(s0), val(s1)));
            kb += 2;
        }
        if (kb < d.y) acc = RV::template combine<OP>(acc, val((int)tp[kb * 32]));
        acc.store(restv + (2 * T + c * 32 + lane) * R);
    }
}

// header of a fetched pair (written by the producer thread before it arms pairFull)
struct PairHdr { int t, g, n0, n1, er0, ec0, nchunks, pc0, pc1; };

template <typename VT, int R>
__global__ void __launch_bounds__(kThreads, 2) mass_kernel(PlanView P, MassArgs<VT> A) {
    using RV = RowVec<VT, R>;
    constexpr int B = (int)sizeof(VT) * R;  // bytes per slot
    static_assert(B == 16, "value slots are 16 bytes");
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const MassSmem L(P, B);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw + L.bars);
    uint64_t* pairFull = bars;       // [2]
    uint64_t* pairEmpty = bars + 2;  // [2]
    uint64_t* full = bars + 4;       // [2] rest buffer filled by the compute group
    uint64_t* empty = bars + 6;      // [2] rest buffer drained by the emit group

    const int T = P.T;
    const int n_rows = A.n_rows;
    const int RG = (n_rows + R - 1) / R;
    const int nops = (A.ops == (unsigned)(GT_OP_SUM | GT_OP_MAX)) ? 2 : 1;
    const int first_op = (A.ops & GT_OP_SUM) ? OP_SUM : OP_MAX;
    const int G = (int)gridDim.x;
    const int n_pairs = P.NT * RG;
    const int my_pairs = (int)blockIdx.x < n_pairs ? (n_pairs - (int)blockIdx.x + G - 1) / G : 0;
    const int dbg = P.debug_stop;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (threadIdx.x == 0) {
        mbar_init(pairFull, 1); mbar_init(pairFull + 1, 1);
        mbar_init(pairEmpty, kEmitThreads); mbar_init(pairEmpty + 1, kEmitThreads);
        mbar_init(full, kComputeThreads); mbar_init(full + 1, kComputeThreads);
        mbar_init(empty, kEmitThreads); mbar_init(empty + 1, kEmitThreads);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    GT_PTRACE(threadIdx.x == 0, kTraceItems - 1, 11);  // CTA start

    if (warp == kProducerWarp) {
        // =========================== producer: one thread fetches pair after pair ====================================
        // Plan metadata may be fetched while the permute kernel is still running (programmatic dependent launch); the
        // leaf blocks may not: griddepcontrol.wait precedes the first one.
        if (lane == 0) {
            for (int q = 0; q < my_pairs; ++q) {
                const int p = (int)blockIdx.x + q * G;
                const int g = p / P.NT, t = p - g * P.NT;
                const int buf = q & 1;
                unsigned char* meta = smem_raw + L.meta + (size_t)buf * L.meta_bytes;
                // tile boundaries (independent loads, one round trip, requested before the wait for the buffers)
                const int n0 = __ldg(P.tile_node_lo + t), n1 = __ldg(P.tile_node_lo + t + 1);
                const int er0 = __ldg(P.ell_row_ptr + t), er1 = __ldg(P.ell_row_ptr + t + 1);
                const int ec0 = __ldg(P.ell_chunk_ptr + t), ec1 = __ldg(P.ell_chunk_ptr + t + 1);
                const int pc0 = __ldg(P.piece_ptr + t), pc1 = __ldg(P.piece_ptr + t + 1);
                mbar_wait(pairEmpty + buf, ((unsigned)(q >> 1) & 1u) ^ 1u);  // the pair two back has been drained
                PairHdr* h = reinterpret_cast<PairHdr*>(meta + L.hdr);
                h->t = t; h->g = g; h->n0 = n0; h->n1 = n1; h->er0 = er0; h->ec0 = ec0; h->nchunks = ec1 - ec0;
                h->pc0 = pc0; h->pc1 = pc1;
                const int ea = ec0 & ~1, na = n0 & ~7;
                const unsigned lb = (unsigned)T * (unsigned)B;
                const unsigned tb = (unsigned)(er1 - er0) * 64u, db = (unsigned)((ec1 - ea + 1) >> 1) * 16u;
                const unsigned sb = (unsigned)((n1 - na + 7) >> 3) * 16u;
                mbar_expect_tx(pairFull + buf, lb + tb + db + sb);
                if (tb) bulk_g2s(meta + L.terms, P.ell_terms + (size_t)er0 * 32, tb, pairFull + buf);
                if (db) bulk_g2s(meta + L.desc, P.ell_desc + ea, db, pairFull + buf);
                bulk_g2s(meta + L.slots, P.node_slot + na, sb, pairFull + buf);
                if (q == 0) { pdl_wait(); pdl_trigger(); }  // z comes from permute_kernel
                bulk_g2s(smem_raw + L.leaf + (size_t)buf * L.leaf_bytes, A.z + ((size_t)g * P.ZG + (size_t)t * T) * R, lb, pairFull + buf);
                if (q == 0) GT_PTRACE(true, kTraceItems - 1, 0);
            }
        }
    } else {
        if (warp < kComputeWarps) {
            // =========================== compute group ===========================================================
            const int gtid = threadIdx.x;
            for (int q = 0; q < my_pairs; ++q) {
                const int buf = q & 1;
                const unsigned char* meta = smem_raw + L.meta + (size_t)buf * L.meta_bytes;
                mbar_wait(pairFull + buf, (unsigned)(q >> 1) & 1u);
                const PairHdr* h = reinterpret_cast<const PairHdr*>(meta + L.hdr);
                const int er0 = h->er0, ec0 = h->ec0, nchunks = h->nchunks;
                const uint16_t* s_terms = reinterpret_cast<const uint16_t*>(meta + L.terms);
                const int2* dsc = reinterpret_cast<const int2*>(meta + L.desc) + (ec0 & 1);
                const VT* leafv = reinterpret_cast<const VT*>(smem_raw + L.leaf + (size_t)buf * L.leaf_bytes);
                for (int j = 0; j < nops; ++j) {
                    const int k = q * nops + j;
                    VT* restv = reinterpret_cast<VT*>(smem_raw + L.rest + (size_t)(k & 1) * L.rest_bytes) - (size_t)T * R;
                    const bool is_sum = (j == 0 ? first_op : OP_MAX) == OP_SUM;
                    GT_TRACE(0);
                    mbar_wait(empty + (k & 1), ((unsigned)(k >> 1) & 1u) ^ 1u);  // the emit group has drained this rest buffer
                    GT_TRACE(1);
                    if (dbg != 9) {
                        if (is_sum) phase_pyramid<VT, R, OP_SUM, kComputeWarps>(leafv, restv, T, warp, lane);
                        else phase_pyramid<VT, R, OP_MAX, kComputeWarps>(leafv, restv, T, warp, lane);
                    }
                    if (gtid == kComputeThreads - 1) {  // identity slot (spanning nodes' placeholder)
                        if (is_sum) RV::template ident<OP_SUM>().store(restv + swz<B>(2 * T - 1) * R);
                        else RV::template ident<OP_MAX>().store(restv + swz<B>(2 * T - 1) * R);
                    }
                    GT_TRACE(2);
                    group_sync<1, kComputeThreads>();
                    GT_TRACE(3);
                    if (dbg != 9) {
                        if (is_sum) phase_ell<VT, R, OP_SUM, kComputeWarps>(leafv, restv, s_terms, dsc, er0, nchunks, T, warp, lane);
                        else phase_ell<VT, R, OP_MAX, kComputeWarps>(leafv, restv, s_terms, dsc, er0, nchunks, T, warp, lane);
                    }
                    GT_TRACE(4);
                    mbar_arrive(full + (k & 1));  // this thread's share of the value array is complete
                }
            }
        } else if (warp < kProducerWarp) {
            // =========================== emit group ==============================================================
            const int gtid = threadIdx.x - kComputeThreads;
            pdl_wait();  // the outputs and piece buffers may still be in use by the previous kernels of the stream
            for (int q = 0; q < my_pairs; ++q) {
                const int buf = q & 1;
                const unsigned char* meta = smem_raw + L.meta + (size_t)buf * L.meta_bytes;
                mbar_wait(pairFull + buf, (unsigned)(q >> 1) & 1u);
                const PairHdr* h = reinterpret_cast<const PairHdr*>(meta + L.hdr);
                const int g = h->g, n0 = h->n0, n1 = h->n1, pc0 = h->pc0, pc1 = h->pc1;
                const uint16_t* s_slots = reinterpret_cast<const uint16_t*>(meta + L.slots);
                const VT* leafv = reinterpret_cast<const VT*>(smem_raw + L.leaf + (size_t)buf * L.leaf_bytes);
                // this thread's spanning-node piece of the tile, requested long before its first use
                int my_pslot = 0, my_pidx = 0;
                if (pc0 + gtid < pc1) { my_pslot = __ldg(P.piece_slot + pc0 + gtid); my_pidx = __ldg(P.piece_idx + pc0 + gtid); }
                const int b0 = g * R;
                for (int j = 0; j < nops; ++j) {
                    const int k = q * nops + j;
                    const VT* restv = reinterpret_cast<const VT*>(smem_raw + L.rest + (size_t)(k & 1) * L.rest_bytes) - (size_t)T * R;
                    const bool is_sum = (j == 0 ? first_op : OP_MAX) == OP_SUM;
                    VT* out = is_sum ? A.out_sum : A.out_max;
                    VT* part = is_sum ? A.part_sum : A.part_max;
                    VT* orow[R];
#pragma unroll
                    for (int r = 0; r < R; ++r) {
                        orow[r] = out + (size_t)min(b0 + r, n_rows - 1) * A.ld_out;
                        asm volatile("" : "+l"(orow[r]));  // keep the row pointers in registers (no rematerialisation per store)
                    }
                    GT_TRACE(8);
                    mbar_wait(full + (k & 1), (unsigned)(k >> 1) & 1u);  // the compute group has filled this rest buffer
                    GT_TRACE(9);
                    // emit the tile's node-id interval: lane = consecutive node id, so the slot reads of a warp cluster on
                    // a few neighbouring slots (unary chains broadcast) and every store instruction writes 128 contiguous
                    // bytes per row.  The sweep starts at the 128-byte line of row 0 that holds node n0, so with a row
                    // stride that is a multiple of 32 elements every store instruction covers exactly one line.
                    // Spanning nodes inside the interval carry the identity slot: what is written for them here is
                    // overwritten by span_kernel.
                    if (dbg != 3) {
                        constexpr int U = 4;
                        const int na = n0 & ~7;
                        const int lead = (int)(((reinterpret_cast<uintptr_t>(orow[0]) / sizeof(VT)) + (unsigned)n0) & 31u);
                        const unsigned count = (unsigned)(n1 - n0);
                        const uint16_t* sl_base = s_slots - na;
                        // a warp's U node groups are consecutive and its stores go row by row: U * 128 contiguous bytes
                        // per row and warp trip
                        const int nb0 = n0 - lead + (gtid >> 5) * (U * 32) + (gtid & 31);
                        for (int nb = nb0; nb < n1; nb += U * kEmitThreads) {
                            VT* p[R];
#pragma unroll
                            for (int r = 0; r < R; ++r) p[r] = orow[r] + nb;
                            RV x[U];
                            bool ok[U];
#pragma unroll
                            for (int u = 0; u < U; ++u) {
                                const int n = nb + u * 32;
                                ok[u] = (unsigned)(n - n0) < count;
                                if (ok[u]) {
                                    const int sl = sl_base[n];
                                    x[u] = RV::load((sl < T ? leafv : restv) + sl * R);
                                }
                            }
#pragma unroll
                            for (int r = 0; r < R; ++r)
#pragma unroll
                                for (int u = 0; u < U; ++u)
                                    if (ok[u]) __stcs(p[r] + u * 32, x[u].v[r]);
                        }
                        // pieces of spanning nodes that overlap this tile (reduced by span_kernel, which runs next on the stream)
                        for (int i = pc0 + gtid; i < pc1; i += kEmitThreads) {
                            const bool mine = i == pc0 + gtid;
                            const int sl = mine ? my_pslot : (int)__ldg(P.piece_slot + i);
                            const RV x = RV::load((sl < T ? leafv : restv) + sl * R);
                            const int idx = mine ? my_pidx : __ldg(P.piece_idx + i);
#pragma unroll
                            for (int r = 0; r < R; ++r) part[(size_t)min(b0 + r, n_rows - 1) * P.n_pieces + idx] = x.v[r];
                        }
                    }
                    GT_TRACE(10);
                    mbar_arrive(empty + (k & 1));  // this thread no longer reads the rest buffer
                }
                mbar_arrive(pairEmpty + buf);  // ... nor the pair's leaf block and metadata
            }
        }
    }

}

// ---- phase 3: nodes whose leaf range crosses tiles, reduced from their per-tile pieces (fp64 for sums) ------------
// One thread per (spanning node, row); consecutive lanes take consecutive spanning nodes of one row, whose pieces
// are adjacent in `part`.  Most spanning nodes have two or three pieces, which a thread loads all at once; the few
// with many (the root has one per tile) are reduced by the whole warp, 32 pieces per step, so that no thread walks a
// long chain of dependent loads.  Runs after mass_kernel in stream order and overwrites the placeholder it emitted.
// blockIdx.z selects the reduction when both were requested.
constexpr int kSpanInline = 8;  // pieces a thread reduces by itself

template <typename VT, bool SUM> __device__ __forceinline__ VT span_reduce(const VT* __restrict__ pr, int q0, int q1, int lane) {
    using AT = std::conditional_t<SUM, double, VT>;  // sums across tiles accumulate in fp64; max is exact
    const AT ident = SUM ? AT(0) : -std::numeric_limits<AT>::infinity();
    const int cnt = q1 - q0;
    AT acc = ident;
    if (cnt <= kSpanInline) {
        VT v[kSpanInline];
#pragma unroll
        for (int i = 0; i < kSpanInline; ++i) v[i] = i < cnt ? pr[q0 + i] : (VT)ident;  // independent loads
#pragma unroll
        for (int i = 0; i < kSpanInline; ++i) acc = SUM ? acc + (AT)v[i] : (AT)fmax((VT)acc, v[i]);
    }
    // nodes with many pieces, one at a time, by the whole warp (fixed order: results do not depend on the launch)
    unsigned heavy = __ballot_sync(0xffffffffu, cnt > kSpanInline);
    while (heavy) {
        const int src = __ffs(heavy) - 1;
        heavy &= heavy - 1;
        const int h0 = __shfl_sync(0xffffffffu, q0, src), h1 = __shfl_sync(0xffffffffu, q1, src);
        AT a = ident;
        for (int q = h0 + lane; q < h1; q += 32) a = SUM ? a + (AT)pr[q] : (AT)fmax((VT)a, pr[q]);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const AT y = __shfl_xor_sync(0xffffffffu, a, o);
            a = SUM ? a + y : (AT)fmax((VT)a, (VT)y);
        }
        if (lane == src) acc = a;
    }
    return cnt > 0 ? (VT)acc : VT(0);  // an empty range (root of an empty vocabulary) has no mass
}

template <typename VT>
__global__ void __launch_bounds__(256) span_kernel(PlanView P, MassArgs<VT> A) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31;
    const bool live = k < P.n_span;
    // plan metadata first: these loads may run ahead of the tile kernel's completion
    const int q0 = live ? __ldg(P.span_pp + k) : 0, q1 = live ? __ldg(P.span_pp + k + 1) : 0;
    const int node = live ? __ldg(P.span_node + k) : 0;
    pdl_wait();  // pieces and placeholders come from mass_kernel
    pdl_trigger();
    const bool is_sum = (A.ops & GT_OP_SUM) && blockIdx.z == 0;
    const VT* part = is_sum ? A.part_sum : A.part_max;
    VT* out = is_sum ? A.out_sum : A.out_max;
    for (int b = blockIdx.y; b < A.n_rows; b += gridDim.y) {  // whole warps stay together: dead lanes have no pieces
        const VT* pr = part + (size_t)b * P.n_pieces;
        const VT res = is_sum ? span_reduce<VT, true>(pr, q0, q1, lane) : span_reduce<VT, false>(pr, q0, q1, lane);
        if (live) out[(size_t)b * A.ld_out + node] = res;
    }
}

// ---- host side ---------------------------------------------------------------------------------------

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

template <typename VT, int R> static size_t mass_smem(const PlanView& v) { return MassSmem(v, (int)sizeof(VT) * R).total; }

// Opt in to > 48 KB dynamic shared memory once per (kernel, device, size): the attribute call is kept off the
// steady-state launch path (and out of CUDA graph captures).  Keyed by the kernel's address: instantiations
// with the same signature share a function type.
static cudaError_t allow_smem_impl(const void* kernel, size_t bytes) {
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
template <typename K> static cudaError_t allow_smem(K kernel, size_t bytes) {
    return allow_smem_impl(reinterpret_cast<const void*>(kernel), bytes);
}

// Scratch layout: a batch is reduced in *chunks* of at most kMaxChunkRows rows (what the staging buffer holds), and the
// pieces of spanning nodes are collected over a *span group* of up to kMaxSpanRows rows, so that span_kernel runs once
// per span group instead of once per chunk (it costs ~6 us in the chain for 2.5 us of work: it cannot become resident
// before the tile kernel's CTAs leave).
//   z [chunk row groups][ZG slots][R] VT | part_sum [span rows][n_pieces] VT | part_max likewise
constexpr int64_t kMaxChunkRows = 64;    // 34 MB of staging at 128k tokens: stays in the 126 MB L2 between permute and tile kernel
constexpr int64_t kMaxSpanRows = 1024;   // 9.9 MB of pieces per reduction at 128k tokens
template <typename VT, int R> struct Scratch {
    VT* z; VT* part_sum; VT* part_max;
    int64_t chunk_rows, span_rows;  // capacities
    static size_t pad(size_t b) { return (b + 255) & ~size_t(255); }
    static size_t z_bytes(const PlanView& v, int64_t rows) { return pad((size_t)((rows + R - 1) / R) * (size_t)v.ZG * R * sizeof(VT)); }
    static size_t part_bytes(const PlanView& v, int64_t rows) { return pad((size_t)rows * v.n_pieces * sizeof(VT)); }
    static size_t total(const PlanView& v, int64_t chunk, int64_t span) { return z_bytes(v, chunk) + 2 * part_bytes(v, span); }
    static int64_t max_chunk() {
        static const int64_t n = []() { const char* e = getenv("GT_CHUNK_ROWS"); const long x = e ? atol(e) : 0; return x > 0 ? (int64_t)x : kMaxChunkRows; }();
        return n;
    }
    // what a workspace of `bytes` holds (chunk_rows = 0: not even one row)
    Scratch(const PlanView& v, void* base, size_t bytes) {
        int64_t lo = 0, hi = max_chunk();
        while (lo < hi) {  // total() is monotone in the row count
            const int64_t mid = (lo + hi + 1) / 2;
            if (total(v, mid, mid) <= bytes) lo = mid; else hi = mid - 1;
        }
        chunk_rows = lo;
        lo = chunk_rows; hi = std::max<int64_t>(chunk_rows, kMaxSpanRows);
        while (lo < hi) {
            const int64_t mid = (lo + hi + 1) / 2;
            if (total(v, chunk_rows, mid) <= bytes) lo = mid; else hi = mid - 1;
        }
        span_rows = lo;
        char* p = static_cast<char*>(base);
        z = reinterpret_cast<VT*>(p);
        p += z_bytes(v, chunk_rows);
        part_sum = reinterpret_cast<VT*>(p);
        p += part_bytes(v, span_rows);
        part_max = reinterpret_cast<VT*>(p);
    }
};

// Resident CTAs per SM of a kernel at a given dynamic shared-memory size (cached: the query is not free).
static int resident_ctas(const void* kernel, int threads, size_t smem) {
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
static int sm_count() {
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

// One chunk: permute -> tile kernel.  part_sum / part_max: where this chunk's rows start in the span group's piece arrays.
template <typename VT, int R>
static int launch_mass(const PlanView& v, const void* ws, int in_type, int64_t ld_ws, unsigned flags, VT* z, VT* part_sum, VT* part_max,
                       VT* out_sum, VT* out_max, int64_t ld_out, int rows, unsigned ops, unsigned phases, cudaStream_t st) {
    MassArgs<VT> A;
    A.ws = ws; A.in_type = in_type; A.ld_ws = ld_ws;
    A.log_input = (flags & GT_FLAG_LOG_INPUT) ? 1 : 0; A.dfs_order = (flags & GT_FLAG_DFS_ORDER) ? 1 : 0;
    A.z = z;
    A.out_sum = out_sum; A.out_max = out_max; A.part_sum = part_sum; A.part_max = part_max;
    A.ld_out = ld_out; A.n_rows = rows; A.ops = ops;
    const int RG = (rows + R - 1) / R;
    if (phases & GT_FLAG_PHASE_PERMUTE) {  // one warp per unit of 128 (fp64 rows: 64) positions of a row group
        const int64_t UT = in_type == GT_F64 ? kUnitTokens / 2 : kUnitTokens;
        const int64_t units = (int64_t)RG * ((v.V + UT - 1) / UT);
        const int64_t pgrid = (units + kPermThreads / 32 - 1) / (kPermThreads / 32);
        NvtxRange nv("gt:permute");
        GT_CUDA(launch_pdl(permute_kernel<VT, R>, dim3((unsigned)pgrid), dim3(kPermThreads), 0, st, v, A, (unsigned)units));
    }
    if (phases & GT_FLAG_PHASE_TILE) {
        const size_t smem = mass_smem<VT, R>(v);
        if (smem > 227 * 1024) {
            set_error("tile plan needs %zu bytes of shared memory per CTA (limit 232448): use a smaller tile", smem);
            return GT_ERR_LIMIT;
        }
        GT_CUDA(allow_smem(mass_kernel<VT, R>, smem));
        // persistent grid: one CTA per resident slot; CTA b takes the (row group, tile) pairs b, b + grid, ...
        const int64_t pairs = (int64_t)v.NT * RG;
        const int slots = sm_count() * resident_ctas(reinterpret_cast<const void*>(mass_kernel<VT, R>), kThreads, smem);
        const unsigned grid = (unsigned)std::min<int64_t>(pairs, slots);
        NvtxRange nv("gt:tile");
        GT_CUDA(launch_pdl(mass_kernel<VT, R>, dim3(grid), dim3(kThreads), smem, st, v, A));
    }
    return GT_OK;
}

// The spanning nodes of the `rows` rows whose pieces start at part_sum / part_max and whose outputs start at out_sum / out_max.
template <typename VT>
static int launch_span(const PlanView& v, VT* part_sum, VT* part_max, VT* out_sum, VT* out_max, int64_t ld_out, int rows, unsigned ops,
                       cudaStream_t st) {
    if (v.n_span <= 0 || rows <= 0) return GT_OK;
    MassArgs<VT> A{};
    A.out_sum = out_sum; A.out_max = out_max; A.part_sum = part_sum; A.part_max = part_max;
    A.ld_out = ld_out; A.n_rows = rows; A.ops = ops;
    const int nops = (ops == (unsigned)(GT_OP_SUM | GT_OP_MAX)) ? 2 : 1;
    dim3 sgrid((unsigned)((v.n_span + 255) / 256), (unsigned)std::min(rows, 4096), (unsigned)nops);
    NvtxRange nv("gt:span");
    GT_CUDA(launch_pdl(span_kernel<VT>, sgrid, dim3(256), 0, st, v, A));
    return GT_OK;
}

template <typename VT, int R>
static int reduce_typed(const PlanView& v, const void* ws, int in_type, int64_t n_rows, int64_t ld_ws, void* out_sum,
                        void* out_max, int64_t ld_out, unsigned ops, unsigned flags, void* workspace,
                        size_t workspace_bytes, cudaStream_t st) {
    if (in_type != GT_F32 && in_type != GT_F64 && in_type != GT_F16 && in_type != GT_BF16) {
        set_error("unknown input type %d", in_type);
        return GT_ERR_ARG;
    }
    VT* osum = (ops & GT_OP_SUM) ? static_cast<VT*>(out_sum) : nullptr;
    VT* omax = (ops & GT_OP_MAX) ? static_cast<VT*>(out_max) : nullptr;
    if (v.NT == 0) {  // empty vocabulary: the root is the only node and has no mass
        for (VT* out : {osum, omax})
            if (out) GT_CUDA(cudaMemset2DAsync(out, (size_t)ld_out * sizeof(VT), 0, (size_t)v.N * sizeof(VT), (size_t)n_rows, st));
        return GT_OK;
    }
    // rows per launch: what the caller's scratch can stage (a partial row group is legal: the kernels alias the missing
    // rows to the last valid one)
    const Scratch<VT, R> sc(v, workspace, workspace_bytes);
    if (sc.chunk_rows < 1) {
        set_error("workspace too small: %zu bytes given, one row needs %zu", workspace_bytes, Scratch<VT, R>::total(v, 1, 1));
        return GT_ERR_STATE;
    }
    const unsigned phases = (flags & GT_FLAG_PHASE_MASK) ? (flags & GT_FLAG_PHASE_MASK) : GT_FLAG_PHASE_MASK;
    const size_t in_size = in_type == GT_F64 ? 8 : in_type == GT_F32 ? 4 : 2;
    const int64_t chunk_rows = sc.chunk_rows;
    for (int64_t s0 = 0; s0 < n_rows; s0 += sc.span_rows) {  // span groups
        const int64_t s1 = std::min<int64_t>(n_rows, s0 + sc.span_rows);
        for (int64_t r0 = s0; r0 < s1; r0 += chunk_rows) {  // chunks
            const int rows = (int)std::min<int64_t>(chunk_rows, s1 - r0);
            const void* wsr = static_cast<const char*>(ws) + (size_t)r0 * ld_ws * in_size;
            const size_t poff = (size_t)(r0 - s0) * v.n_pieces;
            const int rc = launch_mass<VT, R>(v, wsr, in_type, ld_ws, flags, sc.z, sc.part_sum + poff, sc.part_max + poff,
                                              osum ? osum + (size_t)r0 * ld_out : nullptr, omax ? omax + (size_t)r0 * ld_out : nullptr,
                                              ld_out, rows, ops, phases, st);
            if (rc != GT_OK) return rc;
        }
        if (phases & GT_FLAG_PHASE_SPAN) {
            const int rc = launch_span<VT>(v, sc.part_sum, sc.part_max, osum ? osum + (size_t)s0 * ld_out : nullptr,
                                           omax ? omax + (size_t)s0 * ld_out : nullptr, ld_out, (int)(s1 - s0), ops, st);
            if (rc != GT_OK) return rc;
        }
    }
    return GT_OK;
}

// ---- read-outs that keep the [B, N] slab on the GPU (SURVEY 8f-2, 8f-4) ---------------------------------------
//
// gather: the caller of the mass path reads a handful of nodes per row (the children of the node a particle stands
// on), so only out[b, k] = mass[b, ids[b, k]] has to cross PCIe.  One thread per (row, k); rows on blockIdx.y.
template <typename VT>
__global__ void __launch_bounds__(256) gather_nodes_kernel(const VT* __restrict__ mass, int64_t ld_mass, int n_rows, int64_t N,
                                                           const int32_t* __restrict__ ids, int n_ids, int64_t ids_ld,
                                                           const int32_t* __restrict__ norm, int log_out,
                                                           VT* __restrict__ out, int64_t ld_out) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_ids) return;
    for (int b = blockIdx.y; b < n_rows; b += gridDim.y) {
        const VT* row = mass + (size_t)b * ld_mass;
        const int id = __ldg(ids + (size_t)b * ids_ld + k);
        VT v = (id >= 0 && id < N) ? row[id] : VT(0);
        if (norm) {
            const int z = __ldg(norm + b);
            const VT d = (z >= 0 && z < N) ? row[z] : VT(0);
            v = log_out ? (VT)(log((double)v) - log((double)d)) : v / d;
        } else if (log_out) {
            v = (VT)log((double)v);
        }
        out[(size_t)b * ld_out + k] = v;
    }
}

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

// ---- token masks under a byte DFA (gt_dfa_token_mask / gt_dfa_advance) ------------------------------------------------
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

__global__ void __launch_bounds__(kDfaThreads) dfa_mask_kernel(PlanView P, DfaArgs A, uint32_t* __restrict__ bits, int64_t ld_bits,
                                                               int64_t words) {
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
            if (st[g] >= 0 && k >= dk[g]) st[g] = dfa_step(A, st[g], s);
            any |= st[g] >= 0;
        }
        if (!any) break;
    }
    const int64_t w = i >> 5;
    const int rows = min(kDfaRows, A.n_rows - b0);
#pragma unroll
    for (int g = 0; g < kDfaRows; ++g) {
        if (g >= rows) break;
        const unsigned word = __ballot_sync(0xffffffffu, st[g] >= 0);
        if ((threadIdx.x & 31) == 0 && w < words) bits[(size_t)(b0 + g) * ld_bits + w] = word;
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

// The plan metadata resident on the current device, for the launches of one call.
static int resident_plan(const gt_trie* t, const PlanView*& v) {
    int device = -1;
    GT_CUDA(cudaGetDevice(&device));
    auto it = t->dev.find(device);
    if (it == t->dev.end()) { set_error("trie metadata is not resident on device %d (call gt_upload)", device); return GT_ERR_STATE; }
    v = &it->second->view;
    return GT_OK;
}

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
    const size_t in_size = A.in_type == GT_F64 ? 8 : A.in_type == GT_F32 ? 4 : 2;
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

int gt_get_plan_info(const gt_trie* t, gt_plan_info* info) {
    if (!t || !info) { gt::set_error("gt_get_plan_info: bad argument"); return GT_ERR_ARG; }
    if (!t->plan) { gt::set_error("gt_get_plan_info: trie has no plan yet (call gt_upload)"); return GT_ERR_STATE; }
    const gt::Plan& P = *t->plan;
    memset(info, 0, sizeof *info);
    info->n_tokens = t->layout.V; info->n_nodes = t->layout.N;
    info->tile_leaves = P.T; info->n_tiles = P.NT;
    info->rows_per_item = P.R; info->permute_unit = gt::kUnitTokens;
    info->n_span = (int32_t)P.span_node.size(); info->span_terms = (int64_t)P.n_pieces;
    info->max_levels = P.max_levels; info->max_tile_values = P.max_tile_values;
    info->staged_slots = (int64_t)P.NT * P.T;
    size_t meta = 0;
    for (auto& kv : t->dev) { meta = kv.second->blob_bytes; break; }
    info->meta_bytes = (int64_t)meta;
    return GT_OK;
}

int64_t gt_debug_read_trace(const gt_trie* t, int device, long long* dst, int64_t capacity, int32_t dims[3]) {
    if (!t) { gt::set_error("gt_debug_read_trace: null trie"); return -1; }
    auto it = t->dev.find(device);
    if (it == t->dev.end() || !it->second->trace) { gt::set_error("no trace buffer on device %d (set GT_TRACE=1 before gt_upload)", device); return -1; }
    const int64_t n = (int64_t)gt::kTraceCtas * gt::kTraceItems * gt::kTraceEvents;
    if (dims) { dims[0] = gt::kTraceCtas; dims[1] = gt::kTraceItems; dims[2] = gt::kTraceEvents; }
    if (dst && capacity > 0) {
        int cur = 0;
        cudaGetDevice(&cur);
        cudaSetDevice(device);
        cudaDeviceSynchronize();
        const cudaError_t e = cudaMemcpy(dst, it->second->trace, (size_t)std::min(n, capacity) * sizeof(long long), cudaMemcpyDeviceToHost);
        cudaMemset(it->second->trace, 0, (size_t)n * sizeof(long long));
        cudaSetDevice(cur);
        if (e != cudaSuccess) { gt::set_error("trace copy failed: %s", cudaGetErrorString(e)); return -1; }
    }
    return n;
}

size_t gt_workspace_bytes(const gt_trie* t, int64_t max_rows) {
    if (!t || !t->plan || max_rows <= 0) return 0;
    gt::PlanView v{};
    v.ZG = (int64_t)t->plan->NT * t->plan->T; v.n_pieces = t->plan->n_pieces;
    // staging for one chunk + the pieces of one span group, sized for the fp64 pipeline (the fp32 one needs half)
    return gt::Scratch<double, 2>::total(v, std::min<int64_t>(max_rows, gt::Scratch<double, 2>::max_chunk()),
                                         std::min<int64_t>(max_rows, gt::kMaxSpanRows)) + 256;
}

static bool ops_ok(unsigned ops) { return (ops & (GT_OP_SUM | GT_OP_MAX)) && !(ops & ~(unsigned)(GT_OP_SUM | GT_OP_MAX)); }

int gt_weight_reduce(const gt_trie* t, const void* ws, int in_type, int64_t n_rows, int64_t ld_ws, void* out_sum,
                     void* out_max, int out_type, int64_t ld_out, unsigned ops, unsigned flags, void* workspace,
                     size_t workspace_bytes, gt_stream stream) {
    if (!t) { gt::set_error("gt_weight_reduce: null trie"); return GT_ERR_ARG; }
    if (n_rows < 0 || !ops_ok(ops)) {
        gt::set_error("gt_weight_reduce: bad n_rows / ops"); return GT_ERR_ARG;
    }
    if (n_rows == 0) return GT_OK;
    if ((t->layout.V > 0 && !ws) || ((ops & GT_OP_SUM) && !out_sum) || ((ops & GT_OP_MAX) && !out_max)) {
        gt::set_error("gt_weight_reduce: null data pointer"); return GT_ERR_ARG;
    }
    if (ld_out > ((int64_t)1 << 28)) {  // the kernels index a row group with 32-bit offsets
        gt::set_error("gt_weight_reduce: output row stride %lld exceeds 2^28 elements", (long long)ld_out);
        return GT_ERR_LIMIT;
    }
    if (ld_ws < t->layout.V || ld_out < t->layout.N) {
        gt::set_error("gt_weight_reduce: row stride smaller than row length (ld_ws=%lld V=%lld ld_out=%lld N=%lld)",
                      (long long)ld_ws, (long long)t->layout.V, (long long)ld_out, (long long)t->layout.N);
        return GT_ERR_ARG;
    }
    const gt::PlanView* v = nullptr;
    if (const int rc = gt::resident_plan(t, v); rc != GT_OK) return rc;
    if (!workspace || (reinterpret_cast<uintptr_t>(workspace) & 255)) { gt::set_error("gt_weight_reduce: workspace must be a 256-byte aligned device pointer"); return GT_ERR_ARG; }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    gt::NvtxRange nv("gt:weight_reduce");
#define GT_REDUCE(VT, R) gt::reduce_typed<VT, R>(*v, ws, in_type, n_rows, ld_ws, out_sum, out_max, ld_out, ops, flags, \
                                                workspace, workspace_bytes, st)
    // 16-byte value slots: four fp32 rows or two fp64 rows per work item
    if (out_type == GT_F32) return GT_REDUCE(float, 4);
    if (out_type == GT_F64) return GT_REDUCE(double, 2);
#undef GT_REDUCE
    gt::set_error("gt_weight_reduce: output type must be GT_F32 or GT_F64");
    return GT_ERR_ARG;
}

int gt_download_rows(void* dst_host, size_t dst_pitch, const void* src_dev, size_t src_pitch, size_t width_bytes, int64_t n_rows,
                     gt_stream stream) {
    if (n_rows < 0 || dst_pitch < width_bytes || src_pitch < width_bytes) { gt::set_error("gt_download_rows: bad size / pitch"); return GT_ERR_ARG; }
    if (n_rows == 0 || width_bytes == 0) return GT_OK;
    if (!dst_host || !src_dev) { gt::set_error("gt_download_rows: null pointer"); return GT_ERR_ARG; }
    GT_CUDA(cudaMemcpy2DAsync(dst_host, dst_pitch, src_dev, src_pitch, width_bytes, (size_t)n_rows, cudaMemcpyDeviceToHost,
                              static_cast<cudaStream_t>(stream)));
    return GT_OK;
}

int gt_gather_nodes(const void* mass, int type, int64_t n_rows, int64_t n_nodes, int64_t ld_mass, const int32_t* node_ids,
                    int64_t n_ids, int64_t ids_ld, const int32_t* norm_node, unsigned flags, void* out, int64_t ld_out,
                    gt_stream stream) {
    if (n_rows < 0 || n_ids < 0 || n_nodes < 0 || ld_mass < n_nodes || ld_out < n_ids || ids_ld < 0 || (flags & ~(unsigned)GT_GATHER_LOG)) {
        gt::set_error("gt_gather_nodes: bad size / stride / flags"); return GT_ERR_ARG;
    }
    if (n_rows == 0 || n_ids == 0) return GT_OK;
    if (!mass || !node_ids || !out) { gt::set_error("gt_gather_nodes: null data pointer"); return GT_ERR_ARG; }
    if (n_rows > INT32_MAX || n_ids > INT32_MAX) { gt::set_error("gt_gather_nodes: too many rows / ids"); return GT_ERR_LIMIT; }
    if (type != GT_F32 && type != GT_F64) { gt::set_error("gt_gather_nodes: type must be GT_F32 or GT_F64"); return GT_ERR_ARG; }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    dim3 grid((unsigned)((n_ids + 255) / 256), (unsigned)std::min<int64_t>(n_rows, 32768));
    const int lg = (flags & GT_GATHER_LOG) ? 1 : 0;
    if (type == GT_F32)
        gt::gather_nodes_kernel<float><<<grid, 256, 0, st>>>(static_cast<const float*>(mass), ld_mass, (int)n_rows, n_nodes, node_ids,
                                                            (int)n_ids, ids_ld, norm_node, lg, static_cast<float*>(out), ld_out);
    else
        gt::gather_nodes_kernel<double><<<grid, 256, 0, st>>>(static_cast<const double*>(mass), ld_mass, (int)n_rows, n_nodes, node_ids,
                                                             (int)n_ids, ids_ld, norm_node, lg, static_cast<double*>(out), ld_out);
    GT_CUDA(cudaGetLastError());
    return GT_OK;
}

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

size_t gt_child_workspace_bytes(const gt_trie* t, int64_t max_rows) {
    if (!t || max_rows <= 0) return 0;
    return gt::ChildScratch::total(std::min<int64_t>(max_rows, gt::kMaxChildRows), gt::ChildScratch::slots(t->layout)) + 256;
}

static bool child_in_type_ok(int in_type) { return in_type == GT_F32 || in_type == GT_F64 || in_type == GT_F16 || in_type == GT_BF16; }

// Checks shared by the next-symbol read-outs.  Each of the four calls and its *_masked twin share one implementation
// (the unmasked call passes no mask), which makes its checks in one order: the scalars and strides
// (child_check_scalars, then its own), the early return for no rows, the data pointers (its own outputs, then
// child_check_pointers) and last the workspace, so that a call without rows accepts null pointers.
// child_check_scalars fills the input half of A.
static int child_check_scalars(const gt_trie* t, const void* ws, int in_type, int64_t n_rows, int64_t ld_ws,
                               const int32_t* nodes, const uint32_t* mask, int64_t mask_ld, unsigned flags, unsigned known,
                               const char* what, gt::ChildArgs& A) {
    if (!t) { gt::set_error("%s: null trie", what); return GT_ERR_ARG; }
    if (n_rows < 0 || (flags & ~known) || !child_in_type_ok(in_type)) {
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
    if (!ops_ok(ops) || ld_out < D) {
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
    if (!ops_ok(ops) || ld_out < S + 1) {
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
    gt::dfa_mask_kernel<<<grid, gt::kDfaThreads, 0, static_cast<cudaStream_t>(stream)>>>(*v, A, mask_bits, mask_ld, words);
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
