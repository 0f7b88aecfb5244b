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
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <type_traits>
#include <algorithm>

#include "trie_device.cuh"

namespace gt {

constexpr int OP_SUM = 1, OP_MAX = 2;

// ---- small device helpers -----------------------------------------------------------------------

template <int OP, typename VT> __device__ __forceinline__ VT op_apply(VT a, VT b) {
    if constexpr (OP == OP_SUM) return a + b;
    else return fmax(a, b);  // fmaxf/fmax overloads; NaN operands are ignored like numba's max()
}
template <int OP, typename VT> __device__ __forceinline__ VT op_ident() {
    if constexpr (OP == OP_SUM) return VT(0);
    else return -std::numeric_limits<VT>::infinity();
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

// one SM-clock stamp of the profiling trace (layout: kTraceCtas / kTraceItems / kTraceEvents, trie_device.cuh)
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

template <typename VT, int R> static size_t mass_smem(const PlanView& v) { return MassSmem(v, (int)sizeof(VT) * R).total; }

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
    const size_t in_size = in_type_size(in_type);
    if (!in_size) {
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

}  // namespace gt

extern "C" {

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

int gt_weight_reduce(const gt_trie* t, const void* ws, int in_type, int64_t n_rows, int64_t ld_ws, void* out_sum,
                     void* out_max, int out_type, int64_t ld_out, unsigned ops, unsigned flags, void* workspace,
                     size_t workspace_bytes, gt_stream stream) {
    if (!t) { gt::set_error("gt_weight_reduce: null trie"); return GT_ERR_ARG; }
    if (n_rows < 0 || !gt::ops_ok(ops)) {
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

}  // extern "C"
