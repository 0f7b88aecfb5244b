// Particle resampling for sm_100a: per group of P particles, the effective sample size and, when it falls below a
// threshold, multinomial, stratified or systematic ancestors (gt_resample).
//
// One CTA per group, everything in shared memory: the group's fp32 log-weights (read once, before anything is written,
// so logw_out may be logw) and its fp64 CDF.  The CDF is scanned in R = ceil(P / r) runs of r = ceil(sqrt(P)) particles:
// thread k scans run k sequentially from 0, one thread chains the run bases B_{k+1} = B_k + L_k, and c_i = B_k + local_i.
// The last value of run k and the base of run k + 1 are then the same fp64 expression, so the CDF is non-decreasing and
// exactly flat across every zero weight, run boundaries included: a dead particle is never picked.  (A tree scan of the
// run totals rounds the bases differently from B_k + L_k.)  The critical path is r + R ~ 2 sqrt(P) dependent adds.
// Each run occupies r + 1 slots, so the run-wise scans of 32 lanes fall into distinct shared-memory banks.
#include <cmath>
#include <cstdint>

#include "trie_device.cuh"
#include "philox.cuh"

namespace gt {

constexpr int kRThreads = 512;  // largest block: 32 particles per thread at P = GT_RESAMPLE_MAX_GROUP
constexpr int kRMaxRuns = 128;  // ceil(sqrt(GT_RESAMPLE_MAX_GROUP))
static_assert(kRMaxRuns * kRMaxRuns >= GT_RESAMPLE_MAX_GROUP, "runs of the CDF scan");
constexpr uint32_t kResampleStream = 1u;  // third Philox counter word: the samplers use 0

struct ResampleArgs {
    const float* logw; int P; int method; double thr_P;  // thr_P = ess_threshold * P
    int r, R;                                             // run length and run count of the CDF scan
    uint64_t seed, offset;
    int32_t* anc; float* logw_out; float* ess; float* log_mean_w; uint8_t* resampled;
};

// Block sum in a fixed order: an xor-shuffle tree per warp (every lane gets the same value), then the warp totals in
// warp order.  Every thread returns the result.
__device__ __forceinline__ double block_sum(double x, double* s_red) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
    if (lane == 0) s_red[warp] = x;
    __syncthreads();
    double t = 0.0;
    for (int w = 0; w < nw; ++w) t += s_red[w];
    __syncthreads();
    return t;
}

__device__ __forceinline__ float block_max(float x, float* s_red) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x = fmaxf(x, __shfl_xor_sync(0xffffffffu, x, o));
    if (lane == 0) s_red[warp] = x;
    __syncthreads();
    float t = -INFINITY;
    for (int w = 0; w < nw; ++w) t = fmaxf(t, s_red[w]);
    __syncthreads();
    return t;
}

__device__ __forceinline__ int block_max_int(int x, int* s_red) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    x = __reduce_max_sync(0xffffffffu, x);
    if (lane == 0) s_red[warp] = x;
    __syncthreads();
    int t = -1;
    for (int w = 0; w < nw; ++w) t = max(t, s_red[w]);
    __syncthreads();
    return t;
}

__global__ void __launch_bounds__(kRThreads) resample_kernel(ResampleArgs A) {
    extern __shared__ double s_dyn[];
    double* s_c = s_dyn;                                   // [R][r + 1]: run k's CDF values at k * (r + 1) + [0, r)
    float* s_lw = reinterpret_cast<float*>(s_c + (size_t)A.R * (A.r + 1));  // [P]
    __shared__ double s_base[kRMaxRuns + 1];               // s_base[k] = B_k, the CDF before run k; s_base[R] = S
    __shared__ double s_dred[kRThreads / 32];
    __shared__ float s_fred[kRThreads / 32];
    __shared__ int s_ired[kRThreads / 32];

    const int P = A.P, r = A.r, R = A.R, tid = threadIdx.x, T = blockDim.x;
    const int64_t g0 = (int64_t)blockIdx.x * P;  // first particle of the group

    float m = -INFINITY;
    bool has_nan = false, has_pinf = false;
    for (int j = tid; j < P; j += T) {
        const float x = A.logw[g0 + j];
        s_lw[j] = x;
        m = fmaxf(m, x);  // NaN-blind: the NaN flag decides
        has_nan |= x != x;
        has_pinf |= x == INFINITY;
    }
    has_nan = __syncthreads_or(has_nan);
    has_pinf = __syncthreads_or(has_pinf);
    const float M = block_max(m, s_fred);

    bool resample = false;
    float log_mean_w = 0.f;
    if (has_nan || has_pinf || M == -INFINITY) {  // no resampling: ess NaN / NaN / 0, log mean weight NaN / +inf / -inf
        if (tid == 0) {
            A.ess[blockIdx.x] = has_nan || has_pinf ? NAN : 0.f;
            A.log_mean_w[blockIdx.x] = has_nan ? NAN : has_pinf ? INFINITY : -INFINITY;
            A.resampled[blockIdx.x] = 0;
        }
    } else {
        const double md = (double)M;
        double q = 0.0;
        int last = -1;  // this thread's last particle with w > 0
        for (int j = tid; j < P; j += T) {
            const double w = exp((double)s_lw[j] - md);
            s_c[j + j / r] = w;
            q = fma(w, w, q);
            if (w > 0.0) last = j;
        }
        const double Q = block_sum(q, s_dred);
        const int last_live = block_max_int(last, s_ired);  // the syncs inside also publish s_c
        if (tid < R) {  // run tid, scanned from 0
            double* c = s_c + tid * (r + 1);
            const int len = min(r, P - tid * r);
            double acc = 0.0;
            for (int i = 0; i < len; ++i) {
                acc += c[i];
                c[i] = acc;
            }
            s_base[tid + 1] = acc;
        }
        __syncthreads();
        if (tid == 0) {
            double b = 0.0;
            s_base[0] = 0.0;
            for (int k = 1; k <= R; ++k) s_base[k] = b = b + s_base[k];
        }
        __syncthreads();
        for (int j = tid; j < P; j += T) {
            const int k = j / r;
            s_c[j + k] = s_base[k] + s_c[j + k];
        }
        __syncthreads();
        const double S = s_base[R];
        const double ess = S * S / Q;
        resample = ess < A.thr_P;
        log_mean_w = (float)(md + log(S) - log((double)P));
        if (tid == 0) {
            A.ess[blockIdx.x] = (float)ess;
            A.log_mean_w[blockIdx.x] = log_mean_w;
            A.resampled[blockIdx.x] = resample;
        }
        if (resample) {
            const double u_group = A.method == GT_RESAMPLE_SYSTEMATIC
                                       ? philox_uniform53(A.seed, A.offset + (uint64_t)g0, kResampleStream) : 0.0;
            for (int j = tid; j < P; j += T) {
                const int64_t b = g0 + j;
                double t;
                if (A.method == GT_RESAMPLE_MULTINOMIAL) {
                    t = philox_uniform53(A.seed, A.offset + (uint64_t)b, kResampleStream) * S;
                } else {
                    const double u = A.method == GT_RESAMPLE_STRATIFIED
                                         ? philox_uniform53(A.seed, A.offset + (uint64_t)b, kResampleStream) : u_group;
                    t = ((double)j + u) / (double)P * S;
                }
                // first run whose last value (= the next base) exceeds t, then the first value inside it that does
                int lo = 0, hi = R;
                while (lo < hi) {
                    const int mid = (lo + hi) >> 1;
                    if (s_base[mid + 1] > t) hi = mid; else lo = mid + 1;
                }
                int i = last_live;  // no value exceeds t: the last live particle
                if (lo < R) {
                    const double* c = s_c + lo * (r + 1);
                    int a = 0, e = min(r, P - lo * r) - 1;  // c[e] = s_base[lo + 1] > t
                    while (a < e) {
                        const int mid = (a + e) >> 1;
                        if (c[mid] > t) e = mid; else a = mid + 1;
                    }
                    i = lo * r + a;
                }
                A.anc[b] = (int32_t)(g0 + i);
                A.logw_out[b] = log_mean_w;
            }
            return;
        }
    }
    for (int j = tid; j < P; j += T) {
        A.anc[g0 + j] = (int32_t)(g0 + j);
        A.logw_out[g0 + j] = s_lw[j];
    }
}

}  // namespace gt

extern "C" int gt_resample(const float* logw, int64_t n_groups, int64_t group_size, int method, float ess_threshold,
                           uint64_t seed, uint64_t offset, int32_t* ancestors, float* logw_out, float* ess_out,
                           float* log_mean_w_out, uint8_t* resampled_out, gt_stream stream) {
    if (n_groups < 0 || group_size < 1) { gt::set_error("gt_resample: bad n_groups or group_size"); return GT_ERR_ARG; }
    if (method < GT_RESAMPLE_MULTINOMIAL || method > GT_RESAMPLE_SYSTEMATIC) {
        gt::set_error("gt_resample: unknown method %d", method); return GT_ERR_ARG;
    }
    if (ess_threshold != ess_threshold) { gt::set_error("gt_resample: NaN ess_threshold"); return GT_ERR_ARG; }
    if (group_size > GT_RESAMPLE_MAX_GROUP) { gt::set_error("gt_resample: group_size above %d", GT_RESAMPLE_MAX_GROUP); return GT_ERR_LIMIT; }
    if (n_groups > INT32_MAX / group_size) { gt::set_error("gt_resample: more than 2^31 - 1 particles"); return GT_ERR_LIMIT; }
    if (n_groups == 0) return GT_OK;
    if (!logw || !ancestors || !logw_out || !ess_out || !log_mean_w_out || !resampled_out) {
        gt::set_error("gt_resample: null pointer"); return GT_ERR_ARG;
    }
    gt::ResampleArgs A;
    A.logw = logw; A.P = (int)group_size; A.method = method; A.thr_P = (double)ess_threshold * (double)group_size;
    A.r = (int)std::ceil(std::sqrt((double)group_size));
    A.R = (A.P + A.r - 1) / A.r;
    A.seed = seed; A.offset = offset;
    A.anc = ancestors; A.logw_out = logw_out; A.ess = ess_out; A.log_mean_w = log_mean_w_out; A.resampled = resampled_out;
    const int threads = A.P >= gt::kRThreads ? gt::kRThreads : (A.P + 31) / 32 * 32;
    const size_t smem = sizeof(double) * (size_t)A.R * (A.r + 1) + sizeof(float) * (size_t)A.P;
    gt::NvtxRange nv("gt:resample");
    if (smem > 48 * 1024) GT_CUDA(gt::allow_smem(gt::resample_kernel, smem));
    gt::resample_kernel<<<(unsigned)n_groups, threads, smem, static_cast<cudaStream_t>(stream)>>>(A);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { gt::set_error("resample launch failed: %s", cudaGetErrorString(e)); return GT_ERR_CUDA; }
    return GT_OK;
}
