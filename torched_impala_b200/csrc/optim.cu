// Per-group gradient clipping + Adam + step counter in ONE launch
// (reference learner.py:176-183: two clip_grad_norm_ calls, Adam.step, LambdaLR.step).
//
// The parameter vector is tiny (14 144 floats at H=256, 69 312 at H=512) but the two clip
// norms need every gradient entry before any parameter can move.  One thread-block
// cluster of 8 CTAs (8 x 1024 threads, co-scheduled by hardware) does both phases in a
// single launch: each CTA reduces the squares of its slice in float64, the 8 partial pairs
// are exchanged through distributed shared memory, one cluster barrier later every CTA
// holds the same two norms and applies Adam to its slice.  The gradient arrives as float64
// (sum of per-CTA float32 partials, possibly all-reduced over ranks) and the norms are reduced
// in float64; optimizer state stays float32 in HBM and the per-element update runs in float32.
#include <cooperative_groups.h>
#include <math.h>

#include "common.cuh"

namespace cg = cooperative_groups;

namespace {

constexpr int kAdamThreads = 1024;
constexpr int kAdamCluster = 8;

// state[0] = step count (int64), state[1] / state[2] = beta1^t / beta2^t as float64 bit patterns
// (all-zero state = fresh optimizer): running powers replace two float64 pow() calls per step.
__global__ void __cluster_dims__(kAdamCluster, 1, 1) __launch_bounds__(kAdamThreads)
clip_adam_kernel(float* __restrict__ params, const double* __restrict__ grad, float* __restrict__ m,
                 float* __restrict__ v, int64_t* __restrict__ state, int64_t n_policy,
                 int64_t n_total, float max_norm, float lr, float beta1, float beta2, float eps,
                 double* __restrict__ norms_out) {
    cg::cluster_group cluster = cg::this_cluster();
    __shared__ double s_warp[2][kAdamThreads / 32];
    __shared__ double s_cta[2];   // this CTA's partial sums of squares (read by the peers)
    __shared__ float s_coef[2];
    __shared__ float s_bias[2];   // step_size = lr / (1 - beta1^t), 1 / sqrt(1 - beta2^t)
    __shared__ double s_pow[2];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t first = (int64_t)cluster.block_rank() * kAdamThreads + tid;
    const int64_t stride = (int64_t)kAdamCluster * kAdamThreads;

    // phase 1: this thread's gradient entries (kept in registers when there are at most two, the
    // benchmark sizes) and the float32 state they will update - all loads issued up front
    constexpr int kKeep = 2;
    double gk[kKeep];
    float pk[kKeep], mk[kKeep], vk[kKeep];
    double ss0 = 0.0, ss1 = 0.0;
#pragma unroll
    for (int k = 0; k < kKeep; ++k) {
        const int64_t i = first + k * stride;
        pk[k] = i < n_total ? params[i] : 0.f;
        mk[k] = i < n_total ? m[i] : 0.f;
        vk[k] = i < n_total ? v[i] : 0.f;
    }
#pragma unroll
    for (int k = 0; k < kKeep; ++k) {
        const int64_t i = first + k * stride;
        gk[k] = i < n_total ? grad[i] : 0.0;
    }
#pragma unroll
    for (int k = 0; k < kKeep; ++k) {
        const int64_t i = first + k * stride;
        if (i < n_policy) ss0 += gk[k] * gk[k];
        else ss1 += gk[k] * gk[k];
    }
    for (int64_t i = first + kKeep * stride; i < n_total; i += stride) {
        const double g = grad[i];
        if (i < n_policy) ss0 += g * g;
        else ss1 += g * g;
    }
    ss0 = warp_sum_f64(ss0);
    ss1 = warp_sum_f64(ss1);
    if (lane == 0) s_warp[0][warp] = ss0, s_warp[1][warp] = ss1;
    if (tid == 64) {  // bias corrections from the running powers (nobody writes state before the end)
        const double p1 = state[0] == 0 ? 1.0 : __longlong_as_double(state[1]);
        const double p2 = state[0] == 0 ? 1.0 : __longlong_as_double(state[2]);
        s_pow[0] = p1 * (double)beta1, s_pow[1] = p2 * (double)beta2;
        s_bias[0] = (float)((double)lr / (1.0 - s_pow[0]));
        s_bias[1] = (float)(1.0 / sqrt(1.0 - s_pow[1]));
    }
    __syncthreads();
    if (tid < 2) {
        double s = 0.0;
        for (int i = 0; i < kAdamThreads / 32; ++i) s += s_warp[tid][i];
        s_cta[tid] = s;
    }
    cluster.sync();  // all 8 partial pairs are in place
    if (tid < 2) {
        double s = 0.0;
        for (int r = 0; r < kAdamCluster; ++r) s += *cluster.map_shared_rank(&s_cta[tid], r);
        const double norm = sqrt(s);
        // torch.nn.utils.clip_grad_norm_: coef = max_norm / (norm + 1e-6), clamped to 1
        s_coef[tid] = (float)fmin(1.0, (double)max_norm / (norm + 1e-6));
        if (norms_out && cluster.block_rank() == 0) norms_out[tid] = norm;
    }
    __syncthreads();
    // phase 2: Adam in float32 arithmetic (the state is float32; one step's rounding is ~1e-7)
    const float b1 = beta1, b2 = beta2, step_size = s_bias[0], inv_bc2_sqrt = s_bias[1];
    const float c0 = s_coef[0], c1 = s_coef[1];
    auto update = [&](int64_t i, float g, float p, float mi, float vi) {
        g *= (i < n_policy ? c0 : c1);
        mi = fmaf(b1, mi, (1.f - b1) * g);
        vi = fmaf(b2, vi, (1.f - b2) * g * g);
        const float denom = fmaf(sqrtf(vi), inv_bc2_sqrt, eps);
        params[i] = p - step_size * mi / denom;
        m[i] = mi;
        v[i] = vi;
    };
#pragma unroll
    for (int k = 0; k < kKeep; ++k) {
        const int64_t i = first + k * stride;
        if (i < n_total) update(i, (float)gk[k], pk[k], mk[k], vk[k]);
    }
    for (int64_t i = first + kKeep * stride; i < n_total; i += stride)
        update(i, (float)grad[i], params[i], m[i], v[i]);
    cluster.sync();  // peers finished reading this CTA's shared memory; every CTA has read state
    if (cluster.block_rank() == 0 && tid == 64) {
        state[0] += 1;
        state[1] = __double_as_longlong(s_pow[0]);
        state[2] = __double_as_longlong(s_pow[1]);
    }
}


// ---------------------------------------------------------------------------------------------
// Data-parallel learners: one-shot all-reduce over NVLink peer memory - PUSH, LL format.
//
// Every rank owns a gather buffer  G[2 parities][world slots][slot_stride]  of 16-byte LL elements
// (common.cuh) that the other ranks of the node have mapped (CUDA IPC).  The producer of a rank's
// float64 [gradient | extra scalars] contribution - the reduction tail of the paired tensor-core
// backward kernel (mlp_bwd_tc.cu), or peer_push_kernel below for shapes that kernel does not cover
// - STORES every value, tagged with the step number, into slot `rank` of every rank's buffer:
// posted NVLink writes, nobody waits for a round trip, no fence, no flag.  The optimizer kernel of
// each rank polls the `world` slots of its OWN buffer (local memory) until each element carries
// the current step, adds them in rank order - every rank forms bit-identical sums, so the
// replicas cannot drift - and runs the clip norms and Adam on the sum.  The data path costs one
// NVLink one-way latency.
//
// The buffers are double-buffered by step parity, which makes an "I have read your slot" message
// unnecessary: a rank overwrites parity s & 1 in the backward of step s + 2, i.e. after its
// optimizer kernel of step s + 1 consumed every peer's step-(s + 1) values - and a peer sends
// those only from a backward that runs after its optimizer kernel of step s (the one that read
// the slots) has finished.  The step number lives in device memory (`seq`, advanced by the
// optimizer kernel), so producer and consumer derive parity and tag themselves and ONE captured
// CUDA graph serves every step.
//
// A rank that never delivers (its host is stuck) does not kill the others' CUDA contexts: after
// `timeout_ns` of polling the optimizer kernel sets an error word, leaves parameters, optimizer
// state and `seq` untouched and exits normally; the host raises when it reads the word.
__device__ __forceinline__ unsigned long long global_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}

constexpr int kPushThreads = 256;  // remote stores are credit-limited per SM: spread the message over many CTAs

// Stand-alone producer: local[0, n) -> slot `rank` of every rank's gather buffer.
__global__ void __launch_bounds__(kPushThreads)
peer_push_kernel(const double* __restrict__ local, int64_t n, PushArgs p) {
    const long long step = *p.seq + 1;
    const int64_t off = (step & 1) * p.buf_stride + (int64_t)p.rank * p.slot_stride;
    for (int64_t i = (int64_t)blockIdx.x * kPushThreads + threadIdx.x; i < n; i += (int64_t)gridDim.x * kPushThreads) {
        const double v = local[i];
#pragma unroll 8
        for (int r = 0; r < p.world; ++r) ll_store(p.gather[r] + off + i, v, (unsigned)step);
    }
}

// Consumer: poll the local slots, add them in rank order, clip + Adam.
__global__ void __cluster_dims__(kAdamCluster, 1, 1) __launch_bounds__(kAdamThreads)
gather_clip_adam_kernel(float* __restrict__ params, double* __restrict__ reduced,
                        const ulonglong2* __restrict__ gather, long long* __restrict__ seq,
                        int64_t slot_stride, int64_t buf_stride, int world, int n_extra,
                        float* __restrict__ m, float* __restrict__ v, int64_t* __restrict__ state,
                        int64_t n_policy, int64_t n_total, float max_norm, float lr, float beta1,
                        float beta2, float eps, double* __restrict__ norms_out, int* __restrict__ err,
                        unsigned long long timeout_ns) {
    cg::cluster_group cluster = cg::this_cluster();
    __shared__ double s_warp[2][kAdamThreads / 32];
    __shared__ double s_cta[2];
    __shared__ int s_abort;     // a thread of this CTA gave up waiting (read by the peers of the cluster)
    __shared__ int s_any_abort;
    __shared__ float s_coef[2];
    __shared__ float s_bias[2];
    __shared__ double s_pow[2];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int crank = (int)cluster.block_rank();
    const int64_t first = (int64_t)crank * kAdamThreads + tid;
    const int64_t stride = (int64_t)kAdamCluster * kAdamThreads;

    // optimizer state that does not depend on the peers: issued before anything else
    constexpr int kKeep = 2, kMaxWorld = 8;  // one NVLink node
    float pk[kKeep], mk[kKeep], vk[kKeep];
#pragma unroll
    for (int k = 0; k < kKeep; ++k) {
        const int64_t i = first + k * stride;
        pk[k] = i < n_total ? params[i] : 0.f;
        mk[k] = i < n_total ? m[i] : 0.f;
        vk[k] = i < n_total ? v[i] : 0.f;
    }
    if (tid == 0) s_abort = 0;
    if (tid == 64) {  // bias corrections from the running powers (nobody writes state before the end)
        const double p1 = state[0] == 0 ? 1.0 : __longlong_as_double(state[1]);
        const double p2 = state[0] == 0 ? 1.0 : __longlong_as_double(state[2]);
        s_pow[0] = p1 * (double)beta1, s_pow[1] = p2 * (double)beta2;
        s_bias[0] = (float)((double)lr / (1.0 - s_pow[0]));
        s_bias[1] = (float)(1.0 / sqrt(1.0 - s_pow[1]));
    }
    const long long step64 = *seq + 1;
    const unsigned step = (unsigned)step64;
    __syncthreads();

    // rank-ordered sum of entry i: all `world` loads are issued together, then each is re-polled
    // until it carries this step's tag (local memory: the peers' values arrive by themselves)
    const ulonglong2* gb = gather + (step64 & 1) * buf_stride;
    const unsigned long long t_start = global_ns();
    bool ok = true;
    auto gsum = [&](int64_t i) {
        ulonglong2 w[kMaxWorld];
#pragma unroll
        for (int r = 0; r < kMaxWorld; ++r)
            if (r < world) w[r] = ll_load(gb + r * slot_stride + i);
        double s = 0.0;
#pragma unroll
        for (int r = 0; r < kMaxWorld; ++r) {
            if (r < world) {
                unsigned spins = 0;
                while (!ll_ready(w[r], step)) {
                    if ((++spins & 255u) == 0 && global_ns() - t_start > timeout_ns) {
                        ok = false;
                        break;
                    }
                    if (spins > 16) __nanosleep(20);
                    w[r] = ll_load(gb + r * slot_stride + i);
                }
                s += ll_value(w[r]);
            }
        }
        return s;
    };
    double gk[kKeep];
    double ss0 = 0.0, ss1 = 0.0;
#pragma unroll
    for (int k = 0; k < kKeep; ++k) {
        const int64_t i = first + k * stride;
        gk[k] = i < n_total ? gsum(i) : 0.0;
        if (i < n_total) reduced[i] = gk[k];
        if (i < n_policy) ss0 += gk[k] * gk[k];
        else ss1 += gk[k] * gk[k];
    }
    for (int64_t i = first + kKeep * stride; i < n_total; i += stride) {
        const double g = gsum(i);
        reduced[i] = g;
        if (i < n_policy) ss0 += g * g;
        else ss1 += g * g;
    }
    if (crank == 0 && tid < n_extra) reduced[n_total + tid] = gsum(n_total + tid);  // logged scalars
    if (!ok) s_abort = 1;
    ss0 = warp_sum_f64(ss0);
    ss1 = warp_sum_f64(ss1);
    if (lane == 0) s_warp[0][warp] = ss0, s_warp[1][warp] = ss1;
    __syncthreads();
    if (tid < 2) {
        double s = 0.0;
        for (int i = 0; i < kAdamThreads / 32; ++i) s += s_warp[tid][i];
        s_cta[tid] = s;
    }
    cluster.sync();  // all 8 partial pairs (and abort flags) are in place
    if (tid == 0) {
        int ab = 0;
        for (int r = 0; r < kAdamCluster; ++r) ab |= *cluster.map_shared_rank(&s_abort, r);
        s_any_abort = ab;
    }
    if (tid < 2) {
        double s = 0.0;
        for (int r = 0; r < kAdamCluster; ++r) s += *cluster.map_shared_rank(&s_cta[tid], r);
        const double norm = sqrt(s);
        s_coef[tid] = (float)fmin(1.0, (double)max_norm / (norm + 1e-6));
        if (norms_out && crank == 0) norms_out[tid] = norm;
    }
    __syncthreads();
    if (!s_any_abort) {
        const float b1 = beta1, b2 = beta2, step_size = s_bias[0], inv_bc2_sqrt = s_bias[1];
        const float c0 = s_coef[0], c1 = s_coef[1];
        auto update = [&](int64_t i, float g, float p, float mi, float vi) {
            g *= (i < n_policy ? c0 : c1);
            mi = fmaf(b1, mi, (1.f - b1) * g);
            vi = fmaf(b2, vi, (1.f - b2) * g * g);
            const float denom = fmaf(sqrtf(vi), inv_bc2_sqrt, eps);
            params[i] = p - step_size * mi / denom;
            m[i] = mi;
            v[i] = vi;
        };
#pragma unroll
        for (int k = 0; k < kKeep; ++k) {
            const int64_t i = first + k * stride;
            if (i < n_total) update(i, (float)gk[k], pk[k], mk[k], vk[k]);
        }
        for (int64_t i = first + kKeep * stride; i < n_total; i += stride)
            update(i, (float)reduced[i], params[i], m[i], v[i]);
    }
    cluster.sync();  // peers finished reading this CTA's shared memory; every CTA has read state
    if (crank == 0 && tid == 64) {
        if (s_any_abort) {
            if (err) *err = 1;  // the host raises; state and seq stay as they were
        } else {
            state[0] += 1;
            state[1] = __double_as_longlong(s_pow[0]);
            state[2] = __double_as_longlong(s_pow[1]);
            *seq = step64;
        }
    }
}

}  // namespace

extern "C" int impala_clip_adam(float* params, const double* grad, float* m, float* v,
                                int64_t* state, int64_t n_policy, int64_t n_total, float max_norm,
                                float lr, float beta1, float beta2, float eps, double* norms_out,
                                void* stream) {
    if (!params || !grad || !m || !v || !state) return IMPALA_ERR_BAD_ARG;
    if (n_total < 1 || n_policy < 0 || n_policy > n_total) return IMPALA_ERR_BAD_ARG;
    clip_adam_kernel<<<kAdamCluster, kAdamThreads, 0, (cudaStream_t)stream>>>(params, grad, m, v, state, n_policy, n_total,
                                                                              max_norm, lr, beta1, beta2, eps, norms_out);
    return impala_launch_status();
}

extern "C" int impala_peer_push(const double* local, int64_t n, void* const* peer_gather, const long long* seq,
                                int64_t slot_stride, int64_t buf_stride, int rank, int world, void* stream) {
    if (!local || !peer_gather || !seq) return IMPALA_ERR_BAD_ARG;
    if (n < 1 || world < 1 || world > 8 || rank < 0 || rank >= world) return IMPALA_ERR_BAD_ARG;
    if (slot_stride < n || buf_stride < (int64_t)world * slot_stride) return IMPALA_ERR_BAD_ARG;
    PushArgs p{reinterpret_cast<ulonglong2* const*>(peer_gather), seq, slot_stride, buf_stride, rank, world};
    int sms = 0;
    cudaError_t e = impala_sm_count(&sms);
    if (e != cudaSuccess) return (int)e;
    int grid = (int)((n + kPushThreads - 1) / kPushThreads);
    if (grid > sms) grid = sms;
    peer_push_kernel<<<grid, kPushThreads, 0, (cudaStream_t)stream>>>(local, n, p);
    return impala_launch_status();
}

extern "C" int impala_gather_clip_adam(float* params, double* reduced, const void* gather, long long* seq,
                                       int64_t slot_stride, int64_t buf_stride, int world, int n_extra, float* m,
                                       float* v, int64_t* state, int64_t n_policy, int64_t n_total, float max_norm,
                                       float lr, float beta1, float beta2, float eps, double* norms_out, int* err,
                                       double timeout_s, void* stream) {
    if (!params || !reduced || !gather || !seq || !m || !v || !state) return IMPALA_ERR_BAD_ARG;
    if (n_total < 1 || n_policy < 0 || n_policy > n_total) return IMPALA_ERR_BAD_ARG;
    if (world < 1 || world > 8 || n_extra < 0 || n_extra > kAdamThreads) return IMPALA_ERR_BAD_ARG;
    if (slot_stride < n_total + n_extra || buf_stride < (int64_t)world * slot_stride) return IMPALA_ERR_BAD_ARG;
    if (reinterpret_cast<uintptr_t>(gather) & 15) return IMPALA_ERR_BAD_ARG;
    const unsigned long long timeout_ns =
        timeout_s > 0 ? (unsigned long long)(timeout_s * 1e9) : 600ull * 1000000000ull;
    gather_clip_adam_kernel<<<kAdamCluster, kAdamThreads, 0, (cudaStream_t)stream>>>(
        params, reduced, static_cast<const ulonglong2*>(gather), seq, slot_stride, buf_stride, world, n_extra, m, v, state,
        n_policy, n_total, max_norm, lr, beta1, beta2, eps, norms_out, err, timeout_ns);
    return impala_launch_status();
}
