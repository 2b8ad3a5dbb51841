// V-trace targets, the three losses and their closed-form backward
// (reference learner.py:116-162 + helpers :298-321 + the non-MLP part of :175).
//
// Lane = trajectory, warp = time segment (vtrace_lane_kernel below): every tensor of the
// time-major (T, B[, A]) batch is read and written as fully coalesced row segments straight from /
// to global memory (128-bit accesses for the logits), the T-step recurrence is split over the
// warps of a CTA as composed affine maps (one barrier per chunk), and everything else stays in
// registers.
//
// Transcendentals use the hardware approximations (ex2/lg2.approx.ftz, relative error ~2^-22) in
// the base-2 domain: the arguments are differences from the row maximum (<= 0) and sums in
// [1, A], so the absolute error stays ~1e-7, far inside the 1e-5 parity budget, at a fraction of
// the instruction count of expf/logf.
//
// Reference quirks reproduced in IMPALA_MODE_REFERENCE (SURVEY.md section 0.2):
//   delta_t = rho_t (r_t + gamma v_{t+1} - v_0)                  learner.py:126  (v[:1])
//   acc_i   = delta_i + disc_i c_i (acc_{i+1} - v_{i+1})          learner.py:130
//   vs = acc + v (:131);  pg_t = rho_t (r_t + disc_t vs_{t+1} - v_t)   (:135)
// i.e. the affine map F_i(x) = (delta_i - g_i v_{i+1}) + g_i x with g_i = disc_i c_i.
#include <math.h>

#include "common.cuh"

namespace {

// ex2 / lg2 hardware approximations with flush-to-zero (no denormal fix-up code): relative error
// ~2^-22.  Softmax is evaluated in the base-2 domain: zs = z * log2(e), p_k = 2^(zs_k - lse2).
__device__ __forceinline__ float ex2f(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float lg2f(float x) {
    float y;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
constexpr float kLog2e = 1.4426950408889634f, kLn2 = 0.6931471805599453f;
// p ? x : y as an opaque selp: a plain C++ select chain over the logits of a step ("the logit of the
// taken action") is turned into a dynamically indexed load by the compiler, which sends the whole
// register array to local memory.
__device__ __forceinline__ float selp_f32(bool p, float x, float y) {
    float d;
    asm("{\n\t.reg .pred q;\n\tsetp.ne.s32 q, %3, 0;\n\tselp.f32 %0, %1, %2, q;\n\t}" : "=f"(d) : "f"(x), "f"(y), "r"((int)p));
    return d;
}

constexpr int kMaxSeg = 32;  // time segments (= warps) per CTA

struct VtArgs {
    const float* cur_logits;
    const float* beh_logits;
    const int32_t* actions;
    const float* rewards;
    const uint8_t* done;
    const int32_t* lens;
    const float* v;
    float* vs;
    float* pg_adv;
    float* dlogits;
    float* dv;
    double* scalars;
    double* partials;        // [gridDim.x][4] per-CTA loss sums (workspace)
    unsigned int* counter;   // CTA arrival counter (workspace; zero on entry, zero on exit)
    int T, B, A, mode;
    float gamma, rho_bar, c_bar, v_loss_c, policy_loss_c, entropy_c, inv_batch;
};

// Row loads / stores of the (T, B, A) logits: lane = trajectory, so a warp reads 32 * A consecutive
// floats of a time step.  VEC (A == AP, 16-byte aligned bases): one 128-bit (A = 4), one 64-bit
// (A = 2) or AP/4 128-bit accesses per lane, i.e. 512 contiguous bytes per warp instruction at A = 4.
template <int AP, bool VEC>
__device__ __forceinline__ void load_logits(const float* __restrict__ p, unsigned elem, int A, float (&z)[AP]) {
    if constexpr (VEC && AP == 2) {
        const float2 q = __ldg(reinterpret_cast<const float2*>(p + elem * 2));
        z[0] = q.x, z[1] = q.y;
    } else if constexpr (VEC) {
#pragma unroll
        for (int k = 0; k < AP; k += 4) {
            const float4 q = __ldg(reinterpret_cast<const float4*>(p + elem * AP + k));
            z[k] = q.x, z[k + 1] = q.y, z[k + 2] = q.z, z[k + 3] = q.w;
        }
    } else {
#pragma unroll
        for (int k = 0; k < AP; ++k) z[k] = k < A ? __ldg(p + elem * A + k) : 0.f;
    }
}
template <int AP, bool VEC>
__device__ __forceinline__ void store_logits(float* __restrict__ p, unsigned elem, int A, const float (&z)[AP]) {
    if constexpr (VEC && AP == 2) {
        *reinterpret_cast<float2*>(p + elem * 2) = make_float2(z[0], z[1]);
    } else if constexpr (VEC) {
#pragma unroll
        for (int k = 0; k < AP; k += 4)
            *reinterpret_cast<float4*>(p + elem * AP + k) = make_float4(z[k], z[k + 1], z[k + 2], z[k + 3]);
    } else {
#pragma unroll
        for (int k = 0; k < AP; ++k)
            if (k < A) p[elem * A + k] = z[k];
    }
}

// ------------------------------------------------------------------------------------------------
// Lane = trajectory, warp = time segment.
//
// A CTA owns 32 consecutive trajectories (one per lane: every global access of a time step is a
// fully coalesced row segment - 512 B of logits, 128 B of rewards / actions / values, 32 B of done
// flags per warp instruction - with no shared-memory transposition) and NSEG warps; warp w owns
// the S consecutive time steps [t0 + w S, t0 + (w + 1) S) of the current chunk of S * NSEG steps.
// The unroll is walked backwards chunk by chunk.  Per chunk a thread
//   1. loads its S rows (all loads independent of the recurrence, issued up front),
//   2. evaluates the per-step terms (log-softmax of both logit vectors, rho, c, the affine map
//      F_t(x) = fa_t + g_t x of the recurrence) and scans its segment with carry 0, keeping
//      acc0_t and the running product P_t = g_t ... g_(end of segment),
//   3. publishes the segment's composed map (acc0, P) in shared memory; after ONE barrier every
//      thread composes the maps of the later segments (<= NSEG - 1 FMAs) on top of the carry of the
//      previous chunk and gets the accumulator that enters its segment,
//   4. fixes up acc_t = acc0_t + P_t * carry in registers, forms vs / pg_adv (and, WITH_LOSS, the
//      loss terms and closed-form gradients) and stores them row-contiguously.
// Total threads = B * NSEG, so the small benchmark batch (T = 20, B = 4096) still spreads over
// 1280 warps and the long unroll (T = 100, B = 8192) keeps ~2 500 warps x S rows of loads in flight.
// ------------------------------------------------------------------------------------------------
template <int AP, int S, bool WITH_LOSS, bool VEC>
__global__ void __launch_bounds__(512, 1) vtrace_lane_kernel(const VtArgs a) {
    __shared__ float2 s_map[2][kMaxSeg][32];
    __shared__ double s_red[kMaxSeg][4];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const int T = a.T, B = a.B, A = VEC ? AP : a.A;
    const int b = blockIdx.x * 32 + lane;
    const bool live = b < B;
    const int bl = live ? b : B - 1;  // column this lane loads
    const int L = live ? min(max(__ldg(a.lens + bl), 0), T) : 0;
    const float v0 = __ldg(a.v + bl);  // V(x_0): the reference's v[:1]
    const int rows = S * nw;
    const int nch = (T + rows - 1) / rows;
    const bool ref_mode = a.mode == IMPALA_MODE_REFERENCE;

    double sum_vl = 0.0, sum_pl = 0.0, sum_ent = 0.0, sum_rw = 0.0;
    float chunk_carry = 0.f;  // accumulator at the first step after the current chunk
    // One chunk's raw rows of this thread (registers).  Unpredicated loads: steps past the unroll
    // (last chunk only) re-read step T - 1 and dead lanes read trajectory B - 1; both are masked
    // by `valid` below (rho = c = disc = 0).
    struct Rows {
        float zc[S][AP], zb[S][AP], r[S], vv[S + 1];
        int act[S];
        unsigned char dn[S];  // raw: compared where it is used, so the load is not waited for at issue
    };
    auto load_rows = [&](Rows& R, const int c) {
        const int tb = c * rows + w * S;
#pragma unroll
        for (int i = 0; i < S; ++i) {
            const unsigned e = (unsigned)min(tb + i, T - 1) * (unsigned)B + (unsigned)bl;
            load_logits<AP, VEC>(a.cur_logits, e, A, R.zc[i]);
            load_logits<AP, VEC>(a.beh_logits, e, A, R.zb[i]);
            R.r[i] = __ldg(a.rewards + e);
            R.act[i] = __ldg(a.actions + e);
            R.dn[i] = __ldg(a.done + e);
        }
#pragma unroll
        for (int i = 0; i <= S; ++i) R.vv[i] = __ldg(a.v + (unsigned)min(tb + i, T) * (unsigned)B + (unsigned)bl);
    };
    auto process = [&](Rows& R, const int c) {
        const int tb = c * rows + w * S;  // first step of this thread's segment
        // ---- 2. per-step terms and the zero-carry scan of this segment
        float rho[S], disc[S], fa[S], g[S], lp2a[S];
#pragma unroll
        for (int i = 0; i < S; ++i) {
            const bool valid = tb + i < L;
            // log-softmax of both logit vectors in the base-2 domain (learner.py:298-303)
            float mx = R.zc[i][0], mxb = R.zb[i][0];
#pragma unroll
            for (int k = 1; k < AP; ++k)
                if (k < A) mx = fmaxf(mx, R.zc[i][k]), mxb = fmaxf(mxb, R.zb[i][k]);
            float se = 0.f, seb = 0.f;
            const float mxl = -mx * kLog2e, mxbl = -mxb * kLog2e;
#pragma unroll
            for (int k = 0; k < AP; ++k) {
                R.zc[i][k] = fmaf(R.zc[i][k], kLog2e, mxl);   // (z - max) log2(e), one rounding
                R.zb[i][k] = fmaf(R.zb[i][k], kLog2e, mxbl);
                if (k < A) se += ex2f(R.zc[i][k]), seb += ex2f(R.zb[i][k]);
            }
            const float lse = lg2f(se), lseb = lg2f(seb);
            float z_a = R.zc[i][0], zb_a = R.zb[i][0];
#pragma unroll
            for (int k = 1; k < AP; ++k) {
                const bool hit = k == R.act[i];
                z_a = selp_f32(hit, R.zc[i][k], z_a), zb_a = selp_f32(hit, R.zb[i][k], zb_a);
            }
#pragma unroll
            for (int k = 0; k < AP; ++k) R.zc[i][k] -= lse;  // log2 pi(k)
            lp2a[i] = z_a - lse;                                               // log2 pi(a)
            const float ratio = ex2f(lp2a[i] - (zb_a - lseb));                 // :121-123
            rho[i] = valid ? fminf(ratio, a.rho_bar) : 0.f;                    // :124
            const float cc = valid ? fminf(ratio, a.c_bar) : 0.f;              // :125
            disc[i] = (valid && R.dn[i] == 0) ? a.gamma : 0.f;                       // :109
            g[i] = disc[i] * cc;
            if (ref_mode) {
                const float delta = rho[i] * (R.r[i] + a.gamma * R.vv[i + 1] - v0);  // :126
                fa[i] = delta - g[i] * R.vv[i + 1];                                // :130
            } else {
                fa[i] = rho[i] * (R.r[i] + disc[i] * R.vv[i + 1] - R.vv[i]);
            }
        }
        float acc[S + 1], P[S];
        acc[S] = 0.f;
        float prod = 1.f;
#pragma unroll
        for (int i = S - 1; i >= 0; --i) {
            acc[i] = fmaf(g[i], acc[i + 1], fa[i]);
            prod *= g[i];
            P[i] = prod;
        }
        // ---- 3. exchange the composed maps of the segments, find the carry entering this segment.
        // The carry entering segment s is  A_s + Pm_s * x  with x the carry entering the LAST segment
        // (the previous chunk's carry); composing all nw maps gives the carry this chunk passes on.
        const int par = c & 1;
        s_map[par][w][lane] = make_float2(acc[0], P[0]);
        __syncthreads();
        float cA = 0.f, cP = 1.f, mineA = 0.f, mineP = 1.f;
        for (int s2 = nw - 1; s2 >= 0; --s2) {
            if (s2 == w) mineA = cA, mineP = cP;
            const float2 q = s_map[par][s2][lane];
            cA = fmaf(q.y, cA, q.x);
            cP = q.y * cP;
        }
        const float x = chunk_carry;
        chunk_carry = fmaf(cP, x, cA);
        const float mine = fmaf(mineP, x, mineA);

        // ---- 4. fix-up, outputs, loss terms
        acc[S] = mine;
#pragma unroll
        for (int i = S - 1; i >= 0; --i) {
            const int t = tb + i;
            const bool valid = t < L;
            acc[i] = fmaf(P[i], mine, acc[i]);
            const float vs_n = acc[i + 1] + R.vv[i + 1];                         // :131
            const float pg = rho[i] * (R.r[i] + disc[i] * vs_n - R.vv[i]);         // :135
            const unsigned e = (unsigned)t * (unsigned)B + (unsigned)b;
            if (live && t < T) {
                if (a.vs) a.vs[e] = (t <= L) ? acc[i] + R.vv[i] : 0.f;
                if (a.pg_adv) a.pg_adv[e] = pg;  // rho == 0 on padding
                if (t == T - 1 && a.vs) a.vs[e + B] = (L == T) ? R.vv[i + 1] : 0.f;  // bootstrap row
            }
            if constexpr (WITH_LOSS) {
                // d total / d v = v_loss_c (v - vs) / B = -v_loss_c acc / B  (:149, :306-307)
                float ent = 0.f, pk[AP], lz[AP], dz[AP];
#pragma unroll
                for (int k = 0; k < AP; ++k) {
                    lz[k] = R.zc[i][k] * kLn2;
                    pk[k] = (k < A) ? ex2f(R.zc[i][k]) : 0.f;
                    if (k < A) ent -= pk[k] * lz[k];                           // :310-314, :153
                }
#pragma unroll
                for (int k = 0; k < AP; ++k) {
                    const float onehot = (k == R.act[i]) ? 1.f : 0.f;
                    const float d = a.inv_batch * (a.policy_loss_c * pg * (pk[k] - onehot) +
                                                   a.entropy_c * pk[k] * (lz[k] + ent));
                    dz[k] = (valid && k < A) ? d : 0.f;
                }
                if (live && t < T) {
                    a.dv[e] = valid ? -a.v_loss_c * a.inv_batch * acc[i] : 0.f;
                    if (t == T - 1) a.dv[e + B] = 0.f;
                    store_logits<AP, VEC>(a.dlogits, e, A, dz);
                }
                if (valid) {
                    sum_vl += 0.5 * (double)acc[i] * (double)acc[i];
                    sum_pl += (double)(-(lp2a[i] * kLn2) * pg);                // :317-321
                    sum_ent += (double)ent;
                    sum_rw += (double)R.r[i];                                    // :108
                }
            }
        }
    };
    // Chunks are walked backwards with the NEXT chunk's loads already in flight while the current one
    // is processed (two register sets, loop unrolled by two): without it every CTA alternates between
    // a pure memory phase and a pure compute phase and, all CTAs having started together, so does
    // the whole GPU.
    {
        Rows R0, R1;
        int c = nch - 1;
        load_rows(R0, c);
        while (true) {
            if (c > 0) load_rows(R1, c - 1);
            process(R0, c);
            if (--c < 0) break;
            if (c > 0) load_rows(R0, c - 1);
            process(R1, c);
            if (--c < 0) break;
        }
    }

    if constexpr (WITH_LOSS) {
        // per-CTA sums -> workspace; the last CTA to arrive adds them up in a fixed order
        // (bitwise reproducible, no float64 atomics, no memset node) and re-arms the counter.
        __shared__ bool s_last;
        __shared__ double s_fin[32][4];
        const int tid = threadIdx.x;
        sum_vl = warp_sum_f64(sum_vl);
        sum_pl = warp_sum_f64(sum_pl);
        sum_ent = warp_sum_f64(sum_ent);
        sum_rw = warp_sum_f64(sum_rw);
        if (lane == 0) s_red[w][0] = sum_vl, s_red[w][1] = sum_pl, s_red[w][2] = sum_ent, s_red[w][3] = sum_rw;
        __syncthreads();
        if (tid < 4) {
            double s = 0.0;
            for (int i = 0; i < nw; ++i) s += s_red[i][tid];
            a.partials[(size_t)blockIdx.x * 4 + tid] = s;
            __threadfence();
        }
        __syncthreads();
        if (tid == 0) s_last = atomicAdd(a.counter, 1u) == gridDim.x - 1;
        __syncthreads();
        if (s_last) {
            __threadfence();
            const int nthr = (int)blockDim.x, which = tid & 3, stripe = tid >> 2, nstripes = nthr >> 2;
            double s = 0.0;
            for (unsigned cta = stripe; cta < gridDim.x; cta += nstripes)
                s += __ldcg(a.partials + (size_t)cta * 4 + which);
            // fixed-order tree over the stripes of each scalar: lanes {which, which + 4, ...} of a warp,
            // then the warps through shared memory
            s += __shfl_xor_sync(IMPALA_FULL_MASK, s, 4);
            s += __shfl_xor_sync(IMPALA_FULL_MASK, s, 8);
            s += __shfl_xor_sync(IMPALA_FULL_MASK, s, 16);
            if (lane < 4) s_fin[w][lane] = s;
            __syncthreads();
            if (tid < 4) {
                double tot = 0.0;
                for (int i = 0; i < nw; ++i) tot += s_fin[i][tid];
                a.scalars[tid] = tot * (double)a.inv_batch;
            }
            if (tid == 0) *a.counter = 0u;
        }
    }
}

int pick_ap(int A) {
    if (A <= 2) return 2;
    if (A <= 4) return 4;
    if (A <= 8) return 8;
    if (A <= 16) return 16;
    return 0;
}

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

template <int AP, int S, bool WITH_LOSS>
int launch_s(const VtArgs& a, bool vec, unsigned groups, int nw, cudaStream_t st) {
    if (vec)
        vtrace_lane_kernel<AP, S, WITH_LOSS, true><<<groups, 32 * nw, 0, st>>>(a);
    else
        vtrace_lane_kernel<AP, S, WITH_LOSS, false><<<groups, 32 * nw, 0, st>>>(a);
    return impala_launch_status();
}

// Steps per thread (S) and warps per CTA (nw); the widest action set trades S for registers.
// Measured on B200 (ncu): S = 2; up to 10 segments (T <= 20) one CTA holds the whole unroll in one
// chunk; longer unrolls walk chunks of 8 x S steps with 8 warps per CTA (T = 100, B = 8192: 17.4 us).
// Spreading the segments of a long unroll over a thread-block cluster (DSMEM carry exchange, 4 or 8
// CTAs) was measured SLOWER - 34-42 us at T = 100, B = 8192: the cluster barriers cost more than
// the chunk loop they replace.
template <bool WITH_LOSS>
int launch(VtArgs& a, cudaStream_t st) {
    if (a.T < 1 || a.B < 1 || a.A < 1) return IMPALA_ERR_BAD_ARG;
    const int AP = pick_ap(a.A);
    if (!AP) return IMPALA_ERR_UNSUPPORTED_SHAPE;
    // 32-bit element offsets inside the kernel
    if ((int64_t)(a.T + 1) * a.B * AP >= (int64_t)1 << 31) return IMPALA_ERR_UNSUPPORTED_SHAPE;
    const unsigned groups = (unsigned)((a.B + 31) / 32);
    const bool vec = a.A == AP && aligned16(a.cur_logits) && aligned16(a.beh_logits) &&
                     (!WITH_LOSS || aligned16(a.dlogits));
    const int S = AP == 16 ? 1 : 2;
    const int nseg = (a.T + S - 1) / S;
    const int nw = nseg <= 10 ? nseg : 8;
    if (AP == 2) return launch_s<2, 2, WITH_LOSS>(a, vec, groups, nw, st);
    if (AP == 4) return launch_s<4, 2, WITH_LOSS>(a, vec, groups, nw, st);
    if (AP == 8) return launch_s<8, 2, WITH_LOSS>(a, vec, groups, nw, st);
    return launch_s<16, 1, WITH_LOSS>(a, vec, groups, nw, st);
}

}  // namespace

extern "C" int impala_vtrace(const float* cur_logits, const float* beh_logits,
                             const int32_t* actions, const float* rewards, const uint8_t* done,
                             const int32_t* lens, const float* v, float* vs, float* pg_adv, int T,
                             int B, int A, float gamma, float rho_bar, float c_bar, int mode,
                             void* stream) {
    if (!cur_logits || !beh_logits || !actions || !rewards || !done || !lens || !v || !vs || !pg_adv)
        return IMPALA_ERR_BAD_ARG;
    if (mode != IMPALA_MODE_REFERENCE && mode != IMPALA_MODE_PAPER) return IMPALA_ERR_BAD_ARG;
    VtArgs a{};
    a.cur_logits = cur_logits, a.beh_logits = beh_logits, a.actions = actions, a.rewards = rewards;
    a.done = done, a.lens = lens, a.v = v, a.vs = vs, a.pg_adv = pg_adv;
    a.T = T, a.B = B, a.A = A, a.mode = mode;
    a.gamma = gamma, a.rho_bar = rho_bar, a.c_bar = c_bar;
    return launch<false>(a, (cudaStream_t)stream);
}

extern "C" int64_t impala_vtrace_loss_workspace(int T, int B, int A) {
    if (T < 1 || B < 1 || A < 1) return IMPALA_ERR_BAD_ARG;
    const int64_t grid = ((int64_t)B + 31) / 32;  // one row per CTA
    return grid * 4 * (int64_t)sizeof(double) + 16;  // per-CTA sums + arrival counter
}

extern "C" int impala_vtrace_loss(const float* cur_logits, const float* beh_logits,
                                  const int32_t* actions, const float* rewards,
                                  const uint8_t* done, const int32_t* lens, const float* v,
                                  float* vs, float* pg_adv, float* dlogits, float* dv,
                                  double* scalars, void* workspace, int64_t workspace_bytes, int T,
                                  int B, int A, float gamma, float rho_bar, float c_bar,
                                  float v_loss_c, float policy_loss_c, float entropy_c,
                                  float inv_batch, int mode, void* stream) {
    if (!cur_logits || !beh_logits || !actions || !rewards || !done || !lens || !v || !dlogits ||
        !dv || !scalars || !workspace)
        return IMPALA_ERR_BAD_ARG;
    if (mode != IMPALA_MODE_REFERENCE && mode != IMPALA_MODE_PAPER) return IMPALA_ERR_BAD_ARG;
    const int64_t need = impala_vtrace_loss_workspace(T, B, A);
    if (need < 0) return (int)need;
    if (workspace_bytes < need) return IMPALA_ERR_WORKSPACE_TOO_SMALL;
    if (reinterpret_cast<uintptr_t>(workspace) & 15) return IMPALA_ERR_BAD_ARG;
    VtArgs a{};
    a.cur_logits = cur_logits, a.beh_logits = beh_logits, a.actions = actions, a.rewards = rewards;
    a.done = done, a.lens = lens, a.v = v, a.vs = vs, a.pg_adv = pg_adv, a.dlogits = dlogits;
    a.dv = dv, a.scalars = scalars;
    // workspace = [counter (16 bytes) | per-CTA sums]
    a.counter = reinterpret_cast<unsigned int*>(workspace);
    a.partials = reinterpret_cast<double*>(reinterpret_cast<char*>(workspace) + 16);
    a.T = T, a.B = B, a.A = A, a.mode = mode;
    a.gamma = gamma, a.rho_bar = rho_bar, a.c_bar = c_bar;
    a.v_loss_c = v_loss_c, a.policy_loss_c = policy_loss_c, a.entropy_c = entropy_c;
    a.inv_batch = inv_batch;
    return launch<true>(a, (cudaStream_t)stream);
}
