// MLP forward on the 5th-gen tensor cores (tcgen05 + TMEM), error-compensated 3xTF32.
//
//   out[m,:] = relu(x[m,:] W1^T + b1) W2^T + b2          (models.py:23-25 / :51-52, eval mode)
//
// Layer 1 is the GEMM: per 128-row tile  D[128, H] = X'[128, K'] * W1'[H, K']^T  with the bias
// folded into K (X' = [x | 1 | 0..], W1' = [W1 | b1 | 0..], K' = 32 = one 128-byte swizzle row).
// To stay within 1e-5 of the float64 reference, every fp32 operand is split into a tf32 "hi"
// (round-to-nearest) and a "lo" remainder and three UMMAs are accumulated per K step:
// hi*hi + lo*hi + hi*lo (the dropped lo*lo term is ~2^-22 relative).  Accumulators live in
// TMEM (2 stages x 256 columns), so the CUDA cores only see the H hidden activations of a row
// once: the epilogue thread that owns TMEM lane r applies ReLU and the tiny second layer
// (<= 4 outputs) in registers and writes the row of logits / the value.
//
// Warp roles (672 threads, one persistent CTA per SM):
//   warps 0-15  epilogue: tcgen05.ld row r -> relu -> dot with W2 (smem broadcast, packed FFMA2)
//               -> global; four warps per TMEM lane quarter, each taking every fourth 32-column
//               chunk of the hidden units (partial sums meet in shared memory).  The epilogue is
//               latency- and FMA-pipe-bound, hence four warps per SM sub-partition
//   warps 16-19 producer: TMA bulk copies of raw x rows (4-deep ring, one 12 KiB copy per tile) ->
//               hi/lo split -> 128B-swizzled K-major smem tiles
//   warp  20    TMEM allocator + UMMA issuer (warp-uniform schedule, one elected lane issues)
// Pipelines: smem stage full/empty mbarriers (producer <-> UMMA, freed by tcgen05.commit) and
// TMEM stage full/empty mbarriers (UMMA <-> epilogue).
#include <cstdlib>

#include "mlp_kernels.cuh"
#include "tc_common.cuh"

// Debug timeline of CTA 0 (IMPALA_TC_TRACE=1), [tile < 24][event < 16]; see mlp_bwd_tc.cu.
__device__ long long g_trace_fwd[24 * 16];

namespace {

constexpr int kTileM = 128;
constexpr int kKPad = 32;     // floats per operand row = 128 bytes
constexpr int kStages = 2;    // x tile stages in shared memory
constexpr int kAccCols = 256; // TMEM columns per accumulator stage
constexpr int kThreads = 21 * 32;
constexpr int kTileBytes = kTileM * kKPad * 4;  // 16 KiB
constexpr int kRawStages = 4;                   // bulk-copy ring depth
constexpr int kRawStageBytes = kTileM * 28 * 4; // 14 KiB: 128 rows x O <= 28 floats

struct FwdTcArgs {
    const float* x;
    const float* params;
    float* out;
    int M, O, H, N2, num_tiles;
    int trace;
    MlpLayout lay;
};

struct __align__(8) Barriers {
    uint64_t raw_full[kRawStages], full[kStages], empty[kStages], acc_full[2], acc_empty[2];
    uint32_t tmem_base;
};

// One persistent CTA's share of a network: CTA `cta` of `ncta` takes tiles cta, cta + ncta, ...
// (a launch may give different CTA ranges to different networks, see mlp_fwd_tc_pair_kernel).
template <int NP>
__device__ __forceinline__ void fwd_tc_body(const FwdTcArgs& a, const int cta, const int ncta,
                                            long long* s_trace) {
    extern __shared__ uint8_t smem_raw[];
    // 1024-byte alignment by OFFSETTING the __shared__ array (a round trip through an integer
    // would make every derived pointer generic: LD/ST instead of LDS/STS)
    uint8_t* smem = smem_raw + ((1024u - (tc::smem_u32(smem_raw) & 1023u)) & 1023u);
    // carve-up (all tile bases 1024-byte aligned for SWIZZLE_128B)
    uint8_t* w_hi = smem;                                   // [H rows][128 B]  (<= 32 KiB)
    uint8_t* w_lo = w_hi + 256 * 128;
    uint8_t* x_hi = w_lo + 256 * 128;                       // kStages tiles
    uint8_t* x_lo = x_hi + kStages * kTileBytes;
    uint8_t* raw = x_lo + kStages * kTileBytes;             // kRawStages x 14 KiB
    float* w2s = reinterpret_cast<float*>(raw + kRawStages * kRawStageBytes);  // [H][NP]
    float* part = w2s + 256 * NP;                           // [2][3][128 rows][NP] partial sums of column groups 1-3
    Barriers* bars = reinterpret_cast<Barriers*>(part + 2 * 3 * kTileM * NP);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const bool tr = a.trace && blockIdx.x == 0 && lane == 0 && (warp == 0 || warp == 16 || warp == 20);
#define TRACE(tile, ev)                                              \
    if (tr && (tile) < 24) s_trace[(tile) * 16 + (ev)] = clock64();
    if (a.trace && blockIdx.x == 0)
        for (int k = tid; k < 24 * 16; k += kThreads) s_trace[k] = 0;
    TRACE(0, 15)
    const float* __restrict__ W1 = a.params + a.lay.oW1;
    const float* __restrict__ b1 = a.params + a.lay.ob1;
    const float* __restrict__ W2 = a.params + a.lay.oW2;
    const float* __restrict__ b2 = a.params + a.lay.ob2;
    const int O = a.O, H = a.H, ochunks = O >> 2;

    // ---- one-time setup.  The mbarriers come first, so that the bulk copies of the first x tiles
    // are already in flight while every thread stages W1' = [W1 | b1 | 0] (hi/lo swizzled tiles)
    // and W2 (transposed).
    if (warp == 20 && lane == 0) {
        for (int s = 0; s < kRawStages; ++s) tc::mbar_init(&bars->raw_full[s], 1);
        for (int s = 0; s < kStages; ++s) {
            tc::mbar_init(&bars->full[s], 4 * 32);  // every producer thread arrives
            tc::mbar_init(&bars->empty[s], 1);      // tcgen05.commit
        }
        for (int s = 0; s < 2; ++s) {
            tc::mbar_init(&bars->acc_full[s], 1);         // tcgen05.commit
            tc::mbar_init(&bars->acc_empty[s], 16 * 32);  // every epilogue thread arrives
        }
        tc::mbar_fence_init();
    }
    __syncthreads();
    const int n_my = (a.num_tiles - cta + ncta - 1) / ncta;
    // raw ring: stage i % kRawStages <- the x rows of this CTA's i-th tile (full tiles only)
    auto issue_raw = [&](int i) {
        const int tile = cta + i * ncta;
        if ((tile + 1) * kTileM <= a.M) {
            const int rs = i % kRawStages;
            const uint32_t bytes = kTileM * O * 4;
            tc::fence_proxy_async();  // earlier generic reads of this stage precede the async write
            tc::mbar_arrive_expect_tx(&bars->raw_full[rs], bytes);
            tc::bulk_g2s(raw + rs * kRawStageBytes, a.x + (size_t)tile * kTileM * O, bytes, &bars->raw_full[rs]);
        }
    };
    if (warp == 16 && lane == 0)
        for (int i = 0; i < n_my && i < kRawStages; ++i) issue_raw(i);
    if (warp == 20) tc::tmem_alloc(&bars->tmem_base, 512);
    tc::stage_w1_tiles(w_hi, w_lo, W1, b1, H, O, tid, kThreads);
    for (int idx = tid; idx < H * NP; idx += kThreads) {
        const int j = idx / NP, n = idx - j * NP;
        w2s[idx] = n < a.N2 ? __ldg(W2 + (size_t)n * H + j) : 0.f;
    }
    tc::fence_proxy_async();
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem_base = bars->tmem_base;

    if (warp < 16) {
        // =============================== epilogue ===============================
        const int q = warp & 3, grp = warp >> 2;  // TMEM lane quarter, column group
        const int nch = H >> 5;                   // 32-column chunks; group g takes chunks g, g + 4
        float2 b2p[NP == 4 ? 2 : 1];
        if constexpr (NP == 4) {
            b2p[0] = make_float2(grp == 0 && 0 < a.N2 ? __ldg(b2 + 0) : 0.f, grp == 0 && 1 < a.N2 ? __ldg(b2 + 1) : 0.f);
            b2p[1] = make_float2(grp == 0 && 2 < a.N2 ? __ldg(b2 + 2) : 0.f, grp == 0 && 3 < a.N2 ? __ldg(b2 + 3) : 0.f);
        } else {
            b2p[0] = make_float2(grp == 0 ? __ldg(b2) : 0.f, 0.f);
        }
        int it = 0;
        for (int tile = cta; tile < a.num_tiles; tile += ncta, ++it) {
            const int as = it & 1, aph = (it >> 1) & 1;
            TRACE(it, 0)
            tc::mbar_wait(&bars->acc_full[as], aph);
            tc::tc_fence_after();
            TRACE(it, 1)
            const uint32_t taddr = tmem_base + (static_cast<uint32_t>(32 * q) << 16) + as * kAccCols;
            // NP == 4: acc[0] = outputs (0,1), acc[1] = outputs (2,3); NP == 1: acc[0] = (even, odd
            // column) partial sums of the single output
            float2 acc[NP == 4 ? 2 : 1];
#pragma unroll
            for (int k = 0; k < (NP == 4 ? 2 : 1); ++k) acc[k] = b2p[k];
            // chunk by chunk (32 live accumulator registers at a time: 672 threads leave 80 each)
#pragma unroll 1
            for (int hb = 0; hb < 2; ++hb) {
                const int ch = grp + 4 * hb;
                const bool last = ch + 4 >= nch || hb == 1;
                float raw[32];
                if (ch < nch) tc::tmem_ld32(taddr + 32 * ch, raw);  // waits for the data
                if (last) {  // all of this thread's TMEM reads are complete: release the stage
                    tc::tc_fence_before();
                    tc::mbar_arrive(&bars->acc_empty[as]);
                }
                if (ch < nch) {
                    const int c0 = 32 * ch;
#pragma unroll
                    for (int i = 0; i < 32; i += 2) {
                        const float h0 = fmaxf(raw[i], 0.f);
                        const float h1 = fmaxf(raw[i + 1], 0.f);
                        if constexpr (NP == 4) {
                            const float4 wa = *reinterpret_cast<const float4*>(w2s + (c0 + i) * 4);
                            const float4 wb = *reinterpret_cast<const float4*>(w2s + (c0 + i + 1) * 4);
                            const float2 h0p = make_float2(h0, h0), h1p = make_float2(h1, h1);
                            acc[0] = tc::ffma2(h0p, make_float2(wa.x, wa.y), acc[0]);
                            acc[1] = tc::ffma2(h0p, make_float2(wa.z, wa.w), acc[1]);
                            acc[0] = tc::ffma2(h1p, make_float2(wb.x, wb.y), acc[0]);
                            acc[1] = tc::ffma2(h1p, make_float2(wb.z, wb.w), acc[1]);
                        } else {
                            const float2 w = *reinterpret_cast<const float2*>(w2s + c0 + i);
                            acc[0] = tc::ffma2(make_float2(h0, h1), w, acc[0]);
                        }
                    }
                }
                if (last) break;
            }
            TRACE(it, 2)
            const int rl = 32 * q + lane;  // row of the tile
            float* pbuf = part + (it & 1) * 3 * kTileM * NP;
            if (grp > 0) {
                float* pb = pbuf + ((grp - 1) * kTileM + rl) * NP;
                if constexpr (NP == 4) *reinterpret_cast<float4*>(pb) = make_float4(acc[0].x, acc[0].y, acc[1].x, acc[1].y);
                else pb[0] = acc[0].x + acc[0].y;
            }
            asm volatile("bar.sync 2, 512;" ::: "memory");  // the four column groups meet
            const int row = tile * kTileM + rl;
            if (grp == 0 && row < a.M) {
                if constexpr (NP == 4) {
                    const float4 p1 = *reinterpret_cast<const float4*>(pbuf + (0 * kTileM + rl) * 4);
                    const float4 p2 = *reinterpret_cast<const float4*>(pbuf + (1 * kTileM + rl) * 4);
                    const float4 p3 = *reinterpret_cast<const float4*>(pbuf + (2 * kTileM + rl) * 4);
                    const float o[4] = {((acc[0].x + p1.x) + p2.x) + p3.x, ((acc[0].y + p1.y) + p2.y) + p3.y,
                                        ((acc[1].x + p1.z) + p2.z) + p3.z, ((acc[1].y + p1.w) + p2.w) + p3.w};
                    if (a.N2 == 4) {
                        *reinterpret_cast<float4*>(a.out + (size_t)row * 4) = make_float4(o[0], o[1], o[2], o[3]);
                    } else {
#pragma unroll
                        for (int n = 0; n < 4; ++n)
                            if (n < a.N2) a.out[(size_t)row * a.N2 + n] = o[n];
                    }
                } else {
                    a.out[row] = (((acc[0].x + acc[0].y) + pbuf[rl]) + pbuf[kTileM + rl]) + pbuf[2 * kTileM + rl];
                }
            }
        }
    } else if (warp < 20) {
        // =============================== producer ===============================
        const int r = 32 * (warp - 16) + lane;  // row of the tile this thread converts
        auto tile_of = [&](int i) { return cta + i * ncta; };
        auto is_full = [&](int i) { return (tile_of(i) + 1) * kTileM <= a.M; };
        for (int it = 0; it < n_my; ++it) {
            const int s = it % kStages, ph = (it / kStages) & 1;
            const int rs = it % kRawStages, rph = (it / kRawStages) & 1;
            float4 v[8];
#pragma unroll
            for (int c = 0; c < 8; ++c) v[c] = make_float4(0.f, 0.f, 0.f, 0.f);
            TRACE(it, 5)
            if (is_full(it)) {
                tc::mbar_wait(&bars->raw_full[rs], rph);
                const float4* rx = reinterpret_cast<const float4*>(raw + rs * kRawStageBytes) + r * ochunks;
#pragma unroll
                for (int c = 0; c < 8; ++c)
                    if (c < ochunks) v[c] = rx[c];
            } else {  // ragged last tile: plain guarded loads
                const int row = tile_of(it) * kTileM + r;
                if (row < a.M) {
#pragma unroll
                    for (int c = 0; c < 8; ++c)
                        if (c < ochunks) v[c] = __ldg(reinterpret_cast<const float4*>(a.x + (size_t)row * O) + c);
                }
            }
            TRACE(it, 6)
#pragma unroll
            for (int c = 0; c < 8; ++c)
                if (c == ochunks) v[c].x = 1.f;  // the column that multiplies b1
            asm volatile("bar.sync 1, 128;" ::: "memory");  // all 4 producer warps drained the raw stage
            if (warp == 16 && lane == 0 && it + kRawStages < n_my) issue_raw(it + kRawStages);
            tc::mbar_wait(&bars->empty[s], ph ^ 1);  // UMMAs that read this stage have retired
            TRACE(it, 7)
            uint8_t* th = x_hi + s * kTileBytes;
            uint8_t* tl = x_lo + s * kTileBytes;
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                float4 hi, lo;
                tc::split_tf32(v[c].x, hi.x, lo.x);
                tc::split_tf32(v[c].y, hi.y, lo.y);
                tc::split_tf32(v[c].z, hi.z, lo.z);
                tc::split_tf32(v[c].w, hi.w, lo.w);
                const uint32_t off = tc::sw128_offset(r, c);
                *reinterpret_cast<float4*>(th + off) = hi;
                *reinterpret_cast<float4*>(tl + off) = lo;
            }
            tc::fence_proxy_async();
            tc::mbar_arrive(&bars->full[s]);
            TRACE(it, 8)
        }
    } else {
        // =============================== UMMA issuer ===============================
        // The whole warp runs the schedule (warp-uniform descriptors stay in uniform registers);
        // one elected lane issues the UMMAs and their commits.
        const uint32_t idesc = tc::instr_desc_tf32_m128(static_cast<uint32_t>(H));
        const int ksteps = (O + 1 + 7) >> 3;  // K' = O data columns + the bias column
        const uint64_t dw_hi = tc::smem_desc_k_sw128(w_hi, 0), dw_lo = tc::smem_desc_k_sw128(w_lo, 0);
        const uint64_t dx_hi = tc::smem_desc_k_sw128(x_hi, 0), dx_lo = tc::smem_desc_k_sw128(x_lo, 0);
        int it = 0;
        for (int tile = cta; tile < a.num_tiles; tile += ncta, ++it) {
            const int s = it % kStages, ph = (it / kStages) & 1;
            const int as = it & 1, aph = (it >> 1) & 1;
            TRACE(it, 9)
            tc::mbar_wait(&bars->full[s], ph);
            tc::mbar_wait(&bars->acc_empty[as], aph ^ 1);
            tc::tc_fence_after();
            TRACE(it, 10)
            if (tc::elect_one()) {
                const uint32_t d = tmem_base + as * kAccCols;
                const uint64_t xh = dx_hi + static_cast<uint64_t>((s * kTileBytes) >> 4);
                const uint64_t xl = dx_lo + static_cast<uint64_t>((s * kTileBytes) >> 4);
                // The tensor core TRUNCATES when it adds into the fp32 accumulator (measured: gradient norms
                // ~1e-6 low, growing with the number of accumulations), so the small correction terms of all
                // K steps are accumulated first and the hi*hi terms last: 4 full-magnitude additions, not 12.
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) {  // unrolled with uniform guards: constant descriptor offsets
                    if (kk < ksteps) {
                        const uint64_t ko = 2 * kk;  // 32 bytes per K = 8 step, in 16-byte units
                        tc::umma_tf32(d, xl + ko, dw_hi + ko, idesc, kk > 0);
                        tc::umma_tf32(d, xh + ko, dw_lo + ko, idesc, true);
                    }
                }
#pragma unroll
                for (int kk = 0; kk < 4; ++kk)
                    if (kk < ksteps) tc::umma_tf32(d, xh + 2 * kk, dw_hi + 2 * kk, idesc, true);
                tc::umma_commit(&bars->empty[s]);      // smem stage reusable once the UMMAs retire
                tc::umma_commit(&bars->acc_full[as]);  // accumulator ready for the epilogue
            }
            __syncwarp();
            TRACE(it, 11)
        }
    }

    tc::tc_fence_before();
    __syncthreads();
    if (warp == 20) {
        tc::tc_fence_after();
        tc::tmem_dealloc(tmem_base, 512);
    }
    if (a.trace && blockIdx.x == 0) {
        if (tid == 0) s_trace[1 * 16 + 15] = clock64();
        __syncthreads();
        for (int k = tid; k < 24 * 16; k += kThreads) g_trace_fwd[k] = s_trace[k];
    }
#undef TRACE
}

template <int NP>
__global__ void __launch_bounds__(kThreads, 1) mlp_fwd_tc_kernel(const __grid_constant__ FwdTcArgs a) {
    __shared__ long long s_trace[24 * 16];
    fwd_tc_body<NP>(a, blockIdx.x, gridDim.x, s_trace);
}

// Policy and value network of one learner step in ONE launch: CTAs [0, n_pi) run the policy
// tiles, the rest the value-function tiles.  Both read the same observations; one launch means
// one prologue per SM and a finer tile quantisation (8.9 instead of 4.3 + 4.5 tiles per CTA at c4).
__global__ void __launch_bounds__(kThreads, 1)
mlp_fwd_tc_pair_kernel(const __grid_constant__ FwdTcArgs a_pi, const __grid_constant__ FwdTcArgs a_vf,
                       const int n_pi) {
    __shared__ long long s_trace[24 * 16];
    if ((int)blockIdx.x < n_pi) fwd_tc_body<4>(a_pi, blockIdx.x, n_pi, s_trace);
    else fwd_tc_body<1>(a_vf, (int)blockIdx.x - n_pi, (int)gridDim.x - n_pi, s_trace);
}

constexpr size_t kSmemBytes = 1024 /*alignment slack*/ + 2 * 256 * 128 + 2 * kStages * kTileBytes +
                              kRawStages * kRawStageBytes + (256 + 2 * 3 * kTileM) * 4 * sizeof(float) + sizeof(Barriers);

}  // namespace

// Shapes the tensor-core path covers; everything else stays on the FP32 kernels.
bool impala_mlp_fwd_tc_eligible(const float* x, int M, int O, int H, int N2) {
    return M >= 1 && O >= 4 && O <= 28 && (O & 3) == 0 && H >= 16 && H <= 256 && (H & 31) == 0 &&
           N2 >= 1 && N2 <= 4 && (reinterpret_cast<uintptr_t>(x) & 15) == 0;
}

namespace {
FwdTcArgs make_fwd_args(const float* x, const float* params, float* out, int M, int O, int H, int N2) {
    FwdTcArgs a{};
    a.x = x, a.params = params, a.out = out;
    a.M = M, a.O = O, a.H = H, a.N2 = N2;
    a.num_tiles = (M + kTileM - 1) / kTileM;
    a.lay = impala_make_layout(O, H, N2);
    const char* tr_env = std::getenv("IMPALA_TC_TRACE");
    a.trace = tr_env && tr_env[0] == '1';
    return a;
}
}  // namespace

int impala_mlp_fwd_tc(const float* x, const float* params, float* out, int M, int O, int H, int N2,
                      cudaStream_t st) {
    const FwdTcArgs a = make_fwd_args(x, params, out, M, O, H, N2);
    static bool opted[64][2] = {};  // per device
    cudaError_t e;
    int sms = 0, dev = 0;
    if ((e = impala_sm_count(&sms)) != cudaSuccess) return (int)e;
    if ((e = cudaGetDevice(&dev)) != cudaSuccess) return (int)e;
    const int which = N2 == 1 ? 0 : 1;
    auto kernel = which ? mlp_fwd_tc_kernel<4> : mlp_fwd_tc_kernel<1>;
    if (dev < 0 || dev >= 64 || !opted[dev][which]) {
        e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemBytes);
        if (e != cudaSuccess) return (int)e;
        if (dev >= 0 && dev < 64) opted[dev][which] = true;
    }
    const int grid = a.num_tiles < sms ? a.num_tiles : sms;
    kernel<<<grid, kThreads, kSmemBytes, st>>>(a);
    return impala_launch_status();
}

// Both networks in one launch (policy: 2..4 outputs, value fn: 1 output); the caller has checked
// impala_mlp_fwd_tc_eligible for each.  Per-tile cost weights (policy epilogue does 4 FFMA per
// hidden unit, the value fn 1) split the SMs between the two tile lists.
int impala_mlp_fwd_tc_pair(const float* x, const float* params_pi, const float* params_vf, float* logits,
                           float* values, int M_pi, int M_vf, int O, int H_pi, int H_vf, int A,
                           cudaStream_t st) {
    const FwdTcArgs a_pi = make_fwd_args(x, params_pi, logits, M_pi, O, H_pi, A);
    const FwdTcArgs a_vf = make_fwd_args(x, params_vf, values, M_vf, O, H_vf, 1);
    static bool opted[64] = {};  // per device
    cudaError_t e;
    int sms = 0, dev = 0;
    if ((e = impala_sm_count(&sms)) != cudaSuccess) return (int)e;
    if ((e = cudaGetDevice(&dev)) != cudaSuccess) return (int)e;
    if (dev < 0 || dev >= 64 || !opted[dev]) {
        e = cudaFuncSetAttribute(mlp_fwd_tc_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)kSmemBytes);
        if (e != cudaSuccess) return (int)e;
        if (dev >= 0 && dev < 64) opted[dev] = true;
    }
    const int total_tiles = a_pi.num_tiles + a_vf.num_tiles;
    const int grid = total_tiles < sms ? total_tiles : sms;
    // per-tile cost of a policy tile in % of a value-function tile, per 32 hidden units: measured on a B200 (c4)
    constexpr int kPairCostFwd = 160;
    const int n_pi = impala_pair_split(a_pi.num_tiles, a_vf.num_tiles, grid,
                                       kPairCostFwd * (H_pi / 32),
                                       100 * (H_vf / 32));
    mlp_fwd_tc_pair_kernel<<<grid, kThreads, kSmemBytes, st>>>(a_pi, a_vf, n_pi);
    return impala_launch_status();
}

// Debug only: the [24 tiles][16 events] clock stamps of the last traced forward launch (CTA 0).
extern "C" int impala_debug_read_trace_fwd(long long* out, int n) {
    cudaDeviceSynchronize();
    if (n > 24 * 16) n = 24 * 16;
    if (cudaMemcpyFromSymbol(out, g_trace_fwd, sizeof(long long) * n) != cudaSuccess) return -1;
    return n;
}
