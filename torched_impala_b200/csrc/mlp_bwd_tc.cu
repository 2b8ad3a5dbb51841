// MLP backward on the 5th-gen tensor cores (tcgen05 + TMEM), error-compensated 3xTF32.
//
// Gradient of sum_m <dout[m,:], mlp(x[m,:])> w.r.t. (W1, b1, W2, b2)  (autograd at learner.py:175).
// Transposed formulation so that a thread owns a HIDDEN unit (TMEM lane = hidden unit), per tile
// of 64 batch rows:
//
//   UMMA1 (SS, recompute)  PRE[H, 64]  = W1'[H, K'] * X'[64, K']^T   X' = [x | 1 | 0], W1' = [W1 | b1 | 0]
//   CUDA cores             h = relu(PRE); dh = W2^T dz; dW2 += dz h;  DP = (PRE > 0) ? dh : 0
//   UMMA2 (TS, reduction)  dW1'[H, K'] += DP[H, 64] * X'[64, K']      column O of dW1' = db1
// The bias rides in K (column O of X' is 1): the pre-activation arrives complete and db1 falls out
// of the reduction GEMM for free.  The epilogue is bound by the FMA pipe (13 packed fp32 ops per
// (row pair, hidden unit) in round 1: bias, two mask multiplies, dh, dW2, DP, db1, hi/lo split);
// with the bias and db1 on the tensor cores and ReLU / ReLU' as FMNMX / FSEL on the ALU pipe, 9
// remain (policy; 3 for the value net) - the fourth K step of UMMA1 at O = 24 is paid by a pipe
// that is idle half of the time.
//
// PRE lands in TMEM; the epilogue thread that owns lane j reads its 64 pre-activations, and
// writes DP back INTO TENSOR MEMORY (hi in place of PRE, lo in a second region) with tcgen05.st,
// so UMMA2 takes its A operand from TMEM and only the small X'^T tile is fetched from shared
// memory (with both operands in smem an M128xN32xK8 UMMA is operand-fetch bound at ~5x its math
// time - measured, see DESIGN.md section 6).  dW1' accumulates in TMEM across every tile of the
// persistent CTA and is read out once.  K' = 32 floats = one 128-byte swizzle row, so W1', X'
// and X'^T tiles share one smem format (K-major, SWIZZLE_128B); the producer writes each x tile
// row-major (B of UMMA1, K = features) and transposed (B of UMMA2, K = batch rows).  Operands
// are split into tf32 hi + lo and three UMMAs (hi*hi + lo*hi + hi*lo) are issued per K step
// (x and W1: hi = round-to-nearest tf32; DP: hi = dp with the low 13 mantissa bits cleared - one
// LOP3 where cvt.rna.tf32 is a four-instruction sequence - and lo = the exact remainder).
//
// UMMA2 issues two instead of three products per K step: the x^T tile stacks the hi and lo
// features as 64 rows, so  DP_hi x [X'^T_hi ; X'^T_lo]  (N = 64) yields dp_hi*x_hi and dp_hi*x_lo
// in adjacent accumulator columns (summed at read-out) and  DP_lo x X'^T_hi  (N = 32) adds the
// third term - small-N UMMAs cost ~40 cycles each regardless of N, so fewer, wider ones win.
//
// TMEM map (512 columns): [0,256) two PRE/DP_hi buffers x (2 hidden blocks x 64 rows),
//                         [256,384) DP_lo, [384,512) dW1' accumulators (2 blocks x (32 + 32)).
// Warp roles (608 threads, one persistent CTA per SM):
//   warps 0-15  epilogue: thread = (hidden unit j, half of the tile's 64 batch rows); TMEM lane
//               j % 128, block j / 128.  The epilogue is latency-bound, so four warps per SM
//               sub-partition (instead of two with 64 rows per thread) is what keeps it off the
//               critical path; the two halves' dW2 / db1 sums meet in shared memory at the end
//   warps 16-17 producer: TMA bulk copies of raw x / dout rows (4-deep ring) -> hi/lo tiles; db2
//   warp  18    TMEM allocator + UMMA issuer (warp-uniform schedule, one elected lane issues)
//
// Cross-CTA reduction: every CTA writes its float32 partial gradient row, the grid meets at an
// arrival counter (grid <= SM count and one CTA per SM, so all CTAs are co-resident), and CTA c
// then sums entries [64c, 64c+64) over all rows in float64 in a fixed order - the rows are still
// in L2, the result is bitwise reproducible, and no second launch sits between the two backward
// kernels of a step.
#include <cstdlib>

#include "mlp_kernels.cuh"
#include "tc_common.cuh"

// Debug timeline (IMPALA_TC_TRACE=1): CTA 0 keeps clock64() stamps of its pipeline events in
// shared memory and dumps them at exit; read back through impala_debug_read_trace (not part of
// the public ABI).  Layout: [tile < 24][event < 16].
__device__ long long g_trace[24 * 16];

namespace {

constexpr int kRowsT = 64;       // batch rows per tile: N of UMMA1, K of UMMA2
constexpr int kKPad = 32;        // padded feature count K' (data + bias column + zeros)
constexpr int kXStages = 3;      // converted x / x^T / dz stages
constexpr int kRawStages = 4;    // bulk-copy ring depth
constexpr int kWarps = 19;
constexpr int kThreads = kWarps * 32;
constexpr int kEpiThreads = 16 * 32;
constexpr int kWTileBytes = 256 * 128;      // 256 hidden rows x 128 B
constexpr int kXTileBytes = kRowsT * 128;   // 8 KiB: 64 rows x 128 B (also 2 x [32 rows x 128 B])
constexpr int kRawStageBytes = 8192;        // x rows (<= 64*28*4 = 7168 B) | dout rows at +7168
constexpr int kRawDzOffset = 7168;
constexpr int kColLo = 256;                 // TMEM column of DP_lo
constexpr int kColAcc = 384;                // TMEM column of the dW1' accumulators

struct BwdTcArgs {
    const float* x;
    const float* params;
    const float* dout;
    float* ws;
    double* grad;        // float64 [lay.total], written by the in-kernel reduction
    unsigned int* ctl;   // {arrivals, departures}: zero on entry, zero on exit
    int M, O, H, N2, num_tiles;
    int trace;
    MlpLayout lay;
};

struct __align__(8) Barriers {
    uint64_t raw_full[kRawStages], full[kXStages], empty[kXStages];
    uint64_t d1_full[2], dp_full[2], lo_free, done;
    float gb2_part[4];
    uint32_t tmem_base;
};

// One persistent CTA's share of a network's backward: CTA `cta` of `ncta` takes tiles cta,
// cta + ncta, ... and leaves its float32 partial gradient in row `cta` of a.ws.  Returns the
// (idle) bulk-copy ring for use as scratch by the reduction.
template <int NP>
__device__ __forceinline__ uint8_t* bwd_tc_body(const BwdTcArgs& a, const int cta, const int ncta,
                                                long long* s_trace) {
    extern __shared__ uint8_t smem_raw[];
    // 1024-byte alignment by OFFSETTING the __shared__ array (a round trip through an integer
    // would make every derived pointer generic: LD/ST instead of LDS/STS)
    uint8_t* smem = smem_raw + ((1024u - (tc::smem_u32(smem_raw) & 1023u)) & 1023u);
    uint8_t* w_hi = smem;
    uint8_t* w_lo = w_hi + kWTileBytes;
    uint8_t* x_hi = w_lo + kWTileBytes;               // kXStages tiles, [64 rows][128 B]
    uint8_t* x_lo = x_hi + kXStages * kXTileBytes;
    // transposed tiles: per stage 2 K-chunks (32 batch rows each) x [64 rows][128 B], rows 0-31 =
    // hi of feature n, rows 32-63 = lo of feature n
    uint8_t* xt = x_lo + kXStages * kXTileBytes;
    uint8_t* raw = xt + 2 * kXStages * kXTileBytes;   // kRawStages x 8 KiB
    float* dzs = reinterpret_cast<float*>(raw + kRawStages * kRawStageBytes);  // [kXStages][64][NP]
    float* exch = dzs + kXStages * kRowsT * NP;  // [NP + 1][256]: dW2 / db1 sums of the odd half
    Barriers* bars = reinterpret_cast<Barriers*>(exch + (NP + 1) * 256);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const float* __restrict__ W1 = a.params + a.lay.oW1;
    const float* __restrict__ b1 = a.params + a.lay.ob1;
    const float* __restrict__ W2 = a.params + a.lay.oW2;
    const int O = a.O, H = a.H, ochunks = O >> 2, nblk = H >> 7;
    const int n_my = (a.num_tiles - cta + ncta - 1) / ncta;
    const bool tr = a.trace && blockIdx.x == 0 && lane == 0 && (warp == 0 || warp == 16 || warp == 18);
#define TRACE(tile, ev)                                              \
    if (tr && (tile) < 24) s_trace[(tile) * 16 + (ev)] = clock64();
    if (a.trace && blockIdx.x == 0)
        for (int k = tid; k < 24 * 16; k += kThreads) s_trace[k] = 0;
    TRACE(0, 15)

    // ---- one-time setup.  The mbarriers come first, so that the bulk copies of the first x / dout
    // tiles are already in flight while every thread stages W1'.
    if (warp == 18 && lane == 0) {
        for (int s = 0; s < kRawStages; ++s) tc::mbar_init(&bars->raw_full[s], 1);
        for (int s = 0; s < kXStages; ++s) {
            tc::mbar_init(&bars->full[s], 64);   // every producer thread arrives
            tc::mbar_init(&bars->empty[s], 1);   // tcgen05.commit after UMMA2
        }
        for (int s = 0; s < 2; ++s) {
            tc::mbar_init(&bars->d1_full[s], 1);           // tcgen05.commit after UMMA1
            tc::mbar_init(&bars->dp_full[s], nblk * 256);  // every active epilogue thread
        }
        tc::mbar_init(&bars->lo_free, 1);  // tcgen05.commit after UMMA2
        tc::mbar_init(&bars->done, 1);
        tc::mbar_fence_init();
    }
    __syncthreads();
    // raw ring: stage i % kRawStages <- x rows (and dout rows) of this CTA's i-th tile, full tiles only
    auto issue_raw = [&](int i) {
        const int tile = cta + i * ncta;
        if ((tile + 1) * kRowsT <= a.M) {
            const int rs = i % kRawStages;
            uint8_t* dst = raw + rs * kRawStageBytes;
            const size_t row0 = (size_t)tile * kRowsT;
            const uint32_t bytes_x = kRowsT * O * 4, bytes_z = kRowsT * a.N2 * 4;
            tc::fence_proxy_async();  // earlier generic reads of this stage precede the async write
            tc::mbar_arrive_expect_tx(&bars->raw_full[rs], bytes_x + bytes_z);
            tc::bulk_g2s(dst, a.x + row0 * O, bytes_x, &bars->raw_full[rs]);
            tc::bulk_g2s(dst + kRawDzOffset, a.dout + row0 * a.N2, bytes_z, &bars->raw_full[rs]);
        }
    };
    // the first bulk copies are in flight while the W1' tiles are staged
    if (warp == 16 && lane == 0)
        for (int i = 0; i < n_my && i < kRawStages; ++i) issue_raw(i);
    if (warp == 18) tc::tmem_alloc(&bars->tmem_base, 512);
    tc::stage_w1_tiles(w_hi, w_lo, W1, b1, H, O, tid, kThreads, /*bias_column=*/true);
    tc::fence_proxy_async();
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem_base = bars->tmem_base;

    if (warp < 16) {
        // =============================== epilogue ===============================
        const int hh = warp >> 3, blk = (warp >> 2) & 1, q = warp & 3;  // row half, hidden block, lane quarter
        const int jl = 32 * q + lane, j = 128 * blk + jl;
        // Two batch rows per step in packed fp32 pairs (.x = even row, .y = odd row).
        float2 w2p[NP], gw2p[NP];
#pragma unroll
        for (int n = 0; n < NP; ++n) gw2p[n] = make_float2(0.f, 0.f);
        const uint32_t lane_addr = tmem_base + (static_cast<uint32_t>(32 * q) << 16);
        if (blk < nblk) {
#pragma unroll
            for (int n = 0; n < NP; ++n) {
                const float w = n < a.N2 ? __ldg(W2 + (size_t)n * H + j) : 0.f;
                w2p[n] = make_float2(w, w);
            }
            for (int i = 0; i < n_my; ++i) {
                const int s = i % kXStages, ph = (i / kXStages) & 1;
                const int d1 = i & 1, dph = (i >> 1) & 1;
                const uint32_t c_hi = lane_addr + d1 * 128 + blk * 64 + 32 * hh;   // PRE in, DP_hi out
                const uint32_t c_lo = lane_addr + kColLo + blk * 64 + 32 * hh;
                TRACE(i, 0)
                tc::mbar_wait(&bars->full[s], ph);       // dz rows of this tile are visible
                tc::mbar_wait(&bars->d1_full[d1], dph);  // PRE of this tile is in TMEM
                tc::tc_fence_after();
                TRACE(i, 1)
                const float* dz_half = dzs + (s * kRowsT + 32 * hh) * NP;  // [row pair][n][2]
                // The thread's 32 pre-activations are processed as two halves of 16 columns so that
                // tensor-memory traffic overlaps the math: the second half is in flight while the first
                // is consumed, and DP_hi of the first half is already on its way back while the second
                // is computed (all 16 epilogue warps start a tile together: TMEM reads at 64 B/clk
                // and the math would otherwise simply alternate).
                uint32_t va[16], vb[16], la[16], lb[16];
                auto half = [&](uint32_t (&v)[16], uint32_t (&lo)[16], const int pr0) {
#pragma unroll
                    for (int q2 = 0; q2 < 8; ++q2) {
                        const int pr = pr0 + q2;
                        const float* zp = dz_half + pr * 2 * NP;
                        float2 dz[NP];
                        if constexpr (NP == 4) {
                            const float4 t0 = *reinterpret_cast<const float4*>(zp);
                            const float4 t1 = *reinterpret_cast<const float4*>(zp + 4);
                            dz[0] = make_float2(t0.x, t0.y), dz[1] = make_float2(t0.z, t0.w);
                            dz[2] = make_float2(t1.x, t1.y), dz[3] = make_float2(t1.z, t1.w);
                        } else {
                            dz[0] = *reinterpret_cast<const float2*>(zp);
                        }
                        // relu on the ALU pipe (FMNMX), relu' as a select (FSEL); relu'(0) = 0 as in torch
                        const float2 pre = make_float2(__uint_as_float(v[2 * q2]), __uint_as_float(v[2 * q2 + 1]));
                        const float2 h = make_float2(fmaxf(pre.x, 0.f), fmaxf(pre.y, 0.f));
                        float2 dh = tc::fmul2(dz[0], w2p[0]);
#pragma unroll
                        for (int n = 1; n < NP; ++n) dh = tc::ffma2(dz[n], w2p[n], dh);
#pragma unroll
                        for (int n = 0; n < NP; ++n) gw2p[n] = tc::ffma2(dz[n], h, gw2p[n]);
                        const float2 dp = make_float2(pre.x > 0.f ? dh.x : 0.f, pre.y > 0.f ? dh.y : 0.f);
                        // hi = dp truncated to tf32 (one LOP3; cvt.rna.tf32 is a 4-instruction
                        // sequence on sm_100), lo = the exact remainder < 2^-10 |dp|
                        float2 hi;
                        hi.x = __uint_as_float(__float_as_uint(dp.x) & 0xffffe000u);
                        hi.y = __uint_as_float(__float_as_uint(dp.y) & 0xffffe000u);
                        const float2 l = tc::fsub2(dp, hi);
                        v[2 * q2] = __float_as_uint(hi.x), v[2 * q2 + 1] = __float_as_uint(hi.y);
                        lo[2 * q2] = __float_as_uint(l.x), lo[2 * q2 + 1] = __float_as_uint(l.y);
                    }
                };
                tc::tmem_ld16_nowait(c_hi, va);
                tc::tmem_wait_ld16(va);
                tc::tmem_ld16_nowait(c_hi + 16, vb);  // in flight while the first half is processed
                half(va, la, 0);
                tc::tmem_st16(c_hi, va);              // DP_hi replaces PRE in place
                tc::tmem_wait_ld16(vb);
                half(vb, lb, 8);
                tc::tmem_st16(c_hi + 16, vb);
                TRACE(i, 2)
                tc::mbar_wait(&bars->lo_free, (i & 1) ^ 1);  // UMMA2 of the previous tile retired
                tc::tc_fence_after();
                TRACE(i, 3)
                tc::tmem_st16(c_lo, la);
                tc::tmem_st16(c_lo + 16, lb);
                tc::tmem_wait_st();
                tc::tc_fence_before();
                tc::mbar_arrive(&bars->dp_full[d1]);
                TRACE(i, 4)
            }
            if (hh == 1) {  // hand this half's dW2 sums to the thread that owns the other half
#pragma unroll
                for (int n = 0; n < NP; ++n) exch[(n + 1) * 256 + j] = gw2p[n].x + gw2p[n].y;
            }
        }
        asm volatile("bar.sync 3, 512;" ::: "memory");  // all 16 epilogue warps
        if (blk < nblk && hh == 0) {
            // ---- read out dW1' (TMEM) and write this CTA's partial gradient row
            tc::mbar_wait(&bars->done, 0);
            tc::tc_fence_after();
            float g[32], g2[32];
            tc::tmem_ld32(lane_addr + kColAcc + blk * 64, g);        // dp_hi*x_hi
            tc::tmem_ld32(lane_addr + kColAcc + blk * 64 + 32, g2);  // dp_hi*x_lo + dp_lo*x_hi
#pragma unroll
            for (int k = 0; k < 32; ++k) g[k] += g2[k];
            float* wsb = a.ws + (size_t)cta * a.lay.total;
            float4* wrow = reinterpret_cast<float4*>(wsb + a.lay.oW1 + (size_t)j * O);
            float gb1 = 0.f;
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                if (c < ochunks) wrow[c] = make_float4(g[4 * c], g[4 * c + 1], g[4 * c + 2], g[4 * c + 3]);
                else if (c == ochunks) gb1 = g[4 * c];  // column O of dW1': sum of DP over the rows = db1
            }
            wsb[a.lay.ob1 + j] = gb1;
#pragma unroll
            for (int n = 0; n < NP; ++n)
                if (n < a.N2) wsb[a.lay.oW2 + (size_t)n * H + j] = (gw2p[n].x + gw2p[n].y) + exch[(n + 1) * 256 + j];
        }
        // pads of the partial row (all epilogue threads)
        {
            float* wsb = a.ws + (size_t)cta * a.lay.total;
            const int64_t lo4[4] = {a.lay.oW1 + (int64_t)H * O, a.lay.ob1 + H,
                                    a.lay.oW2 + (int64_t)a.N2 * H, a.lay.ob2 + a.N2};
            const int64_t hi4[4] = {a.lay.ob1, a.lay.oW2, a.lay.ob2, a.lay.total};
            for (int sgm = 0; sgm < 4; ++sgm)
                for (int64_t p = lo4[sgm] + tid; p < hi4[sgm]; p += kEpiThreads) wsb[p] = 0.f;
        }
    } else if (warp < 18) {
        // ===================== producer (2 warps, 32 rows of the tile each) =====================
        const int pw = warp - 16, r = 32 * pw + lane;  // row of the tile this thread converts
        float gb2[NP];  // db2 = column sums of dout: this thread's rows, combined at the end
#pragma unroll
        for (int n = 0; n < NP; ++n) gb2[n] = 0.f;
        auto tile_of = [&](int i) { return cta + i * ncta; };
        auto is_full = [&](int i) { return (tile_of(i) + 1) * kRowsT <= a.M; };
        for (int i = 0; i < n_my; ++i) {
            const int s = i % kXStages, ph = (i / kXStages) & 1;
            const int rs = i % kRawStages, rph = (i / kRawStages) & 1;
            float4 v[8];
            float z[NP];
#pragma unroll
            for (int c = 0; c < 8; ++c) v[c] = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int n = 0; n < NP; ++n) z[n] = 0.f;
            TRACE(i, 5)
            if (is_full(i)) {
                tc::mbar_wait(&bars->raw_full[rs], rph);
                TRACE(i, 6)
                const float4* rx = reinterpret_cast<const float4*>(raw + rs * kRawStageBytes) + r * ochunks;
                const float* rz = reinterpret_cast<const float*>(raw + rs * kRawStageBytes + kRawDzOffset) + r * a.N2;
#pragma unroll
                for (int c = 0; c < 8; ++c)
                    if (c < ochunks) v[c] = rx[c];
#pragma unroll
                for (int n = 0; n < NP; ++n)
                    if (n < a.N2) z[n] = rz[n];
            } else {  // ragged last tile: plain guarded loads
                const int row = tile_of(i) * kRowsT + r;
                if (row < a.M) {
#pragma unroll
                    for (int c = 0; c < 8; ++c)
                        if (c < ochunks) v[c] = __ldg(reinterpret_cast<const float4*>(a.x + (size_t)row * O) + c);
#pragma unroll
                    for (int n = 0; n < NP; ++n)
                        if (n < a.N2) z[n] = __ldg(a.dout + (size_t)row * a.N2 + n);
                }
            }
#pragma unroll
            for (int c = 0; c < 8; ++c)
                if (c == ochunks) v[c].x = 1.f;  // column O of X': multiplies b1 (UMMA1), sums DP into db1 (UMMA2)
            asm volatile("bar.sync 1, 64;" ::: "memory");  // both producer warps drained the raw stage
            if (pw == 0 && lane == 0 && i + kRawStages < n_my) issue_raw(i + kRawStages);
            tc::mbar_wait(&bars->empty[s], ph ^ 1);  // UMMA2 that read this stage has retired
            TRACE(i, 7)
            uint8_t* th = x_hi + s * kXTileBytes;
            uint8_t* tl = x_lo + s * kXTileBytes;
            // transposed tile of K-chunk pw (this warp's 32 batch rows): row = feature (+32 for lo)
            uint8_t* tth = xt + (2 * s + pw) * kXTileBytes + (lane & 3) * 4;
            uint8_t* ttl = tth + 32 * 128;  // rows 32..63 (32 is a multiple of the 8-row swizzle period)
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
                const float hv[4] = {hi.x, hi.y, hi.z, hi.w}, lv[4] = {lo.x, lo.y, lo.z, lo.w};
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const uint32_t toff = tc::sw128_offset(4 * c + e, lane >> 2);
                    *reinterpret_cast<float*>(tth + toff) = hv[e];
                    *reinterpret_cast<float*>(ttl + toff) = lv[e];
                }
            }
#pragma unroll
            for (int n = 0; n < NP; ++n) {  // [row pair][n][2]: the epilogue reads pairs of rows
                dzs[((s * (kRowsT / 2) + (r >> 1)) * NP + n) * 2 + (r & 1)] = z[n];
                gb2[n] += z[n];
            }
            tc::fence_proxy_async();
            tc::mbar_arrive(&bars->full[s]);
            TRACE(i, 8)
        }
        // db2: fixed-order tree over the 64 producer threads
#pragma unroll
        for (int n = 0; n < NP; ++n) {
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) gb2[n] += __shfl_xor_sync(0xffffffffu, gb2[n], off);
        }
        if (pw == 1 && lane == 0) {
#pragma unroll
            for (int n = 0; n < NP; ++n) bars->gb2_part[n] = gb2[n];
        }
        asm volatile("bar.sync 1, 64;" ::: "memory");
        if (pw == 0 && lane == 0) {
            float* wsb = a.ws + (size_t)cta * a.lay.total;
#pragma unroll
            for (int n = 0; n < NP; ++n)
                if (n < a.N2) wsb[a.lay.ob2 + n] = gb2[n] + bars->gb2_part[n];
        }
    } else {
        // =============================== UMMA issuer ===============================
        // The whole warp runs the schedule (warp-uniform descriptors stay in uniform registers);
        // one elected lane issues the UMMAs and their commits.  UMMAs execute in issue order, so
        // UMMA1(i+2) overwriting the PRE/DP_hi buffer that UMMA2(i) reads needs no extra barrier.
        const uint32_t idesc1 = tc::instr_desc_tf32_m128(kRowsT);  // N = 64 batch rows
        const uint32_t idesc2w = tc::instr_desc_tf32_m128(2 * kKPad);  // N = 64: [hi | lo] features
        const uint32_t idesc2 = tc::instr_desc_tf32_m128(kKPad);       // N = 32: hi features
        const int ksteps1 = (O + 1 + 7) >> 3;  // K' columns in use: O features + the bias column
        const uint64_t dw_hi = tc::smem_desc_k_sw128(w_hi, 0), dw_lo = tc::smem_desc_k_sw128(w_lo, 0);
        const uint64_t dx_hi = tc::smem_desc_k_sw128(x_hi, 0), dx_lo = tc::smem_desc_k_sw128(x_lo, 0);
        const uint64_t dxt = tc::smem_desc_k_sw128(xt, 0);
        constexpr uint64_t kBlkOff = (128 * 128) >> 4;  // next 128-row block of the W1' tile
        auto issue_umma1 = [&](int i) {
            const int s = i % kXStages, ph = (i / kXStages) & 1, d1 = i & 1;
            TRACE(i, 9)
            tc::mbar_wait(&bars->full[s], ph);
            tc::tc_fence_after();
            TRACE(i, 10)
            if (tc::elect_one()) {
                // fully unrolled with uniform guards: descriptor arithmetic folds to constants
                // off two per-tile bases (the rolled loop spent ~12 issue slots per UMMA)
                const uint64_t xh = dx_hi + static_cast<uint64_t>((s * kXTileBytes) >> 4);
                const uint64_t xl = dx_lo + static_cast<uint64_t>((s * kXTileBytes) >> 4);
                const uint32_t d0 = tmem_base + d1 * 128;
#pragma unroll
                for (int b = 0; b < 2; ++b) {
                    if (b < nblk) {
                        // correction terms first, hi*hi last: the accumulator addition truncates (mlp_fwd_tc.cu)
#pragma unroll
                        for (int kk = 0; kk < 4; ++kk) {
                            if (kk < ksteps1) {
                                const uint64_t ko = 2 * kk, bo = b * kBlkOff;
                                tc::umma_tf32(d0 + b * 64, dw_lo + bo + ko, xh + ko, idesc1, kk > 0);
                                tc::umma_tf32(d0 + b * 64, dw_hi + bo + ko, xl + ko, idesc1, true);
                            }
                        }
#pragma unroll
                        for (int kk = 0; kk < 4; ++kk)
                            if (kk < ksteps1) tc::umma_tf32(d0 + b * 64, dw_hi + b * kBlkOff + 2 * kk, xh + 2 * kk, idesc1, true);
                    }
                }
                tc::umma_commit(&bars->d1_full[d1]);
            }
            __syncwarp();
            TRACE(i, 11)
        };
        if (n_my > 0) issue_umma1(0);
        if (n_my > 1) issue_umma1(1);
        for (int i = 0; i < n_my; ++i) {
            const int s = i % kXStages, d1 = i & 1;
            tc::mbar_wait(&bars->dp_full[d1], (i >> 1) & 1);  // DP hi/lo of tile i are in TMEM
            tc::tc_fence_after();
            TRACE(i, 12)
            if (tc::elect_one()) {
                const uint64_t xts = dxt + static_cast<uint64_t>((2 * s * kXTileBytes) >> 4);
                const uint32_t a_hi0 = tmem_base + d1 * 128, a_lo0 = tmem_base + kColLo, acc0 = tmem_base + kColAcc;
                const uint32_t first = i > 0;
#pragma unroll
                for (int b = 0; b < 2; ++b) {
                    if (b < nblk) {
#pragma unroll
                        for (int kk = 0; kk < kRowsT / 8; ++kk) {  // K = 64 batch rows, 8 per step
                            // x^T: K-chunk kk/4 of this stage (8 KiB each), 32 bytes per step inside it
                            constexpr int kChunk16 = kXTileBytes >> 4;
                            const uint64_t ko = static_cast<uint64_t>((kk >> 2) * kChunk16 + (kk & 3) * 2);
                            // columns [0,32) collect dp_hi*x_hi only; both correction terms share [32,64)
                            tc::umma_tf32_ts(acc0 + b * 64, a_hi0 + b * 64 + 8 * kk, xts + ko, idesc2w, first | (kk > 0));
                            tc::umma_tf32_ts(acc0 + b * 64 + 32, a_lo0 + b * 64 + 8 * kk, xts + ko, idesc2, true);
                        }
                    }
                }
                tc::umma_commit(&bars->lo_free);   // DP_lo region reusable
                tc::umma_commit(&bars->empty[s]);  // x / x^T / dz stage reusable
            }
            __syncwarp();
            TRACE(i, 13)
            if (i + 2 < n_my) issue_umma1(i + 2);
        }
        if (tc::elect_one()) tc::umma_commit(&bars->done);
        __syncwarp();
    }

    tc::tc_fence_before();
    __threadfence();  // this thread's partial-row stores are visible device-wide
    __syncthreads();
    if (warp == 18) {
        tc::tc_fence_after();
        tc::tmem_dealloc(tmem_base, 512);
    }
#undef TRACE
    return raw;
}

// Grid barrier: every CTA of the launch is resident (grid <= SM count, one CTA per SM, COOPERATIVE
// launch - it fails instead of hanging where co-residency cannot be had).  ctl[0] counts arrivals; a
// workspace that was not zero-filled once traps instead of hanging.
__device__ __forceinline__ void grid_arrive_and_wait(unsigned int* ctl) {
    if (threadIdx.x == 0) {
        atomicAdd(ctl, 1u);
        const long long t0 = clock64();
        unsigned int seen;
        do {
            asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(ctl) : "memory");
            if (seen != gridDim.x && clock64() - t0 > (1ll << 32)) __trap();
        } while (seen != gridDim.x);
    }
    __syncthreads();
}

// The last CTA out re-arms the barrier for the next launch.
__device__ __forceinline__ void grid_depart(unsigned int* ctl) {
    if (threadIdx.x == 0 && atomicAdd(ctl + 1, 1u) == gridDim.x - 1) {
        ctl[0] = 0u;
        ctl[1] = 0u;
    }
}

// Deterministic float64 sum of `nparts` partial rows: chunk c = entries [64c, 64c + 64); this CTA
// takes chunks first, first + stride, ...; warp w adds rows w, w + kWarps, ... and warp 0 combines.
// `push`: the sums go to entry push_off + e of slot `rank` in every rank's gather buffer instead of
// a.grad (posted, step-tagged peer stores; the all-reduce of the data-parallel learner starts here).
__device__ __forceinline__ void reduce_rows(const BwdTcArgs& a, const int nparts, const int first,
                                            const int stride, double* s_red, const PushArgs* push = nullptr,
                                            const int64_t push_off = 0) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t total = a.lay.total;  // multiple of 32
    const int nchunks = (int)((total + 63) >> 6);
    for (int c = first; c < nchunks; c += stride) {
        const int64_t e0 = (int64_t)c * 64 + 2 * lane;
        double sx = 0.0, sy = 0.0;
        if (e0 < total) {
            const float* col = a.ws + e0;
            int p = warp;
            for (; p + 3 * kWarps < nparts; p += 4 * kWarps) {
                const float2 v0 = __ldcg(reinterpret_cast<const float2*>(col + (size_t)p * total));
                const float2 v1 = __ldcg(reinterpret_cast<const float2*>(col + (size_t)(p + kWarps) * total));
                const float2 v2 = __ldcg(reinterpret_cast<const float2*>(col + (size_t)(p + 2 * kWarps) * total));
                const float2 v3 = __ldcg(reinterpret_cast<const float2*>(col + (size_t)(p + 3 * kWarps) * total));
                sx += v0.x, sy += v0.y, sx += v1.x, sy += v1.y;
                sx += v2.x, sy += v2.y, sx += v3.x, sy += v3.y;
            }
            for (; p < nparts; p += kWarps) {
                const float2 v0 = __ldcg(reinterpret_cast<const float2*>(col + (size_t)p * total));
                sx += v0.x, sy += v0.y;
            }
        }
        s_red[warp * 64 + 2 * lane] = sx;
        s_red[warp * 64 + 2 * lane + 1] = sy;
        __syncthreads();
        if (push) {
            // Warp r sends the chunk to rank r: lane l carries entries l and l + 32, so each store
            // instruction covers 512 contiguous bytes of the peer's slot (4 full 128-byte lines).
            // Remote stores are credit-limited per SM - with 16-byte scattered requests from a single
            // warp this tail cost 12 us at 8 GPUs.  Same summation order as below: every rank (and
            // the single-GPU path) forms bit-identical values.
            if (warp < push->world) {
                const int64_t ea = (int64_t)c * 64 + lane, eb = ea + 32;
                double va = 0.0, vb = 0.0;
#pragma unroll
                for (int w = 0; w < kWarps; ++w) va += s_red[w * 64 + lane], vb += s_red[w * 64 + 32 + lane];
                const long long step = *push->seq + 1;
                ulonglong2* dst = push->gather[warp] + (step & 1) * push->buf_stride +
                                  (int64_t)push->rank * push->slot_stride + push_off;
                if (ea < total) ll_store(dst + ea, va, (unsigned)step);
                if (eb < total) ll_store(dst + eb, vb, (unsigned)step);
            }
        } else if (warp == 0 && e0 < total) {
            double tx = 0.0, ty = 0.0;
#pragma unroll
            for (int w = 0; w < kWarps; ++w) tx += s_red[w * 64 + 2 * lane], ty += s_red[w * 64 + 2 * lane + 1];
            *reinterpret_cast<double2*>(a.grad + e0) = make_double2(tx, ty);
        }
        __syncthreads();
    }
}

__device__ __forceinline__ void dump_trace(const BwdTcArgs& a, long long* s_trace, long long t_barrier) {
    if (a.trace && blockIdx.x == 0) {
        if (threadIdx.x == 0) s_trace[1 * 16 + 15] = clock64(), s_trace[2 * 16 + 15] = t_barrier;
        __syncthreads();
        for (int k = threadIdx.x; k < 24 * 16; k += kThreads) g_trace[k] = s_trace[k];
    }
}

template <int NP>
__global__ void __launch_bounds__(kThreads, 1) mlp_bwd_tc_kernel(const __grid_constant__ BwdTcArgs a) {
    __shared__ long long s_trace[24 * 16];
    uint8_t* scratch = bwd_tc_body<NP>(a, blockIdx.x, gridDim.x, s_trace);
    grid_arrive_and_wait(a.ctl);
    const long long t_barrier = clock64();
    reduce_rows(a, gridDim.x, blockIdx.x, gridDim.x, reinterpret_cast<double*>(scratch));
    grid_depart(a.ctl);
    dump_trace(a, s_trace, t_barrier);
}

// Policy and value network of one learner step in ONE launch: CTAs [0, n_pi) take the policy's
// tiles (partial rows 0 .. n_pi of its workspace), the rest the value function's.  After the grid
// barrier every CTA helps reduce both sets of rows (the value function's chunks are dealt from
// the far end so that no CTA gets two chunks of each).  Uses the policy workspace's control words.
// PUSH: data-parallel learner - the reduced gradient [policy | value fn] and `n_extra` local
// scalars (the loss sums the V-trace kernel left at `extra`) go straight into every rank's gather
// buffer as step-tagged LL elements (protocol in optim.cu); nothing is written to a.grad.
template <bool PUSH>
__global__ void __launch_bounds__(kThreads, 1)
mlp_bwd_tc_pair_kernel(const __grid_constant__ BwdTcArgs a_pi, const __grid_constant__ BwdTcArgs a_vf,
                       const int n_pi, const __grid_constant__ PushArgs push, const double* extra,
                       const int n_extra) {
    __shared__ long long s_trace[24 * 16];
    const int n_vf = (int)gridDim.x - n_pi;
    uint8_t* scratch;
    if ((int)blockIdx.x < n_pi) scratch = bwd_tc_body<4>(a_pi, blockIdx.x, n_pi, s_trace);
    else scratch = bwd_tc_body<1>(a_vf, (int)blockIdx.x - n_pi, n_vf, s_trace);
    grid_arrive_and_wait(a_pi.ctl);
    const long long t_barrier = clock64();
    const PushArgs* pp = PUSH ? &push : nullptr;
    reduce_rows(a_pi, n_pi, blockIdx.x, gridDim.x, reinterpret_cast<double*>(scratch), pp, 0);
    reduce_rows(a_vf, n_vf, (int)gridDim.x - 1 - (int)blockIdx.x, gridDim.x, reinterpret_cast<double*>(scratch), pp,
                a_pi.lay.total);
    if (PUSH && blockIdx.x == gridDim.x / 2 && (int)threadIdx.x < n_extra) {
        const long long step = *push.seq + 1;
        const int64_t off = (step & 1) * push.buf_stride + (int64_t)push.rank * push.slot_stride + a_pi.lay.total +
                            a_vf.lay.total + threadIdx.x;
        const double val = extra[threadIdx.x];
        for (int r = 0; r < push.world; ++r) ll_store(push.gather[r] + off, val, (unsigned)step);
    }
    grid_depart(a_pi.ctl);
    dump_trace(a_pi, s_trace, t_barrier);
}

constexpr size_t kSmemBytes = 1024 + 2 * kWTileBytes + 4 * kXStages * kXTileBytes +  // x hi/lo + x^T (2 chunks)
                              kRawStages * kRawStageBytes + kXStages * kRowsT * 4 * sizeof(float) +
                              5 * 256 * sizeof(float) + sizeof(Barriers);

}  // namespace

bool impala_mlp_bwd_tc_eligible(const float* x, const float* dout, int M, int O, int H, int N2) {
    return M >= 1 && O >= 4 && O <= 28 && (O & 3) == 0 && (H == 128 || H == 256) && N2 >= 1 &&
           N2 <= 4 && (reinterpret_cast<uintptr_t>(x) & 15) == 0 &&
           (reinterpret_cast<uintptr_t>(dout) & 15) == 0;
}

namespace {
BwdTcArgs make_bwd_args(const float* x, const float* params, const float* dout, float* ws, double* grad,
                        unsigned int* ctl, int M, int O, int H, int N2) {
    BwdTcArgs a{};
    a.x = x, a.params = params, a.dout = dout, a.ws = ws, a.grad = grad, a.ctl = ctl;
    a.M = M, a.O = O, a.H = H, a.N2 = N2;
    a.num_tiles = (M + kRowsT - 1) / kRowsT;
    a.lay = impala_make_layout(O, H, N2);
    const char* tr_env = std::getenv("IMPALA_TC_TRACE");
    a.trace = tr_env && tr_env[0] == '1';
    return a;
}
}  // namespace

// Per-CTA partial gradient rows go to ws (same layout as the FP32 kernel), their float64 sum to
// grad; ctl = two zeroed control words (see the grid barrier in the kernel).
int impala_mlp_bwd_tc(const float* x, const float* params, const float* dout, float* ws,
                      double* grad, unsigned int* ctl, int M, int O, int H, int N2, cudaStream_t st) {
    const BwdTcArgs a = make_bwd_args(x, params, dout, ws, grad, ctl, M, O, H, N2);
    static bool opted[64][2] = {};  // per device
    cudaError_t e;
    int sms = 0, dev = 0;
    if ((e = impala_sm_count(&sms)) != cudaSuccess) return (int)e;
    if ((e = cudaGetDevice(&dev)) != cudaSuccess) return (int)e;
    const int which = N2 == 1 ? 0 : 1;
    auto kernel = which ? mlp_bwd_tc_kernel<4> : mlp_bwd_tc_kernel<1>;
    if (dev < 0 || dev >= 64 || !opted[dev][which]) {
        e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemBytes);
        if (e != cudaSuccess) return (int)e;
        if (dev >= 0 && dev < 64) opted[dev][which] = true;
    }
    int grid = a.num_tiles < sms ? a.num_tiles : sms;  // <= SM count: the grid barrier needs residency
    if (grid > kMaxParts) grid = kMaxParts;
    if ((e = impala_launch_cooperative(kernel, grid, kThreads, kSmemBytes, st, a)) != cudaSuccess) return (int)e;
    return impala_launch_status();
}

// Both networks in one launch; the caller has checked eligibility of each and 2 <= A <= 4.
// push != nullptr: data-parallel variant (see mlp_bwd_tc_pair_kernel).
int impala_mlp_bwd_tc_pair(const float* x, const float* params_pi, const float* params_vf,
                           const float* dlogits, const float* dv, float* ws_pi, float* ws_vf,
                           double* grad_pi, double* grad_vf, unsigned int* ctl, int M_pi, int M_vf, int O,
                           int H_pi, int H_vf, int A, cudaStream_t st, const PushArgs* push, const double* extra,
                           int n_extra) {
    const BwdTcArgs a_pi = make_bwd_args(x, params_pi, dlogits, ws_pi, grad_pi, ctl, M_pi, O, H_pi, A);
    const BwdTcArgs a_vf = make_bwd_args(x, params_vf, dv, ws_vf, grad_vf, ctl, M_vf, O, H_vf, 1);
    static bool opted[64][2] = {};  // per device, per variant
    cudaError_t e;
    int sms = 0, dev = 0;
    if ((e = impala_sm_count(&sms)) != cudaSuccess) return (int)e;
    if ((e = cudaGetDevice(&dev)) != cudaSuccess) return (int)e;
    const int var = push ? 1 : 0;
    if (dev < 0 || dev >= 64 || !opted[dev][var]) {
        e = push ? cudaFuncSetAttribute(mlp_bwd_tc_pair_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemBytes)
                 : cudaFuncSetAttribute(mlp_bwd_tc_pair_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemBytes);
        if (e != cudaSuccess) return (int)e;
        if (dev >= 0 && dev < 64) opted[dev][var] = true;
    }
    const int total_tiles = a_pi.num_tiles + a_vf.num_tiles;
    int grid = total_tiles < sms ? total_tiles : sms;
    if (grid > kMaxParts) grid = kMaxParts;
    if (grid < 2) return IMPALA_ERR_UNSUPPORTED_SHAPE;
    // per-tile cost of a policy tile in % of a value-function tile, per 128 hidden units: measured on a B200 (c4)
    constexpr int kPairCostBwd = 105;
    const int n_pi = impala_pair_split(a_pi.num_tiles, a_vf.num_tiles, grid,
                                       kPairCostBwd * (H_pi / 128),
                                       100 * (H_vf / 128));
    // cooperative launch: the in-kernel grid barrier needs every CTA resident (ADVICE r1)
    e = push ? impala_launch_cooperative(mlp_bwd_tc_pair_kernel<true>, grid, kThreads, kSmemBytes, st, a_pi, a_vf, n_pi,
                                         *push, extra, n_extra)
             : impala_launch_cooperative(mlp_bwd_tc_pair_kernel<false>, grid, kThreads, kSmemBytes, st, a_pi, a_vf, n_pi,
                                         PushArgs{}, (const double*)nullptr, 0);
    if (e != cudaSuccess) return (int)e;
    return impala_launch_status();
}

// Debug only: the [24 tiles][16 events] clock stamps of the last traced launch (CTA 0).
extern "C" int impala_debug_read_trace(long long* out, int n) {
    cudaDeviceSynchronize();
    if (n > 24 * 16) n = 24 * 16;
    if (cudaMemcpyFromSymbol(out, g_trace, sizeof(long long) * n) != cudaSuccess) return -1;
    return n;
}
