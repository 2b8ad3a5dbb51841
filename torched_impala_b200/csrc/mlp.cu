// Two-layer MLP forward / backward on FP32 CUDA cores (reference models.py:12-25,40-52
// in eval mode; autograd of the same at learner.py:175).
//
// Mapping ("a thread owns hidden units"): thread `tid` owns hidden units
// j = tid + q*blockDim (q < JPT) and keeps their W1 rows, b1 and W2 columns in registers
// for the lifetime of its persistent CTA.  A tile is 32 consecutive rows of the flattened
// (M, O) observation matrix, staged in shared memory and consumed in register blocks of 8
// rows through warp-broadcast 128-bit loads (8*JPT FFMA per LDS.128).  Hidden activations
// never leave registers: the forward reduces layer 2 across the CTA with a transposing
// warp butterfly (the CTA spans the whole hidden layer); the backward recomputes them,
// and because every gradient entry of W1/b1/W2 belongs to exactly one hidden unit each
// thread accumulates its own slice in registers across all its tiles - no atomics,
// deterministic; wide hidden layers are split over blockIdx.y.  Per-CTA partials are then
// summed in float64 by a second small kernel.
//
// This file: host-side configuration, occupancy cache, the partial reduction and the
// C-ABI entry points.  Kernel templates: mlp_kernels.cuh; instantiations: mlp_inst.cu.
#include <cstdlib>
#include <map>
#include <mutex>
#include <tuple>

#include "mlp_kernels.cuh"

namespace {

struct GridInfo {
    int ctas_per_sm, sms;
};
std::mutex g_cfg_mutex;
std::map<std::tuple<const void*, int, int, size_t>, GridInfo> g_cfg_cache;
// cudaFuncAttributeMaxDynamicSharedMemorySize is a property of the KERNEL (per device), not of one launch
// configuration: it is only ever raised.  (Setting it per (threads, smem) entry lowered it when the same
// instantiation was used with a narrower hidden layer, and the next launch of the wider, already
// cached configuration failed with cudaErrorInvalidValue.)
std::map<std::pair<const void*, int>, size_t> g_smem_opt_in;

// grad[i] = sum_c ws[c][i] in float64.  A CTA covers 32 consecutive entries (one 128-byte
// line per partial row); its 8 warps split the partial rows, so every load instruction is
// one fully coalesced line and 8 x 4 loads are in flight per entry.  Fixed summation
// order -> bitwise reproducible gradients.
constexpr int kRedWarps = 8;
constexpr int64_t kWsHeader = 256;  // control words of the tensor-core backward's grid barrier
__global__ void __launch_bounds__(kRedWarps * 32)
reduce_partials_kernel(const float* __restrict__ ws, double* __restrict__ grad, int nparts,
                       int64_t total) {
    __shared__ double s_sum[kRedWarps][33];
    const int lane = threadIdx.x & 31, g = threadIdx.x >> 5;
    const int64_t i = (int64_t)blockIdx.x * 32 + lane;
    double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
    if (i < total) {
        int c = g;
        for (; c + 3 * kRedWarps < nparts; c += 4 * kRedWarps) {
            const float a0 = __ldg(ws + (size_t)c * total + i);
            const float a1 = __ldg(ws + (size_t)(c + kRedWarps) * total + i);
            const float a2 = __ldg(ws + (size_t)(c + 2 * kRedWarps) * total + i);
            const float a3 = __ldg(ws + (size_t)(c + 3 * kRedWarps) * total + i);
            s0 += a0, s1 += a1, s2 += a2, s3 += a3;
        }
        for (; c < nparts; c += kRedWarps) s0 += __ldg(ws + (size_t)c * total + i);
    }
    s_sum[g][lane] = (s0 + s1) + (s2 + s3);
    __syncthreads();
    if (g == 0 && i < total) {
        double s = 0.0;
#pragma unroll
        for (int w = 0; w < kRedWarps; ++w) s += s_sum[w][lane];
        grad[i] = s;
    }
}

bool pick_config(int O, int H, int N2, bool bwd, MlpConfig* c) {
    if (O < 1 || H < 1 || N2 < 1) return false;
    if (O <= 8) c->op = 8;
    else if (O <= 24) c->op = 24;
    else if (O <= 32) c->op = 32;
    else if (O <= 64) c->op = 64;
    else return false;
    if (N2 <= 1) c->np = 1;
    else if (N2 <= 4) c->np = 4;
    else if (N2 <= 16) c->np = 16;
    else return false;
    // register budget: forward holds JPT*OP weights, backward 2*JPT*OP (weights + gradient); at OP = 64
    // the backward splits the features of a hidden unit over a lane pair (ks = 2: 2 x 32 + 2 x 32)
    c->ks = (bwd && c->op == 64) ? 2 : 1;
    if (H < 128 || (bwd && c->op == 64)) c->jpt = 1, c->maxt = bwd && H >= 128 ? 256 : 128;
    else c->jpt = 2, c->maxt = 256;
    const int want = (int)impala_round_up((int64_t)c->ks * ((H + c->jpt - 1) / c->jpt), 32);
    if (bwd) {
        c->threads = want < c->maxt ? want : c->maxt;
        const int units = c->threads / c->ks * c->jpt;  // hidden units per CTA
        c->slices = (H + units - 1) / units;
    } else {
        if (want > c->maxt) return false;  // forward needs the whole hidden layer in one CTA
        c->threads = want;
        c->slices = 1;
    }
    return true;
}

bool fill_args(MlpArgs* a, MlpConfig* c, size_t* smem, bool bwd, int M, int O, int H, int N2) {
    if (M < 1 || !pick_config(O, H, N2, bwd, c)) return false;
    a->M = M, a->O = O, a->H = H, a->N2 = N2;
    a->num_tiles = (M + kRows - 1) / kRows;
    a->lay = impala_make_layout(O, H, N2);
    const size_t tail = bwd ? (size_t)kRows * c->np : (size_t)(c->threads / 32) * kRows * c->np;
    *smem = ((size_t)kRows * c->op + tail) * sizeof(float);
    return true;
}

int dispatch(bool bwd, const MlpArgs& a, const MlpConfig& c, size_t smem, cudaStream_t st,
             int* grid) {
    switch (c.op) {
        case 8: return bwd ? impala_mlp_bwd_op8(a, c, smem, st, grid) : impala_mlp_fwd_op8(a, c, smem, st, grid);
        case 24: return bwd ? impala_mlp_bwd_op24(a, c, smem, st, grid) : impala_mlp_fwd_op24(a, c, smem, st, grid);
        case 32: return bwd ? impala_mlp_bwd_op32(a, c, smem, st, grid) : impala_mlp_fwd_op32(a, c, smem, st, grid);
        default: return bwd ? impala_mlp_bwd_op64(a, c, smem, st, grid) : impala_mlp_fwd_op64(a, c, smem, st, grid);
    }
}

}  // namespace

// Persistent grid = resident CTAs per SM x SM count, computed once per
// (kernel, device, block size, shared memory) and cached.
int impala_mlp_launch(void (*kernel)(MlpArgs), const MlpArgs& a, const MlpConfig& c, size_t smem,
                      cudaStream_t st, int* grid_out) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return (int)e;
    GridInfo gi;
    {
        std::lock_guard<std::mutex> lock(g_cfg_mutex);
        const auto key = std::make_tuple((const void*)kernel, dev, c.threads, smem);
        auto it = g_cfg_cache.find(key);
        if (it == g_cfg_cache.end()) {
            size_t& opted = g_smem_opt_in[std::make_pair((const void*)kernel, dev)];
            if (smem > opted) {
                e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
                if (e != cudaSuccess) return (int)e;
                opted = smem;
            }
            e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&gi.ctas_per_sm, kernel, c.threads, smem);
            if (e != cudaSuccess) return (int)e;
            e = cudaDeviceGetAttribute(&gi.sms, cudaDevAttrMultiProcessorCount, dev);
            if (e != cudaSuccess) return (int)e;
            if (gi.ctas_per_sm < 1) return IMPALA_ERR_UNSUPPORTED_SHAPE;
            g_cfg_cache[key] = gi;
        } else {
            gi = it->second;
        }
    }
    int grid = gi.ctas_per_sm * gi.sms / c.slices;
    if (grid < 1) grid = 1;
    if (grid > a.num_tiles) grid = a.num_tiles;
    if (grid > kMaxParts) grid = kMaxParts;
    kernel<<<dim3(grid, c.slices), c.threads, smem, st>>>(a);
    *grid_out = grid;
    return impala_launch_status();
}

// GEMM-shaped layers go to the tensor cores (IMPALA_MLP_TC=0 forces the FP32 kernels).
static bool tc_enabled() {
    const char* tc_env = std::getenv("IMPALA_MLP_TC");
    return !(tc_env && tc_env[0] == '0');
}

extern "C" int impala_mlp_forward(const float* x, const float* params, float* out, int M, int O,
                                  int H, int N2, void* stream) {
    if (!x || !params || !out) return IMPALA_ERR_BAD_ARG;
    if (tc_enabled() && impala_mlp_fwd_tc_eligible(x, M, O, H, N2))
        return impala_mlp_fwd_tc(x, params, out, M, O, H, N2, (cudaStream_t)stream);
    if (tc_enabled() && impala_mlp_tcw_eligible(x, M, O, H, N2))
        return impala_mlp_fwd_tcw(x, params, out, M, O, H, N2, (cudaStream_t)stream);
    MlpArgs a{};
    MlpConfig c{};
    size_t smem;
    if (!fill_args(&a, &c, &smem, false, M, O, H, N2)) return IMPALA_ERR_UNSUPPORTED_SHAPE;
    a.x = x, a.params = params, a.out = out;
    int grid = 0;
    return dispatch(false, a, c, smem, (cudaStream_t)stream, &grid);
}

extern "C" int impala_mlp_forward_pair(const float* x, const float* params_pi, const float* params_vf,
                                       float* logits, float* values, int M_pi, int M_vf, int O,
                                       int H_pi, int H_vf, int A, void* stream) {
    if (!x || !params_pi || !params_vf || !logits || !values) return IMPALA_ERR_BAD_ARG;
    if (tc_enabled() && A >= 2 && A <= 4 && impala_mlp_fwd_tc_eligible(x, M_pi, O, H_pi, A) &&
        impala_mlp_fwd_tc_eligible(x, M_vf, O, H_vf, 1))
        return impala_mlp_fwd_tc_pair(x, params_pi, params_vf, logits, values, M_pi, M_vf, O, H_pi, H_vf, A,
                                      (cudaStream_t)stream);
    const int rc = impala_mlp_forward(x, params_pi, logits, M_pi, O, H_pi, A, stream);
    if (rc != IMPALA_OK) return rc;
    return impala_mlp_forward(x, params_vf, values, M_vf, O, H_vf, 1, stream);
}

extern "C" int64_t impala_mlp_backward_workspace(int M, int O, int H, int N2) {
    MlpConfig c{};
    if (M < 1 || !pick_config(O, H, N2, true, &c)) return IMPALA_ERR_UNSUPPORTED_SHAPE;
    int64_t tiles = (M + kRows - 1) / kRows;
    if (tiles > kMaxParts) tiles = kMaxParts;
    return kWsHeader + tiles * impala_make_layout(O, H, N2).total * (int64_t)sizeof(float);
}

extern "C" int impala_mlp_backward(const float* x, const float* params, const float* dout,
                                   double* grad, void* workspace, int64_t workspace_bytes, int M,
                                   int O, int H, int N2, void* stream) {
    if (!x || !params || !dout || !grad || !workspace) return IMPALA_ERR_BAD_ARG;
    MlpArgs a{};
    MlpConfig c{};
    size_t smem;
    if (!fill_args(&a, &c, &smem, true, M, O, H, N2)) return IMPALA_ERR_UNSUPPORTED_SHAPE;
    if (workspace_bytes < impala_mlp_backward_workspace(M, O, H, N2))
        return IMPALA_ERR_WORKSPACE_TOO_SMALL;
    // workspace = [control words (kWsHeader bytes, zero-filled once by the caller) | partial rows]
    a.x = x, a.params = params, a.dout = dout;
    a.ws = reinterpret_cast<float*>(static_cast<char*>(workspace) + kWsHeader);
    int grid = 0;
    if (tc_enabled() && impala_mlp_bwd_tc_eligible(x, dout, M, O, H, N2) &&
        (reinterpret_cast<uintptr_t>(grad) & 15) == 0)
        return impala_mlp_bwd_tc(x, params, dout, a.ws, grad, static_cast<unsigned int*>(workspace), M, O, H,
                                 N2, (cudaStream_t)stream);  // reduces in-kernel
    const bool wide = tc_enabled() && impala_mlp_tcw_eligible(x, M, O, H, N2);
    const int rc = wide ? impala_mlp_bwd_tcw(x, params, dout, a.ws, M, O, H, N2, (cudaStream_t)stream, &grid)
                        : dispatch(true, a, c, smem, (cudaStream_t)stream, &grid);
    if (rc != IMPALA_OK) return rc;
    const int64_t total = a.lay.total;
    reduce_partials_kernel<<<(unsigned)((total + 31) / 32), kRedWarps * 32, 0,
                             (cudaStream_t)stream>>>(a.ws, grad, grid, total);
    return impala_launch_status();
}

extern "C" int impala_mlp_backward_pair(const float* x, const float* params_pi, const float* params_vf,
                                        const float* dlogits, const float* dv, double* grad_pi,
                                        double* grad_vf, void* workspace_pi, int64_t workspace_pi_bytes,
                                        void* workspace_vf, int64_t workspace_vf_bytes, int M_pi, int M_vf,
                                        int O, int H_pi, int H_vf, int A, void* stream) {
    if (!x || !params_pi || !params_vf || !dlogits || !dv || !grad_pi || !grad_vf || !workspace_pi ||
        !workspace_vf)
        return IMPALA_ERR_BAD_ARG;
    if (tc_enabled() && A >= 2 && A <= 4 && impala_mlp_bwd_tc_eligible(x, dlogits, M_pi, O, H_pi, A) &&
        impala_mlp_bwd_tc_eligible(x, dv, M_vf, O, H_vf, 1) &&
        ((reinterpret_cast<uintptr_t>(grad_pi) | reinterpret_cast<uintptr_t>(grad_vf)) & 15) == 0) {
        const int64_t need_pi = impala_mlp_backward_workspace(M_pi, O, H_pi, A);
        const int64_t need_vf = impala_mlp_backward_workspace(M_vf, O, H_vf, 1);
        if (need_pi < 0 || need_vf < 0) return IMPALA_ERR_UNSUPPORTED_SHAPE;
        if (workspace_pi_bytes < need_pi || workspace_vf_bytes < need_vf) return IMPALA_ERR_WORKSPACE_TOO_SMALL;
        return impala_mlp_bwd_tc_pair(
            x, params_pi, params_vf, dlogits, dv,
            reinterpret_cast<float*>(static_cast<char*>(workspace_pi) + kWsHeader),
            reinterpret_cast<float*>(static_cast<char*>(workspace_vf) + kWsHeader), grad_pi, grad_vf,
            static_cast<unsigned int*>(workspace_pi), M_pi, M_vf, O, H_pi, H_vf, A, (cudaStream_t)stream);
    }
    const int rc = impala_mlp_backward(x, params_pi, dlogits, grad_pi, workspace_pi, workspace_pi_bytes, M_pi,
                                       O, H_pi, A, stream);
    if (rc != IMPALA_OK) return rc;
    return impala_mlp_backward(x, params_vf, dv, grad_vf, workspace_vf, workspace_vf_bytes, M_vf, O, H_vf, 1,
                               stream);
}

// ---- data-parallel learner: the paired backward that pushes its result to the peers (optim.cu)
extern "C" int impala_mlp_backward_pair_push_supported(int M_pi, int M_vf, int O, int H_pi, int H_vf, int A) {
    alignas(16) static const float probe[4] = {0.f, 0.f, 0.f, 0.f};  // alignment stand-in for the data pointers
    return tc_enabled() && A >= 2 && A <= 4 && impala_mlp_bwd_tc_eligible(probe, probe, M_pi, O, H_pi, A) &&
           impala_mlp_bwd_tc_eligible(probe, probe, M_vf, O, H_vf, 1) &&
           (M_pi + 63) / 64 + (M_vf + 63) / 64 >= 2;
}

extern "C" int impala_mlp_backward_pair_push(const float* x, const float* params_pi, const float* params_vf,
                                             const float* dlogits, const float* dv, void* workspace_pi,
                                             int64_t workspace_pi_bytes, void* workspace_vf,
                                             int64_t workspace_vf_bytes, int M_pi, int M_vf, int O, int H_pi,
                                             int H_vf, int A, const double* extra, int n_extra,
                                             void* const* peer_gather, const long long* seq,
                                             int64_t slot_stride, int64_t buf_stride, int rank, int world,
                                             void* stream) {
    if (!x || !params_pi || !params_vf || !dlogits || !dv || !workspace_pi || !workspace_vf || !peer_gather ||
        !seq || (n_extra > 0 && !extra))
        return IMPALA_ERR_BAD_ARG;
    if (world < 1 || world > 8 || rank < 0 || rank >= world || n_extra < 0 || n_extra > 32) return IMPALA_ERR_BAD_ARG;
    if (!impala_mlp_backward_pair_push_supported(M_pi, M_vf, O, H_pi, H_vf, A) ||
        !impala_mlp_bwd_tc_eligible(x, dlogits, M_pi, O, H_pi, A) || !impala_mlp_bwd_tc_eligible(x, dv, M_vf, O, H_vf, 1))
        return IMPALA_ERR_UNSUPPORTED_SHAPE;
    const int64_t n_pi = impala_make_layout(O, H_pi, A).total, n_vf = impala_make_layout(O, H_vf, 1).total;
    if (slot_stride < n_pi + n_vf + n_extra || buf_stride < (int64_t)world * slot_stride) return IMPALA_ERR_BAD_ARG;
    const int64_t need_pi = impala_mlp_backward_workspace(M_pi, O, H_pi, A);
    const int64_t need_vf = impala_mlp_backward_workspace(M_vf, O, H_vf, 1);
    if (need_pi < 0 || need_vf < 0) return IMPALA_ERR_UNSUPPORTED_SHAPE;
    if (workspace_pi_bytes < need_pi || workspace_vf_bytes < need_vf) return IMPALA_ERR_WORKSPACE_TOO_SMALL;
    const PushArgs push{reinterpret_cast<ulonglong2* const*>(peer_gather), seq, slot_stride, buf_stride, rank, world};
    return impala_mlp_bwd_tc_pair(
        x, params_pi, params_vf, dlogits, dv,
        reinterpret_cast<float*>(static_cast<char*>(workspace_pi) + kWsHeader),
        reinterpret_cast<float*>(static_cast<char*>(workspace_vf) + kWsHeader), nullptr, nullptr,
        static_cast<unsigned int*>(workspace_pi), M_pi, M_vf, O, H_pi, H_vf, A, (cudaStream_t)stream, &push, extra,
        n_extra);
}
