// MNLE log-likelihood on CUDA cores, fp32 throughout (sm_100a).
//
// One CTA pushes a tile of 64 rows through the categorical net and the ten spline
// conditioners with activations resident in shared memory (never in HBM), applies the
// categorical / spline epilogues row by row and, in potential mode, reduces the per-trial
// log-probabilities of one chain with warp shuffles.  This is the accuracy anchor of the
// tensor-core kernel (mnle_tc.cu) and the path used for shapes the latter does not cover.
//
// Replaces /root/reference/src/sbi_for_diffusion_models/potentials.py:96-115: the reference
// materialises a (T*C, 85) condition matrix and a (1, T*C, 2) x tensor per call (17.8 MB at
// T=50, C=1024) and runs estimator.log_prob over it; here row r = t*C + c is assembled on the
// fly from theta[c], pulses[t], x[t].
#include <type_traits>

#include "mnle_dense.cuh"

namespace mnle {

struct RowSource {
    // rows mode: x (R,2), cond (R,85).   potential mode: theta (C,5), x (T,2), pulses (T,P)
    const float *x;
    const float *cond;
    const float *theta;
    const float *pulses;
    long long ld_cond, ld_theta, ld_pulses;
    long long R;  // rows mode
    int T, C;     // potential mode
    int potential;
};

// PRECISE: the per-row chain (log rt, the ten splines, the categorical head, the final sum) runs in fp64 on the
// fp32 conditioner outputs.  This is the accuracy anchor for trained estimators (see rqs_forward).
template <bool PRECISE>
__global__ void __launch_bounds__(kThreads) mnle_simt_kernel(const float *__restrict__ params, Layout L, RowSource src,
                                                             float mu_y, float sigma_y, float *__restrict__ out)
{
    using Real = typename std::conditional<PRECISE, double, float>::type;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    SimtSmem &S = *reinterpret_cast<SimtSmem *>(smem_raw);
    const int tid = threadIdx.x;

    // ---- which rows does this tile hold? ----------------------------------------------
    // potential mode: blockIdx.y = chain c, blockIdx.x = tile of 64 trials
    // rows mode:      blockIdx.x = tile of 64 rows
    const long long row0 = (long long)blockIdx.x * kTM;
    const int c = blockIdx.y;
    const long long n_rows = src.potential ? (long long)src.T : src.R;

    // ---- assemble the 86-wide context [cond (85), choice] ------------------------------
    for (int idx = tid; idx < kTM * kLdIn; idx += kThreads) {
        const int i = idx / kLdIn, j = idx - i * kLdIn;
        const long long r = row0 + i;
        float v = 0.f;
        if (r < n_rows && j < kCtx) {
            if (j == kCond) v = __ldg(src.x + 2 * r + 1);
            else if (!src.potential) v = __ldg(src.cond + r * src.ld_cond + j);
            else if (j < 5) v = __ldg(src.theta + (long long)c * src.ld_theta + j);
            else v = __ldg(src.pulses + r * src.ld_pulses + (j - 5));
        }
        S.in[i * kLdIn + j] = v;
    }
    __syncthreads();

    // per-row running state lives in the registers of threads 0..63
    const bool owner = tid < kTM;
    const long long my_row = row0 + tid;
    const bool live = owner && my_row < n_rows;
    Real lp = 0, u = 0, logdet = 0, y = 0;
    int choice = 0;
    if (live) {
        const float rt = __ldg(src.x + 2 * my_row);
        choice = (int)__ldg(src.x + 2 * my_row + 1);
        y = rlog((Real)rt);
        u = (y - (Real)mu_y) / (Real)sigma_y;
        logdet = -rlog((Real)sigma_y);
    }

    // ---- categorical head: 85 -> 128 -> 128 -> 128 -> K, sigmoid ------------------------
    dense<8, kSigmoid>(params + L.cat_W0, params + L.cat_b0, kCond, kHidden, S.in, kLdIn, S.ha, kLdH, S.w);
    dense<8, kSigmoid>(params + L.cat_W1, params + L.cat_b1, kHidden, kHidden, S.ha, kLdH, S.hb, kLdH, S.w);
    dense<8, kSigmoid>(params + L.cat_W2, params + L.cat_b2, kHidden, kHidden, S.hb, kLdH, S.ha, kLdH, S.w);
    dense<1, kNone>(params + L.cat_Wo, params + L.cat_bo, kHidden, L.n_choices, S.ha, kLdH, S.hb, kLdH, S.w);
    if (live) lp = categorical_logp<Real>(S.hb + tid * kLdH, 1, L.n_choices, choice);

    // ---- ten spline conditioners: 86 -> 128 -> 128 -> 71, relu --------------------------
    for (int k = 0; k < kTransforms; ++k) {
        dense<8, kRelu>(params + L.fl_W1[k], params + L.fl_b1[k], kCtx, kHidden, S.in, kLdIn, S.ha, kLdH, S.w);
        dense<8, kRelu>(params + L.fl_W2[k], params + L.fl_b2[k], kHidden, kHidden, S.ha, kLdH, S.hb, kLdH, S.w);
        dense<5, kNone>(params + L.fl_W3[k], params + L.fl_b3[k], kHidden, kSplineOut, S.hb, kLdH, S.ha, kLdH, S.w);
        if (live) rqs_forward<Real>(u, logdet, S.ha + tid * kLdH, 1);
    }

    Real total = 0;
    if (live) total = lp + ((Real)-0.5 * u * u - (Real)0.91893853320467274178) + logdet - y;

    if (!src.potential) {
        if (live) out[my_row] = (float)total;
        return;
    }
    // potential mode: deterministic reduction over the tile's trials (warps 0 and 1)
    if (tid < kTM) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) total += __shfl_xor_sync(0xFFFFFFFFu, total, o);
        if ((tid & 31) == 0) S.red[tid >> 5] = total;
    }
    __syncthreads();
    if (tid == 0) out[(long long)c * gridDim.x + blockIdx.x] = S.red[0] + S.red[1];
}

// out[c] = sum over tiles, fixed order
__global__ void reduce_tiles_kernel(const float *__restrict__ partial, int n_tiles, int C, float *__restrict__ out)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    float s = 0.f;
    for (int t = 0; t < n_tiles; ++t) s += partial[(long long)c * n_tiles + t];
    out[c] = s;
}

static int launch(Handle *H, const RowSource &src, dim3 grid, float *out, cudaStream_t st, bool precise = false)
{
    static_assert(sizeof(SimtSmem) < 227 * 1024, "tile does not fit shared memory");
    auto kern = precise ? mnle_simt_kernel<true> : mnle_simt_kernel<false>;
    DDM_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SimtSmem)));
    kern<<<grid, kThreads, sizeof(SimtSmem), st>>>(H->params, H->layout, src, H->mu_y, H->sigma_y, out);
    DDM_CUDA_TRY(cudaGetLastError());
    return DDM_OK;
}

}  // namespace mnle

using namespace mnle;

DDM_API size_t mnle_packed_floats(int n_choices)
{
    if (n_choices < 1 || n_choices > kMaxChoices) return 0;
    return make_layout(n_choices).total;
}

DDM_API int mnle_create(const float *packed_host, size_t n_floats, int n_choices, void **handle_out)
{
    DDM_REQUIRE(handle_out != nullptr && packed_host != nullptr, "mnle_create: null argument");
    DDM_REQUIRE(n_choices >= 1 && n_choices <= kMaxChoices, "mnle_create: n_choices=%d outside [1,%d]", n_choices,
                kMaxChoices);
    Layout L = make_layout(n_choices);
    DDM_REQUIRE(n_floats == L.total, "mnle_create: packed buffer has %zu floats, layout needs %zu", n_floats, L.total);
    const float sigma = packed_host[L.sigma_y];
    DDM_REQUIRE(sigma > 0.0f, "mnle_create: sigma_y must be positive");
    Handle *H = new Handle();
    H->magic = kMagic;
    H->layout = L;
    H->tc_pack = nullptr;
    H->params = nullptr;
    H->mu_y = packed_host[L.mu_y];
    H->sigma_y = sigma;
    cudaError_t e = cudaGetDevice(&H->device);
    if (e == cudaSuccess) e = cudaMalloc(&H->params, L.total * sizeof(float));
    if (e == cudaSuccess) e = cudaMemcpy(H->params, packed_host, L.total * sizeof(float), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) {
        delete H;
        return ddm::cuda_fail(e, "mnle_create");
    }
    const int rc = tc_handle_pack(H);
    if (rc != DDM_OK) {
        cudaFree(H->params);
        if (H->tc_pack) cudaFree(H->tc_pack);
        delete H;
        return rc;
    }
    *handle_out = H;
    return DDM_OK;
}

DDM_API int mnle_destroy(void *handle)
{
    Handle *H = live_handle(handle, "mnle_destroy");
    if (H == nullptr) return DDM_ERR_STATE;
    H->magic = 0;
    cudaFree(H->params);
    if (H->tc_pack) cudaFree(H->tc_pack);
    delete H;
    return DDM_OK;
}

static int rows_impl(void *handle, const float *x_dev, const float *cond_dev, int64_t ld_cond, int64_t R, float *out_dev,
                     void *stream, bool precise)
{
    Handle *H = live_handle(handle, "mnle_log_prob_rows_f32");
    if (H == nullptr) return DDM_ERR_STATE;
    DDM_REQUIRE(R >= 0 && R <= 0x7FFFFFFFll * kTM, "mnle_log_prob_rows_f32: bad R");
    if (R == 0) return DDM_OK;
    DDM_REQUIRE(x_dev && cond_dev && out_dev, "mnle_log_prob_rows_f32: null pointer");
    DDM_REQUIRE(ld_cond >= kCond, "mnle_log_prob_rows_f32: ld_cond=%lld < 85", (long long)ld_cond);
    RowSource src{};
    src.x = x_dev;
    src.cond = cond_dev;
    src.ld_cond = ld_cond;
    src.R = R;
    src.potential = 0;
    return launch(H, src, dim3((unsigned)((R + kTM - 1) / kTM), 1, 1), out_dev, static_cast<cudaStream_t>(stream), precise);
}

DDM_API int mnle_log_prob_rows_f32(void *handle, const float *x_dev, const float *cond_dev, int64_t ld_cond, int64_t R,
                                   float *out_dev, void *stream)
{
    return rows_impl(handle, x_dev, cond_dev, ld_cond, R, out_dev, stream, false);
}

DDM_API int mnle_log_prob_rows_precise_f32(void *handle, const float *x_dev, const float *cond_dev, int64_t ld_cond,
                                           int64_t R, float *out_dev, void *stream)
{
    return rows_impl(handle, x_dev, cond_dev, ld_cond, R, out_dev, stream, true);
}

DDM_API size_t mnle_loglik_workspace_floats(int64_t T, int64_t C)
{
    if (T <= 0 || C <= 0) return 0;
    return (size_t)C * (size_t)((T + kTM - 1) / kTM);
}

static int loglik_sum_impl(void *handle, const float *theta_dev, int64_t ld_theta, const float *x_dev,
                           const float *pulses_dev, int64_t ld_pulses, int64_t T, int64_t C, float *out_dev,
                           float *workspace_dev, void *stream, bool precise)
{
    Handle *H = live_handle(handle, "mnle_loglik_sum_simt_f32");
    if (H == nullptr) return DDM_ERR_STATE;
    DDM_REQUIRE(T >= 0 && C >= 0 && C <= 65535 && T <= 0x7FFFFFFFll, "mnle_loglik_sum: T=%lld C=%lld out of range",
                (long long)T, (long long)C);
    if (C == 0) return DDM_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    DDM_REQUIRE(out_dev != nullptr, "mnle_loglik_sum: null output");
    if (T == 0) {
        DDM_CUDA_TRY(cudaMemsetAsync(out_dev, 0, (size_t)C * sizeof(float), st));
        return DDM_OK;
    }
    DDM_REQUIRE(theta_dev && x_dev && pulses_dev && workspace_dev, "mnle_loglik_sum: null pointer");
    DDM_REQUIRE(ld_theta >= 5 && ld_pulses >= kCond - 5, "mnle_loglik_sum: ld_theta=%lld ld_pulses=%lld too small",
                (long long)ld_theta, (long long)ld_pulses);
    RowSource src{};
    src.x = x_dev;
    src.theta = theta_dev;
    src.pulses = pulses_dev;
    src.ld_theta = ld_theta;
    src.ld_pulses = ld_pulses;
    src.T = (int)T;
    src.C = (int)C;
    src.potential = 1;
    const int n_tiles = (int)((T + kTM - 1) / kTM);
    int rc = launch(H, src, dim3((unsigned)n_tiles, (unsigned)C, 1), workspace_dev, st, precise);
    if (rc != DDM_OK) return rc;
    reduce_tiles_kernel<<<(unsigned)((C + 127) / 128), 128, 0, st>>>(workspace_dev, n_tiles, (int)C, out_dev);
    DDM_CUDA_TRY(cudaGetLastError());
    return DDM_OK;
}

DDM_API int mnle_loglik_sum_simt_f32(void *handle, const float *theta_dev, int64_t ld_theta, const float *x_dev,
                                     const float *pulses_dev, int64_t ld_pulses, int64_t T, int64_t C,
                                     float *out_dev, float *workspace_dev, void *stream)
{
    return loglik_sum_impl(handle, theta_dev, ld_theta, x_dev, pulses_dev, ld_pulses, T, C, out_dev, workspace_dev, stream,
                           false);
}

DDM_API int mnle_loglik_sum_precise_f32(void *handle, const float *theta_dev, int64_t ld_theta, const float *x_dev,
                                        const float *pulses_dev, int64_t ld_pulses, int64_t T, int64_t C,
                                        float *out_dev, float *workspace_dev, void *stream)
{
    return loglik_sum_impl(handle, theta_dev, ld_theta, x_dev, pulses_dev, ld_pulses, T, C, out_dev, workspace_dev, stream,
                           true);
}
