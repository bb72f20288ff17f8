// d/d theta of the MNLE log-likelihood sum, forward mode, fp32 CUDA cores (sm_100a).
//
// The reference samples with NUTS (mnle.py:81) and calls the potential with
// track_gradients=True (potentials.py:33, 112): autograd differentiates estimator.log_prob with
// respect to the five global parameters.  theta has only five components, so forward mode is the
// cheap direction: every (trial, chain) row carries its value and five tangents d/d theta_i
// through the same networks.  A linear layer acts on a tangent exactly as on a value (minus the
// bias), so the six rows of one (trial, chain) go through the dense() routine of the forward
// kernel side by side; activations, the categorical head and the spline are evaluated on dual
// numbers.  Output: value (C,) and gradient (C,5) of sum_t log p(x_t | theta_c, pulses_t).
#include "mnle_dense.cuh"

namespace mnle {

constexpr int kGradRows = kTM / kDualRows;  // 10 (trial, chain) rows per CTA tile

// value + five tangents
struct Dual {
    float v, d[5];
    __device__ __forceinline__ Dual() {}
    __device__ __forceinline__ explicit Dual(float c) : v(c)
    {
#pragma unroll
        for (int i = 0; i < 5; ++i) d[i] = 0.f;
    }
};
__device__ __forceinline__ Dual operator+(const Dual &a, const Dual &b)
{
    Dual r;
    r.v = a.v + b.v;
#pragma unroll
    for (int i = 0; i < 5; ++i) r.d[i] = a.d[i] + b.d[i];
    return r;
}
__device__ __forceinline__ Dual operator-(const Dual &a, const Dual &b)
{
    Dual r;
    r.v = a.v - b.v;
#pragma unroll
    for (int i = 0; i < 5; ++i) r.d[i] = a.d[i] - b.d[i];
    return r;
}
__device__ __forceinline__ Dual operator*(const Dual &a, const Dual &b)
{
    Dual r;
    r.v = a.v * b.v;
#pragma unroll
    for (int i = 0; i < 5; ++i) r.d[i] = a.d[i] * b.v + a.v * b.d[i];
    return r;
}
__device__ __forceinline__ Dual operator/(const Dual &a, const Dual &b)
{
    Dual r;
    const float inv = 1.0f / b.v;
    r.v = a.v * inv;
#pragma unroll
    for (int i = 0; i < 5; ++i) r.d[i] = (a.d[i] - r.v * b.d[i]) * inv;
    return r;
}
__device__ __forceinline__ Dual operator+(const Dual &a, float c)
{
    Dual r = a;
    r.v += c;
    return r;
}
__device__ __forceinline__ Dual operator*(const Dual &a, float c)
{
    Dual r;
    r.v = a.v * c;
#pragma unroll
    for (int i = 0; i < 5; ++i) r.d[i] = a.d[i] * c;
    return r;
}
__device__ __forceinline__ Dual dexp(const Dual &a)
{
    Dual r;
    r.v = expf(a.v);
#pragma unroll
    for (int i = 0; i < 5; ++i) r.d[i] = a.d[i] * r.v;
    return r;
}
__device__ __forceinline__ Dual dlog(const Dual &a)
{
    Dual r;
    r.v = logf(a.v);
    const float inv = 1.0f / a.v;
#pragma unroll
    for (int i = 0; i < 5; ++i) r.d[i] = a.d[i] * inv;
    return r;
}
__device__ __forceinline__ Dual dsoftplus(const Dual &a)  // softplus' = sigmoid
{
    Dual r;
    r.v = softplus_f(a.v);
    const float sg = 1.0f / (1.0f + expf(-a.v));
#pragma unroll
    for (int i = 0; i < 5; ++i) r.d[i] = a.d[i] * sg;
    return r;
}

// element j of dual row g held as six consecutive rows of a shared-memory tile
__device__ __forceinline__ Dual load_dual(const float *tile, int ld, int g, int j)
{
    Dual r;
    r.v = tile[(g * kDualRows) * ld + j];
#pragma unroll
    for (int i = 0; i < 5; ++i) r.d[i] = tile[(g * kDualRows + 1 + i) * ld + j];
    return r;
}

// a = act(z), a' = act'(z) z' in place over the 128 columns of every dual row
template <int ACT>
__device__ __forceinline__ void activate_dual(float *tile, int ld)
{
    for (int idx = threadIdx.x; idx < kGradRows * kHidden; idx += kThreads) {
        const int g = idx / kHidden, j = idx - g * kHidden;
        float *p = tile + (g * kDualRows) * ld + j;
        const float z = p[0];
        float a, da;
        if (ACT == kRelu) {
            a = fmaxf(z, 0.f);
            da = z > 0.f ? 1.f : 0.f;
        } else {
            a = 1.0f / (1.0f + expf(-z));
            da = a * (1.0f - a);
        }
        p[0] = a;
#pragma unroll
        for (int i = 1; i < kDualRows; ++i) p[i * ld] *= da;
    }
    __syncthreads();
}

// The spline of mnle_common.cuh::rqs_forward on dual numbers (same operation order for the values).
// The softmax shift (max) is piecewise constant, so it carries no tangent.
__device__ __forceinline__ void rqs_forward_dual(Dual &u, Dual &logdet, const float *tile, int ld, int g)
{
    if (!(u.v >= -kTail && u.v <= kTail)) return;  // identity outside the tail bound
    const float inv_sqrt_h = 0.08838834764831845f;
    const float span = 1.0f - kMinBin * kBins;
    Dual left(-kTail), right(kTail), bottom(-kTail), top(kTail);
    int b = 0;
    for (int part = 0; part < 2; ++part) {  // 0: widths (locate the bin), 1: heights (read knots b, b+1)
        const int off = part * kBins;
        float m = -INFINITY;
        for (int j = 0; j < kBins; ++j) m = fmaxf(m, tile[(g * kDualRows) * ld + off + j] * inv_sqrt_h);
        Dual s(0.f);
        for (int j = 0; j < kBins; ++j) s = s + dexp(load_dual(tile, ld, g, off + j) * inv_sqrt_h + (-m));
        Dual cs(0.f), prev(-kTail);
        for (int j = 0; j < kBins; ++j) {
            const Dual w = (dexp(load_dual(tile, ld, g, off + j) * inv_sqrt_h + (-m)) / s) * span + kMinBin;
            cs = cs + w;
            const Dual edge = (j == kBins - 1) ? Dual(kTail) : cs * (2.0f * kTail) + (-kTail);
            if (part == 0) {
                if (u.v >= prev.v) {
                    b = j;
                    left = prev;
                    right = edge;
                }
            } else if (j == b) {
                bottom = prev;
                top = edge;
            }
            prev = edge;
        }
    }
    const Dual one(1.0f);
    const Dual d0 = (b == 0) ? one : dsoftplus(load_dual(tile, ld, g, 2 * kBins + b - 1)) + kMinDeriv;
    const Dual d1 = (b == kBins - 1) ? one : dsoftplus(load_dual(tile, ld, g, 2 * kBins + b)) + kMinDeriv;
    const Dual w = right - left, h = top - bottom;
    const Dual delta = h / w;
    const Dual th = (u - left) / w;
    const Dual om = one - th;
    const Dual t1 = th * om;
    const Dual den = delta + (d0 + d1 - delta * 2.0f) * t1;
    const Dual out = bottom + h * (delta * th * th + d0 * t1) / den;
    const Dual dnum = delta * delta * (d1 * th * th + delta * t1 * 2.0f + d0 * om * om);
    logdet = logdet + dlog(dnum) - dlog(den) * 2.0f;
    u = out;
}

// grid = (ceil(T / 10), C): ten trials of one chain per CTA, six tile rows each.
__global__ void __launch_bounds__(kThreads) mnle_grad_kernel(const float *__restrict__ params, Layout L,
                                                             const float *__restrict__ theta, long long ld_theta,
                                                             const float *__restrict__ x,
                                                             const float *__restrict__ pulses, long long ld_pulses, int T,
                                                             float mu_y, float sigma_y, float *__restrict__ partial)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    SimtSmem &S = *reinterpret_cast<SimtSmem *>(smem_raw);
    const int tid = threadIdx.x;
    const int t0 = blockIdx.x * kGradRows, c = blockIdx.y;

    // ---- inputs: primal row = [theta_c, pulses_t, choice_t]; tangent row i = unit vector e_i ----
    for (int idx = tid; idx < kTM * kLdIn; idx += kThreads) {
        const int row = idx / kLdIn, j = idx - row * kLdIn;
        const int g = row / kDualRows, k = row - g * kDualRows, t = t0 + g;
        float v = 0.f;
        if (g < kGradRows && t < T && j < kCtx) {
            if (k == 0) {
                if (j < 5) v = __ldg(theta + (long long)c * ld_theta + j);
                else if (j < kCond) v = __ldg(pulses + (long long)t * ld_pulses + (j - 5));
                else v = __ldg(x + 2 * t + 1);
            } else if (j == k - 1) {
                v = 1.0f;
            }
        }
        S.in[row * kLdIn + j] = v;
    }
    __syncthreads();

    const bool owner = tid < kGradRows;
    const bool live = owner && (t0 + tid) < T;
    Dual u(0.f), logdet(0.f), lp(0.f);
    float y = 0.f;
    int choice = 0;
    if (live) {
        const float rt = __ldg(x + 2 * (t0 + tid));
        choice = (int)__ldg(x + 2 * (t0 + tid) + 1);
        y = logf(rt);
        u = Dual((y - mu_y) / sigma_y);
        logdet = Dual(-logf(sigma_y));
    }

    // ---- categorical head ----
    dense<8, kNone, true>(params + L.cat_W0, params + L.cat_b0, kCond, kHidden, S.in, kLdIn, S.ha, kLdH, S.w);
    activate_dual<kSigmoid>(S.ha, kLdH);
    dense<8, kNone, true>(params + L.cat_W1, params + L.cat_b1, kHidden, kHidden, S.ha, kLdH, S.hb, kLdH, S.w);
    activate_dual<kSigmoid>(S.hb, kLdH);
    dense<8, kNone, true>(params + L.cat_W2, params + L.cat_b2, kHidden, kHidden, S.hb, kLdH, S.ha, kLdH, S.w);
    activate_dual<kSigmoid>(S.ha, kLdH);
    dense<1, kNone, true>(params + L.cat_Wo, params + L.cat_bo, kHidden, L.n_choices, S.ha, kLdH, S.hb, kLdH, S.w);
    if (live) {
        // log softmax(logits)[choice]; torch's clamp of the probabilities to [eps, 1 - eps] only
        // binds at saturation, where the gradient is taken as that of the unclamped value
        float m = -INFINITY;
        for (int j = 0; j < L.n_choices; ++j) m = fmaxf(m, S.hb[(tid * kDualRows) * kLdH + j]);
        Dual s(0.f);
        for (int j = 0; j < L.n_choices; ++j) s = s + dexp(load_dual(S.hb, kLdH, tid, j) + (-m));
        const int cc = min(max(choice, 0), L.n_choices - 1);
        lp = load_dual(S.hb, kLdH, tid, cc) + (-m) - dlog(s);
        const float eps = 1.1920928955078125e-07f, p = expf(lp.v);
        if (p < eps || p > 1.0f - eps) lp.v = logf(fminf(fmaxf(p, eps), 1.0f - eps));
    }

    // ---- ten spline conditioners ----
    for (int k = 0; k < kTransforms; ++k) {
        dense<8, kNone, true>(params + L.fl_W1[k], params + L.fl_b1[k], kCtx, kHidden, S.in, kLdIn, S.ha, kLdH, S.w);
        activate_dual<kRelu>(S.ha, kLdH);
        dense<8, kNone, true>(params + L.fl_W2[k], params + L.fl_b2[k], kHidden, kHidden, S.ha, kLdH, S.hb, kLdH, S.w);
        activate_dual<kRelu>(S.hb, kLdH);
        dense<5, kNone, true>(params + L.fl_W3[k], params + L.fl_b3[k], kHidden, kSplineOut, S.hb, kLdH, S.ha, kLdH, S.w);
        if (live) rqs_forward_dual(u, logdet, S.ha, kLdH, tid);
    }

    // ---- value and gradient of this tile: fixed-order sum over its (at most ten) trials ----
    float *red = S.w;  // the weight staging area is free now
    __syncthreads();
    if (owner) {
        Dual total(0.f);
        if (live) total = lp + (u * u) * -0.5f + (-0.9189385332046727f) + logdet + (-y);
        red[tid * 6] = total.v;
#pragma unroll
        for (int i = 0; i < 5; ++i) red[tid * 6 + 1 + i] = total.d[i];
    }
    __syncthreads();
    if (tid < 6) {
        float s = 0.f;
        for (int g = 0; g < kGradRows; ++g) s += red[g * 6 + tid];
        partial[((size_t)c * gridDim.x + blockIdx.x) * 6 + tid] = s;
    }
}

// out[c] = sum over tiles of the value, grad[c][i] of the tangents; fixed order
__global__ void grad_reduce_kernel(const float *__restrict__ partial, int n_tiles, int C, float *__restrict__ out,
                                   float *__restrict__ grad)
{
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= C * 6) return;
    const int c = idx / 6, k = idx - c * 6;
    float s = 0.f;
    for (int t = 0; t < n_tiles; ++t) s += partial[((size_t)c * n_tiles + t) * 6 + k];
    if (k == 0) out[c] = s;
    else grad[(size_t)c * 5 + (k - 1)] = s;
}

}  // namespace mnle

using namespace mnle;

DDM_API size_t mnle_loglik_grad_workspace_floats(int64_t T, int64_t C)
{
    if (T <= 0 || C <= 0) return 0;
    return (size_t)C * (size_t)((T + kGradRows - 1) / kGradRows) * 6;
}

DDM_API int mnle_loglik_sum_grad_f32(void *handle, const float *theta_dev, int64_t ld_theta, const float *x_dev,
                                     const float *pulses_dev, int64_t ld_pulses, int64_t T, int64_t C, float *out_dev,
                                     float *grad_dev, float *workspace_dev, void *stream)
{
    Handle *H = live_handle(handle, "mnle_loglik_sum_grad_f32");
    if (H == nullptr) return DDM_ERR_STATE;
    DDM_REQUIRE(T >= 0 && C >= 0 && C <= 65535 && T <= 0x7FFFFFFFll, "mnle_loglik_sum_grad: T=%lld C=%lld out of range",
                (long long)T, (long long)C);
    if (C == 0) return DDM_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    DDM_REQUIRE(out_dev != nullptr && grad_dev != nullptr, "mnle_loglik_sum_grad: null output");
    if (T == 0) {
        DDM_CUDA_TRY(cudaMemsetAsync(out_dev, 0, (size_t)C * sizeof(float), st));
        DDM_CUDA_TRY(cudaMemsetAsync(grad_dev, 0, (size_t)C * 5 * sizeof(float), st));
        return DDM_OK;
    }
    DDM_REQUIRE(theta_dev && x_dev && pulses_dev && workspace_dev, "mnle_loglik_sum_grad: null pointer");
    DDM_REQUIRE(ld_theta >= 5 && ld_pulses >= kCond - 5, "mnle_loglik_sum_grad: ld_theta=%lld ld_pulses=%lld too small",
                (long long)ld_theta, (long long)ld_pulses);
    const int n_tiles = (int)((T + kGradRows - 1) / kGradRows);
    DDM_CUDA_TRY(cudaFuncSetAttribute(mnle_grad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SimtSmem)));
    mnle_grad_kernel<<<dim3((unsigned)n_tiles, (unsigned)C), kThreads, sizeof(SimtSmem), st>>>(
        H->params, H->layout, theta_dev, ld_theta, x_dev, pulses_dev, ld_pulses, (int)T, H->mu_y, H->sigma_y, workspace_dev);
    DDM_CUDA_TRY(cudaGetLastError());
    grad_reduce_kernel<<<(unsigned)((C * 6 + 127) / 128), 128, 0, st>>>(workspace_dev, n_tiles, (int)C, out_dev, grad_dev);
    DDM_CUDA_TRY(cudaGetLastError());
    return DDM_OK;
}
