// MNLE (mixed neural likelihood estimator) pieces shared by the fp32 SIMT kernel and the
// tcgen05 kernel: packed-weight layout, rational-quadratic spline, categorical head epilogue.
//
// Semantics: oracle/mnle_spec.py (restatement of sbi 0.25.0 MixedDensityEstimator.log_prob as
// called at /root/reference/src/sbi_for_diffusion_models/potentials.py:113; hyper-parameters
// from /root/reference/src/sbi_for_diffusion_models/mnle.py:31-39).
#pragma once

#include "ddm_common.cuh"

namespace mnle {

constexpr int kHidden = 128;
constexpr int kBins = 24;
constexpr int kTransforms = 10;
constexpr int kCond = 85;           // theta(5) + pulses(80)
constexpr int kCtx = 86;            // + choice
constexpr int kSplineOut = 3 * kBins - 1;  // 71
constexpr int kMaxChoices = 8;
constexpr float kTail = 10.0f;
constexpr float kMinBin = 1e-3f;
constexpr float kMinDeriv = 1e-3f;

// Packed fp32 parameter buffer (host packs with z-scoring folded into the first layers):
//   cat: W0[128][85] b0[128] W1[128][128] b1[128] W2[128][128] b2[128] Wo[K][128] bo[K]
//   flow k = 0..9: W1[128][86] b1[128] W2[128][128] b2[128] W3[71][128] b3[71]
//   tail: mu_y, sigma_y
struct Layout {
    int n_choices;
    size_t cat_W0, cat_b0, cat_W1, cat_b1, cat_W2, cat_b2, cat_Wo, cat_bo;
    size_t fl_W1[kTransforms], fl_b1[kTransforms], fl_W2[kTransforms], fl_b2[kTransforms],
        fl_W3[kTransforms], fl_b3[kTransforms];
    size_t mu_y, sigma_y, total;
};

inline Layout make_layout(int n_choices)
{
    Layout L;
    L.n_choices = n_choices;
    size_t o = 0;
    auto take = [&](size_t n) { size_t at = o; o += n; return at; };
    L.cat_W0 = take((size_t)kHidden * kCond);
    L.cat_b0 = take(kHidden);
    L.cat_W1 = take((size_t)kHidden * kHidden);
    L.cat_b1 = take(kHidden);
    L.cat_W2 = take((size_t)kHidden * kHidden);
    L.cat_b2 = take(kHidden);
    L.cat_Wo = take((size_t)n_choices * kHidden);
    L.cat_bo = take(n_choices);
    for (int k = 0; k < kTransforms; ++k) {
        L.fl_W1[k] = take((size_t)kHidden * kCtx);
        L.fl_b1[k] = take(kHidden);
        L.fl_W2[k] = take((size_t)kHidden * kHidden);
        L.fl_b2[k] = take(kHidden);
        L.fl_W3[k] = take((size_t)kSplineOut * kHidden);
        L.fl_b3[k] = take(kSplineOut);
    }
    L.mu_y = take(1);
    L.sigma_y = take(1);
    L.total = o;
    return L;
}

// ---- tensor-core operand pack (mnle_tc.cu) ------------------------------------------------
// One row tile goes through kTcStages GEMM stages: per net a "theta stage" (K = 32, the five
// global parameters in a six-term bf16 expansion; the pulse / choice part of the first layer is
// a per-trial bias computed once per call) followed by the K = 128 layers with bf16 hi/lo
// operands.  Every stage is one contiguous blob (operand images in the shared-memory layout the
// UMMA descriptors expect, then the fp32 bias) so a single bulk copy stages it.
constexpr int kTcStages = 4 + 3 * kTransforms;  // cat: theta, W1, W2, Wo; flow: theta, W2, W3
constexpr int kNets = 1 + kTransforms;
constexpr int kSplineN = 80;                    // 71 spline parameters padded to a legal UMMA N
enum TcEpilogue { kEpiRelu = 0, kEpiSigmoid = 1, kEpiSpline = 2, kEpiCategorical = 3 };
// theta stage (K = 32, potential mode) | K = 128 hi/lo layer | whole first layer (K = 96, rows mode)
enum TcStageKind { kStageTheta = 0, kStageK128 = 1, kStageInput = 2 };
constexpr int kInputK = 96;                     // 86 context columns padded to a multiple of 16
struct TcStage {
    uint32_t off, bytes;  // blob position in the pack (16-byte multiples)
    uint32_t bias_off;    // where the N bias floats sit relative to the staged blob
    uint16_t n;           // UMMA N (multiple of 16)
    uint8_t kind;         // TcStageKind
    uint8_t epi;          // TcEpilogue
    uint16_t net, pad;    // net: 0 = categorical net, 1 + k = spline conditioner k; pad: 1 + activation slot the
                          // training forward keeps this stage's output in (0: not kept)
};
struct TcPlan {
    TcStage st[kTcStages];
};

struct Handle {
    uint32_t magic;
    int device;
    Layout layout;
    float *params;   // device copy of the packed buffer
    void *tc_pack;   // tensor-core operand pack (bf16 hi/lo tiles) built on the device from params, or null
    TcPlan tc_plan;       // potential mode: rows = (trial, chain), first layers hoisted per trial
    TcPlan tc_rows_plan;  // rows mode: arbitrary (R, 85) conditions, first layers on the tensor cores
    float mu_y, sigma_y;
};
int tc_handle_pack(Handle *H);  // mnle_tc.cu: allocates and writes tc_pack, sets both plans

// Training forward on the tensor cores (mnle_tc.cu): the rows-mode kernel over the minibatch with the
// operand pack rebuilt on the device from the current parameters, keeping what the backward pass needs.
struct TcTrainDump {
    float *H;      // [kNets][3][128][Rp] hidden activations, column-major
    float *Q;      // [kTransforms][Rp][72] raw spline parameters
    float *LG;     // [Rp][kMaxChoices] choice logits
    long long Rp;  // rows allocated (a multiple of 64, >= R)
    float *DH;     // backward pass only: [kNets][3][128][Rp] d loss / d (hidden pre-activations), written
    const unsigned char *ctx;  // forward only: per 128-row tile the bf16 hi / lo context images (tc_prep_kernel)
    float *CX;     // forward only (may be null): [86][Rp] the gathered context rows [cond (85), choice], column-major --
                   // the X operand of the first layers' weight-gradient GEMMs
    // backward pass of the POTENTIAL (d / d theta only; both null in the training step): DH may then be null (nothing
    // but the theta columns of the first layers is wanted), W1T = [kNets][128][8] the five theta columns of every
    // first layer (padded to eight), GP = [kNets][2][5][Rp] per row and column half: sum_j dh1[j] * W1[j][i]
    float *GP;
    const float *W1T;
    // potential mode, forward and backward: [kNets][3][4][Rp] sign masks of the ReLU layers' pre-activations (bit 31 - j
    // of word c: column 32 c + j is negative) kept INSTEAD of the activations -- the backward-data pass needs nothing
    // else from a ReLU layer, and 16 bytes per (row, layer) replace 512.  The sigmoid layers still go through H.
    uint32_t *HM;
    // forward only: the launch runs nets [net0, net0 + nets).  A launch with net0 > 0 rebuilds the context images but
    // not the operand pack: a launch from net 0 in the same call must have written it (the sampler runs the
    // categorical net, draws the choice into x, then runs the ten conditioners on the new context).
    int net0 = 0, nets = kNets;
};
size_t tc_train_pack_bytes(int n_choices, long long R);  // operand pack + context images of R rows
int tc_train_forward(const float *params_dev, const Layout &L, void *pack_dev, const float *x_dev, const float *cond_dev,
                     long long ld_cond, const long long *row_index_dev, long long R, const TcTrainDump &dump,
                     float *lp_dev, cudaStream_t st);
// Backward-data pass on the tensor cores over the same pack (tc_train_forward must have run in this call):
// d loss / d (spline parameters, logits) in dump.Q / dump.LG and the activations dump.H give dump.DH.
int tc_train_backward(const Layout &L, const void *pack_dev, long long R, const TcTrainDump &dump, cudaStream_t st);
constexpr uint32_t kMagic = 0x4D4E4C45u;  // "MNLE"

// `handle` as a live MNLE handle (that also has its tensor-core operand pack when need_tc_pack), or null after setting
// the error string "<entry point>: bad handle"; the entry point then returns DDM_ERR_STATE.
inline Handle *live_handle(void *handle, const char *entry, bool need_tc_pack = false)
{
    Handle *H = static_cast<Handle *>(handle);
    if (H == nullptr || H->magic != kMagic || (need_tc_pack && H->tc_pack == nullptr)) {
        ddm::set_error("%s: bad handle", entry);
        return nullptr;
    }
    return H;
}

__device__ __forceinline__ float softplus_f(float x)
{
    return x > 20.0f ? x : log1pf(expf(x));  // torch.nn.functional.softplus, threshold 20
}
__device__ __forceinline__ double softplus_f(double x) { return x > 20.0 ? x : log1p(exp(x)); }

// scalar helpers so that the spline below reads the same in fp32 and fp64
__device__ __forceinline__ float rexp(float x) { return expf(x); }
__device__ __forceinline__ double rexp(double x) { return exp(x); }
__device__ __forceinline__ float rlog(float x) { return logf(x); }
__device__ __forceinline__ double rlog(double x) { return log(x); }

// One rational-quadratic spline transform with linear tails (Durkan et al. 2019) on a scalar.
// q points at the 71 raw conditioner outputs of this row (stride qs floats between them).
// Real = float: the arithmetic of the fp32 kernels (and of the reference, which evaluates sbi's
// estimator in fp32).  Real = double: the "precise" path.  On a TRAINED estimator the knots of narrow,
// steep bins amplify the rounding of the softmax / cumulative-sum stage by 2-3 orders of magnitude: any
// fp32 evaluation (torch on the CPU included) sits ~3e-4 per row from exact arithmetic, a float64 spline on
// fp32 conditioner outputs ~1e-6 (DESIGN.md section 4).
template <typename Real, typename Stride>
__device__ __forceinline__ void rqs_forward(Real &u, Real &logdet, const float *q, Stride qs)
{
    const Real tail = (Real)kTail, min_bin = (Real)1e-3, min_deriv = (Real)1e-3, one = (Real)1, two = (Real)2;
    if (!(u >= -tail && u <= tail)) return;  // identity outside the tail bound
    const Real inv_sqrt_h = (Real)0.08838834764831844055;  // 1/sqrt(128)
    const Real span = one - min_bin * (Real)kBins;
    // ---- widths: softmax -> cumulative knots, locate the bin -------------------------
    Real m = -(Real)INFINITY;
#pragma unroll 4
    for (int j = 0; j < kBins; ++j) m = fmax(m, (Real)q[j * qs] * inv_sqrt_h);
    Real s = 0;
#pragma unroll 4
    for (int j = 0; j < kBins; ++j) s += rexp((Real)q[j * qs] * inv_sqrt_h - m);
    const Real inv_s = one / s;
    Real cs = 0, prev = -tail, left = -tail, right = tail;
    int b = 0;
#pragma unroll 4
    for (int j = 0; j < kBins; ++j) {
        const Real w = min_bin + span * (rexp((Real)q[j * qs] * inv_sqrt_h - m) * inv_s);
        cs += w;
        const Real edge = (j == kBins - 1) ? tail : (two * tail * cs - tail);
        if (u >= prev) {
            b = j;
            left = prev;
            right = edge;
        }
        prev = edge;
    }
    // ---- heights: same construction, read knots b and b+1 -----------------------------
    const float *qh = q + kBins * qs;
    m = -(Real)INFINITY;
#pragma unroll 4
    for (int j = 0; j < kBins; ++j) m = fmax(m, (Real)qh[j * qs] * inv_sqrt_h);
    s = 0;
#pragma unroll 4
    for (int j = 0; j < kBins; ++j) s += rexp((Real)qh[j * qs] * inv_sqrt_h - m);
    const Real inv_sh = one / s;
    cs = 0;
    prev = -tail;
    Real bottom = -tail, top = tail;
#pragma unroll 4
    for (int j = 0; j < kBins; ++j) {
        const Real h = min_bin + span * (rexp((Real)qh[j * qs] * inv_sqrt_h - m) * inv_sh);
        cs += h;
        const Real edge = (j == kBins - 1) ? tail : (two * tail * cs - tail);
        if (j == b) {
            bottom = prev;
            top = edge;
        }
        prev = edge;
    }
    // ---- knot derivatives (boundary derivatives are exactly 1) ------------------------
    const float *qd = q + 2 * kBins * qs;
    // nflows pads the derivative logits with log(exp(1 - min_derivative) - 1), i.e.
    // min_derivative + softplus(pad) == 1: the spline meets the linear tails with slope 1.
    const Real edge_d = one;
    const Real d0 = (b == 0) ? edge_d : min_deriv + softplus_f((Real)qd[(b - 1) * qs]);
    const Real d1 = (b == kBins - 1) ? edge_d : min_deriv + softplus_f((Real)qd[b * qs]);

    const Real w = right - left, h = top - bottom;
    const Real delta = h / w;
    const Real th = (u - left) / w;
    const Real t1 = th * (one - th);
    const Real den = delta + (d0 + d1 - two * delta) * t1;
    const Real out = bottom + h * (delta * th * th + d0 * t1) / den;
    const Real dnum = delta * delta * (d1 * th * th + two * delta * t1 + d0 * (one - th) * (one - th));
    logdet += rlog(dnum) - two * rlog(den);
    u = out;
}

// log Categorical(choice | softmax(logits)) with torch's probs clamp to [eps, 1 - eps].
template <typename Real = float>
__device__ __forceinline__ Real categorical_logp(const float *logits, int ls, int n_choices, int choice)
{
    Real m = -(Real)INFINITY;
    for (int j = 0; j < n_choices; ++j) m = fmax(m, (Real)logits[j * ls]);
    Real s = 0, pc = 0;
    for (int j = 0; j < n_choices; ++j) {
        const Real e = rexp((Real)logits[j * ls] - m);
        s += e;
        if (j == choice) pc = e;
    }
    Real p = pc / s;
    const Real eps = (Real)1.1920928955078125e-07;
    p = fmin(fmax(p, eps), (Real)1 - eps);
    return rlog(p);
}

// Session of flat trial t (0 <= t < offsets[D]) in a ragged batch: the d with offsets[d] <= t < offsets[d + 1].
// Empty sessions (offsets[d] == offsets[d + 1]) own no trial and are never returned.
__device__ __forceinline__ int session_of(const long long *__restrict__ offsets, int D, long long t)
{
    int lo = 0, hi = D;  // offsets[lo] <= t < offsets[hi]
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (__ldg(offsets + mid) <= t) lo = mid;
        else hi = mid;
    }
    return lo;
}

}  // namespace mnle
