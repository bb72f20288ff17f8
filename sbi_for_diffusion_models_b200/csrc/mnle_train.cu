// MNLE training step on the device (SURVEY 8f row f4): every GEMM on tcgen05, the per-row spline work
// and the reductions on the CUDA cores (sm_100a).
//
// The reference trains the estimator with sbi's MNLE.train (mnle.py:41-48): Adam on
// loss = -mean log p(x | z) over minibatches of TRAIN_BATCH_SIZE = 4096 rows (run_config.py:12),
// autograd through the categorical net and the ten spline conditioners.  Here one call gives the
// loss and its gradient with respect to every packed parameter (layout: mnle_common.cuh):
//
//   1. tc_train_forward        (mnle_tc.cu) the tcgen05 rows-mode kernel over the minibatch, its operand
//                              pack rebuilt on the device from the current parameters; keeps the 71
//                              raw spline parameters per (row, transform), the choice logits and the
//                              hidden activations.
//   2. train_rows_kernel       four lanes per row (six bins per lane): choice log-probability, the ten splines forward
//                              (log p of the row), then backwards (reverse mode written out by
//                              hand), turning the stored spline parameters and logits into
//                              d loss / d (spline parameters, logits) in place.
//   3. tc_train_backward       (mnle_tc.cu) backward-data on tcgen05, one CTA per (row tiles, net):
//                              transposed weight images, the activation derivative fused into the
//                              epilogue, writes d loss / d (hidden pre-activations).  (train_forward_kernel /
//                              train_backward_kernel below: the same two passes on the fp32 CUDA cores,
//                              the accuracy anchor behind DDM_TRAIN_FP32_FORWARD.)
//      train_wgrad_tc_kernel   the weight gradients dW = dY^T X of all 34 layers as tcgen05 GEMMs over
//                              the rows of the minibatch (bf16 hi / lo operands, fp32 accumulation in
//                              tensor memory); each row split owns a slice of the partial-gradient
//                              buffer: no atomics.
//   4. train_reduce_kernel     sums the partials in a fixed order (bit-reproducible gradients) and
//                              the squared gradient norm; train_stats_kernel: loss and norm.
//   5. adam_kernel             torch.optim.Adam update with clip_grad_norm_ folded in.
#include <algorithm>

#include "mnle_dense.cuh"
#include "tc_ptx.cuh"

namespace mnle {

constexpr int kQRows = 72;         // 71 spline parameters per transform, padded
constexpr int kMaxGroups = 8;      // partial-gradient slices = row splits of the weight-gradient kernel (34 layers x 8 = 272 CTAs, two per SM)
constexpr int kWgRows = 64;        // rows of the minibatch per chunk (= K of one accumulation step) of that kernel
constexpr int kReduceThreads = 256;

// Lays out a workspace from `base`: every buffer starts a multiple of 256 bytes past the base (enough for the 16-byte
// bulk copies from the operand pack, the float4 stores into the spline parameters and the fp64 arrays), and floats()
// is what the buffers handed out so far span.  A null base only counts.  Each entry point lays out its workspace in one
// function that runs twice, on a null base for its *_workspace_floats query and on the caller's pointer in the
// launcher, so the size a caller allocates and the buffers the launcher hands out cannot disagree.
class Carver {
  public:
    explicit Carver(float *base) : base_(base) {}
    template <typename T = float>
    T *take(size_t n)
    {
        const size_t at = (used_ + 63) / 64 * 64;
        used_ = at + (n * sizeof(T) + sizeof(float) - 1) / sizeof(float);
        return base_ ? reinterpret_cast<T *>(base_ + at) : nullptr;
    }
    size_t floats() const { return used_; }

  private:
    float *base_;
    size_t used_ = 0;
};

struct TrainBufs {
    unsigned char *pack; // tensor-core operand pack of the current parameters (rebuilt every call) + context images
    float *Q;    // [kTransforms][Rp][kQRows]  spline parameters -> their gradients
    float *LG;   // [Rp][kMaxChoices]          choice logits -> their gradients
    float *LP;   // [Rp]                       log p per row
    float *H;    // [kNets][3][128][Rp]        hidden activations kept for the backward pass, COLUMN-major: the
                 //                            tensor-core epilogues hold one row per lane, so a warp's access to one
                 //                            column of 32 consecutive rows is one 128-byte line
    float *DH;   // [kNets][3][128][Rp]        d loss / d (hidden pre-activations), same layout
    float *P;    // [groups][total]            partial gradients (one slice per row split of the wgrad kernel)
    float *SS;   // [reduce blocks]            partial sums of grad^2
};

struct TrainDims {
    long long R, Rp;
    int tiles, groups, reduce_blocks;
};

static TrainDims train_dims(const Layout &L, long long R)
{
    TrainDims d;
    d.R = R;
    d.tiles = (int)((R + kTM - 1) / kTM);
    d.Rp = (long long)d.tiles * kTM;
    const int chunks = (int)((R + kWgRows - 1) / kWgRows);   // row chunks of the weight-gradient GEMMs
    d.groups = chunks < kMaxGroups ? chunks : kMaxGroups;
    d.reduce_blocks = (int)((L.total + kReduceThreads - 1) / kReduceThreads);
    return d;
}

static TrainBufs train_workspace(Carver &ws, const Layout &L, const TrainDims &d)
{
    TrainBufs b;
    b.pack = ws.take<unsigned char>(tc_train_pack_bytes(L.n_choices, d.R));
    b.Q = ws.take((size_t)kTransforms * kQRows * d.Rp);
    b.LG = ws.take((size_t)kMaxChoices * d.Rp);
    b.LP = ws.take(d.Rp);
    b.H = ws.take((size_t)kNets * 3 * kHidden * d.Rp);
    b.DH = ws.take((size_t)kNets * 3 * kHidden * d.Rp);
    b.P = ws.take((size_t)d.groups * L.total);
    b.SS = ws.take(d.reduce_blocks);
    return b;
}

struct TrainRows {
    const float *x;        // (N,2) [rt seconds, choice]
    const float *cond;     // (N,85), row stride ld_cond
    const long long *idx;  // minibatch row r is dataset row idx[r]; null = identity
    long long ld_cond, R;
};

__device__ __forceinline__ long long data_row(const TrainRows &rows, long long r)
{
    return rows.idx ? rows.idx[r] : r;
}

// 86-wide context [condition, choice] of the tile's rows; rows past R are zero
__device__ __forceinline__ void load_context(const TrainRows &rows, long long row0, float *in_s)
{
    for (int idx = threadIdx.x; idx < kTM * kLdIn; idx += kThreads) {
        const int i = idx / kLdIn, j = idx - i * kLdIn;
        const long long r = row0 + i;
        float v = 0.f;
        if (r < rows.R && j < kCtx) {
            const long long dr = data_row(rows, r);
            v = (j == kCond) ? __ldg(rows.x + 2 * dr + 1) : __ldg(rows.cond + dr * rows.ld_cond + j);
        }
        in_s[i * kLdIn + j] = v;
    }
}

// ---- 1. forward through the nets ------------------------------------------------------------
// hidden activations of one net for the backward pass: [net][slot][row][128]
__device__ __forceinline__ void save_hidden(const float *h_s, float *H, long long Rp, int net, int slot, long long row0)
{
    float *dst = H + ((size_t)net * 3 + slot) * kHidden * (size_t)Rp + row0;
    for (int idx = threadIdx.x; idx < kTM * kHidden; idx += kThreads)  // consecutive threads = consecutive rows
        dst[(size_t)(idx >> 6) * Rp + (idx & (kTM - 1))] = h_s[(idx & (kTM - 1)) * kLdH + (idx >> 6)];
}

__device__ __forceinline__ void load_hidden(float *h_s, const float *H, long long Rp, int net, int slot, long long row0)
{
    const float *src = H + ((size_t)net * 3 + slot) * kHidden * (size_t)Rp + row0;
    for (int idx = threadIdx.x; idx < kTM * kHidden; idx += kThreads)
        h_s[(idx & (kTM - 1)) * kLdH + (idx >> 6)] = src[(size_t)(idx >> 6) * Rp + (idx & (kTM - 1))];
}

// n leading columns of a tile between shared memory [i][ld] and row-major global storage [row][ldg]
__device__ __forceinline__ void store_rows(const float *src_s, int ld, float *dst, int ldg, long long row0, int n)
{
    for (int idx = threadIdx.x; idx < kTM * n; idx += kThreads) {
        const int i = idx / n, j = idx - i * n;
        dst[(size_t)(row0 + i) * ldg + j] = src_s[i * ld + j];
    }
}

__device__ __forceinline__ void load_rows(const float *src, int ldg, long long row0, int n, float *dst_s)
{
    const int n4 = (n + 3) & ~3;  // dense() reads whole groups of four columns: zero the padding
    for (int idx = threadIdx.x; idx < kTM * n4; idx += kThreads) {
        const int i = idx / n4, j = idx - i * n4;
        dst_s[i * kLdIn + j] = j < n ? src[(size_t)(row0 + i) * ldg + j] : 0.f;
    }
}

// fp32 CUDA-core forward (DDM_TRAIN_FP32_FORWARD: the accuracy anchor of the tensor-core forward).
// grid (row tiles, nets): the eleven nets depend only on the context, so they run side by side
__global__ void __launch_bounds__(kThreads) train_forward_kernel(const float *__restrict__ params, Layout L,
                                                                 TrainRows rows, long long Rp, TrainBufs B, int keep)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    SimtSmem &S = *reinterpret_cast<SimtSmem *>(smem_raw);
    const long long row0 = (long long)blockIdx.x * kTM;
    const int net = blockIdx.y;
    load_context(rows, row0, S.in);
    if (net == 0) {
        dense<8, kSigmoid>(params + L.cat_W0, params + L.cat_b0, kCond, kHidden, S.in, kLdIn, S.ha, kLdH, S.w);
        if (keep) save_hidden(S.ha, B.H, Rp, 0, 0, row0);
        dense<8, kSigmoid>(params + L.cat_W1, params + L.cat_b1, kHidden, kHidden, S.ha, kLdH, S.hb, kLdH, S.w);
        if (keep) save_hidden(S.hb, B.H, Rp, 0, 1, row0);
        dense<8, kSigmoid>(params + L.cat_W2, params + L.cat_b2, kHidden, kHidden, S.hb, kLdH, S.ha, kLdH, S.w);
        if (keep) save_hidden(S.ha, B.H, Rp, 0, 2, row0);
        dense<1, kNone>(params + L.cat_Wo, params + L.cat_bo, kHidden, L.n_choices, S.ha, kLdH, S.hb, kLdH, S.w);
        store_rows(S.hb, kLdH, B.LG, kMaxChoices, row0, L.n_choices);
    } else {
        const int k = net - 1;
        dense<8, kRelu>(params + L.fl_W1[k], params + L.fl_b1[k], kCtx, kHidden, S.in, kLdIn, S.ha, kLdH, S.w);
        if (keep) save_hidden(S.ha, B.H, Rp, net, 0, row0);
        dense<8, kRelu>(params + L.fl_W2[k], params + L.fl_b2[k], kHidden, kHidden, S.ha, kLdH, S.hb, kLdH, S.w);
        if (keep) save_hidden(S.hb, B.H, Rp, net, 1, row0);
        dense<5, kNone>(params + L.fl_W3[k], params + L.fl_b3[k], kHidden, kSplineOut, S.hb, kLdH, S.ha, kLdH, S.w);
        store_rows(S.ha, kLdH, B.Q + (size_t)k * kQRows * Rp, kQRows, row0, kSplineOut);
    }
}

// ---- 2. per-row work: four lanes per row, six bins per lane ----------------------------------
// (Round 1 and the first half of round 2 ran one warp per row with lane j owning bin j: 24 of 32 lanes busy, every
// softmax / cumulative sum a pair of five-step warp scans -- ~315 warp-instructions per (row, transform) pass.  With
// six bins per lane the scans are local, the four lanes of a row meet in two-step shuffles, and a warp carries eight
// rows: ~55 warp-instructions per (row, transform) pass.)
constexpr int kRowWarps = 8;
constexpr int kRowLanes = 4;                       // lanes per row
constexpr int kLaneBins = kBins / kRowLanes;       // 6
constexpr int kWarpRows = 32 / kRowLanes;          // 8 rows per warp
constexpr int kBlockRows = kRowWarps * kWarpRows;  // 64 rows per block
static_assert(kBins == kRowLanes * kLaneBins && kSplineOut == 3 * kBins - 1, "six bins per lane");
constexpr unsigned kFull = 0xFFFFFFFFu;

__device__ __forceinline__ float quad_max(float v)
{
    v = fmaxf(v, __shfl_xor_sync(kFull, v, 1));
    return fmaxf(v, __shfl_xor_sync(kFull, v, 2));
}
__device__ __forceinline__ int quad_sum(int v)
{
    v += __shfl_xor_sync(kFull, v, 1);
    return v + __shfl_xor_sync(kFull, v, 2);
}
template <typename T>
__device__ __forceinline__ T quad_get(T v, int base, int sub) { return __shfl_sync(kFull, v, base + sub); }

// entry `i` (0..5, not known at compile time) of a register array: a select chain, no local memory
__device__ __forceinline__ float pick6(const float (&v)[kLaneBins], int i)
{
    float r = v[0];
#pragma unroll
    for (int j = 1; j < kLaneBins; ++j) r = (i == j) ? v[j] : r;
    return r;
}

// softmax over the 24 logits of a row (six per lane, bins 6 s .. 6 s + 5 on sub-lane s) and the knot positions built
// from it: e = softmax probability of the bin, cum = sum of e over the bins before it, lo / hi = the bin's edges
// 20 * cumsum(m + c e) - 10 with both ends pinned to -+10.
struct Knots6 {
    float e[kLaneBins], cum[kLaneBins], lo[kLaneBins], hi[kLaneBins];
};
__device__ __forceinline__ void knots6(const float (&logit)[kLaneBins], int base, int sub, Knots6 &k)
{
    const float inv_sqrt_h = 0.08838834764831845f;  // 1/sqrt(128)
    const float c = 1.0f - kMinBin * kBins;
    float a[kLaneBins];
    float m = -INFINITY;
#pragma unroll
    for (int i = 0; i < kLaneBins; ++i) {
        a[i] = logit[i] * inv_sqrt_h;
        m = fmaxf(m, a[i]);
    }
    m = quad_max(m);
    float pre[kLaneBins];  // inclusive prefix sums within the lane
    float run = 0.f;
#pragma unroll
    for (int i = 0; i < kLaneBins; ++i) {
        k.e[i] = expf(a[i] - m);
        run += k.e[i];
        pre[i] = run;
    }
    // totals of the four lanes, added in the same order everywhere: every lane of the row sees the same sum
    const float t0 = quad_get(run, base, 0), t1 = quad_get(run, base, 1), t2 = quad_get(run, base, 2), t3 = quad_get(run, base, 3);
    const float off = (sub > 0 ? t0 : 0.f) + (sub > 1 ? t1 : 0.f) + (sub > 2 ? t2 : 0.f);
    const float inv_s = 1.0f / (((t0 + t1) + t2) + t3);
#pragma unroll
    for (int i = 0; i < kLaneBins; ++i) {
        const int j = kLaneBins * sub + i;
        k.e[i] *= inv_s;
        const float inc = (off + pre[i]) * inv_s;  // inclusive cumulative probability
        k.cum[i] = inc - k.e[i];
        k.hi[i] = (j >= kBins - 1) ? kTail : 2.0f * kTail * (kMinBin * (float)(j + 1) + c * inc) - kTail;
    }
    const float up = __shfl_up_sync(kFull, k.hi[kLaneBins - 1], 1);  // (sub > 0: the lane below belongs to the same row)
    k.lo[0] = (sub == 0) ? -kTail : up;
#pragma unroll
    for (int i = 1; i < kLaneBins; ++i) k.lo[i] = k.hi[i - 1];
}

// One rational-quadratic spline for the quad's row (Durkan et al. 2019, linear tails).  q points at the row's 71 raw
// parameters of this transform.  Forward: u <- spline(u), logdet += log |du_out / du|.
// BACKWARD (reverse mode written out by hand): u is the transform's INPUT, g = d l / d u_out on entry (l = log p of the
// row, d l / d logdet = 1) and d l / d u on exit; q[j] <- scale * d l / d q[j].  Rows differ within a warp, so nothing
// here branches on the row: a row outside the tail bound (identity, no parameter dependence) computes on u = 0 and
// discards the result.
template <bool BACKWARD>
__device__ __forceinline__ void rqs_quad(float &u, float &logdet, float *q, int base, int sub, bool live, float &g, float scale)
{
    const bool inside = (u >= -kTail && u <= kTail);
    const float ui = inside ? u : 0.f;
    float qw[kLaneBins], qh[kLaneBins], qd[kLaneBins];
    {
        // 6 s floats into each third of the row: 24 s bytes, 8-byte aligned
        const float2 *pw = reinterpret_cast<const float2 *>(q + kLaneBins * sub);
        const float2 *ph = reinterpret_cast<const float2 *>(q + kBins + kLaneBins * sub);
        const float2 *pd = reinterpret_cast<const float2 *>(q + 2 * kBins + kLaneBins * sub);
#pragma unroll
        for (int i = 0; i < kLaneBins / 2; ++i) {
            const float2 w2 = live ? pw[i] : make_float2(0.f, 0.f), h2 = live ? ph[i] : make_float2(0.f, 0.f);
            const float2 d2 = live ? pd[i] : make_float2(0.f, 0.f);   // (element 71 of the row is padding)
            qw[2 * i] = w2.x, qw[2 * i + 1] = w2.y, qh[2 * i] = h2.x, qh[2 * i + 1] = h2.y, qd[2 * i] = d2.x, qd[2 * i + 1] = d2.y;
        }
    }
    Knots6 W, H;
    knots6(qw, base, sub, W);
    knots6(qh, base, sub, H);
    // bin: the last one whose left edge is <= u (left edges are increasing, the first is -10)
    int cnt = 0;
#pragma unroll
    for (int i = 0; i < kLaneBins; ++i) cnt += (ui >= W.lo[i]) ? 1 : 0;
    const int b = quad_sum(cnt) - 1;
    const int sb = (b >= kLaneBins ? 1 : 0) + (b >= 2 * kLaneBins ? 1 : 0) + (b >= 3 * kLaneBins ? 1 : 0), ib = b - kLaneBins * sb;
    const float left = quad_get(pick6(W.lo, ib), base, sb), right = quad_get(pick6(W.hi, ib), base, sb);
    const float bottom = quad_get(pick6(H.lo, ib), base, sb), top = quad_get(pick6(H.hi, ib), base, sb);
    const int bm = b > 0 ? b - 1 : 0;
    const int sm = (bm >= kLaneBins ? 1 : 0) + (bm >= 2 * kLaneBins ? 1 : 0) + (bm >= 3 * kLaneBins ? 1 : 0), im = bm - kLaneBins * sm;
    const float qd0 = quad_get(pick6(qd, im), base, sm), qd1 = quad_get(pick6(qd, ib), base, sb);
    // knot derivatives; the boundary ones are exactly 1 (min_derivative + softplus(pad) == 1)
    const float d0 = (b == 0) ? 1.0f : kMinDeriv + softplus_f(qd0);
    const float d1 = (b == kBins - 1) ? 1.0f : kMinDeriv + softplus_f(qd1);

    const float w = right - left, h = top - bottom;
    const float delta = h / w;
    const float th = (ui - left) / w;
    const float omt = 1.0f - th;
    const float t1 = th * omt;
    const float dd = d0 + d1 - 2.0f * delta;
    const float den = delta + dd * t1;
    const float s1 = delta * th * th + d0 * t1;
    const float num = h * s1;
    const float s2 = d1 * th * th + 2.0f * delta * t1 + d0 * omt * omt;
    const float dnum = delta * delta * s2;
    if (!BACKWARD) {
        if (inside) {
            logdet += logf(dnum) - 2.0f * logf(den);
            u = bottom + num / den;
        }
        return;
    }
    const float inv_den = 1.0f / den;
    const float g_num = g * inv_den;
    const float g_den = -g * num * inv_den * inv_den - 2.0f * inv_den;
    const float g_s2 = 1.0f / s2;  // d log(dnum) / d s2
    const float g_s1 = g_num * h;
    float g_h = g_num * s1;
    const float g_delta = g_s1 * th * th + g_den * (1.0f - 2.0f * t1) + 2.0f / delta + g_s2 * 2.0f * t1;
    float g_th = g_s1 * 2.0f * delta * th + g_s2 * (2.0f * d1 * th - 2.0f * d0 * omt);
    const float g_t1 = g_s1 * d0 + g_den * dd + g_s2 * 2.0f * delta;
    const float g_d0 = g_s1 * t1 + g_den * t1 + g_s2 * omt * omt;
    const float g_d1 = g_den * t1 + g_s2 * th * th;
    g_th += g_t1 * (1.0f - 2.0f * th);
    const float inv_w = 1.0f / w;
    const float g_u = g_th * inv_w;
    g_h += g_delta * inv_w;
    const float g_w = -g_th * th * inv_w - g_delta * delta * inv_w;
    // knots -> softmax logits: edge_j = 20 * sum_{i<j} (m + c e_i) - 10 for 1 <= j <= K-1, ends pinned
    const float gl = (b >= 1) ? -g_u - g_w : 0.f, gr = (b <= kBins - 2) ? g_w : 0.f;
    const float gb = (b >= 1) ? g - g_h : 0.f, gt = (b <= kBins - 2) ? g_h : 0.f;
    const float k20 = 2.0f * kTail * (1.0f - kMinBin * kBins);
    const float Sw = quad_get(pick6(W.cum, ib), base, sb), ew = quad_get(pick6(W.e, ib), base, sb);
    const float Sh = quad_get(pick6(H.cum, ib), base, sb), eh = quad_get(pick6(H.e, ib), base, sb);
    const float dot_w = k20 * (gl * Sw + gr * (Sw + ew));
    const float dot_h = k20 * (gb * Sh + gt * (Sh + eh));
    const float out_scale = inside ? scale * 0.08838834764831845f : 0.f;
    const float v0 = inside ? scale * g_d0 / (1.0f + expf(-qd0)) : 0.f;  // softplus' = sigmoid
    const float v1 = inside ? scale * g_d1 / (1.0f + expf(-qd1)) : 0.f;
    float ow[kLaneBins], oh[kLaneBins], od[kLaneBins];
#pragma unroll
    for (int i = 0; i < kLaneBins; ++i) {
        const int j = kLaneBins * sub + i;
        const float sel_w = k20 * ((j < b ? gl : 0.f) + (j <= b ? gr : 0.f));
        const float sel_h = k20 * ((j < b ? gb : 0.f) + (j <= b ? gt : 0.f));
        ow[i] = out_scale * W.e[i] * (sel_w - dot_w);
        oh[i] = out_scale * H.e[i] * (sel_h - dot_h);
        od[i] = (j >= kBins - 1) ? 0.f : ((j == b - 1) ? v0 : ((j == b) ? v1 : 0.f));   // (j = 23: the padding slot of the row)
    }
    if (live) {
        float2 *pw = reinterpret_cast<float2 *>(q + kLaneBins * sub);
        float2 *ph = reinterpret_cast<float2 *>(q + kBins + kLaneBins * sub);
        float2 *pd = reinterpret_cast<float2 *>(q + 2 * kBins + kLaneBins * sub);
#pragma unroll
        for (int i = 0; i < kLaneBins / 2; ++i) {
            pw[i] = make_float2(ow[2 * i], ow[2 * i + 1]);
            ph[i] = make_float2(oh[2 * i], oh[2 * i + 1]);
            pd[i] = make_float2(od[2 * i], od[2 * i + 1]);
        }
    }
    if (inside) g = g_u;
}

// log p of every row (choice head + ten splines forward) and, when the gradient is wanted, the
// reverse sweep that leaves d loss / d (spline parameters, logits) where the values were.
__global__ void __launch_bounds__(kRowWarps * 32) train_rows_kernel(const float *__restrict__ params, Layout L,
                                                                    TrainRows rows, long long Rp, float scale,
                                                                    int backward, TrainBufs B)
{
    __shared__ float u_in[kRowWarps][kWarpRows][kTransforms];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int sub = lane & (kRowLanes - 1), base = lane & ~(kRowLanes - 1), rw = lane / kRowLanes;
    const long long row = ((long long)blockIdx.x * kRowWarps + wib) * kWarpRows + rw;
    const bool alloc = row < Rp;        // the row exists in the buffers (Rp is padded to whole tiles)
    const bool live = row < rows.R;     // ... and in the minibatch
    const int n_choices = L.n_choices;
    const long long rowc = alloc ? row : 0;
    float *lg = B.LG + (size_t)rowc * kMaxChoices;
    if (alloc && !live && backward) {   // padding rows of the last tile contribute nothing
        for (int k = 0; k < kTransforms; ++k)
            for (int j = sub; j < kSplineOut; j += kRowLanes) B.Q[((size_t)k * Rp + row) * kQRows + j] = 0.f;
        for (int j = sub; j < n_choices; j += kRowLanes) lg[j] = 0.f;
    }
    const long long dr = live ? data_row(rows, row) : 0;
    // categorical head: l = log clamp(softmax(logits)[choice], eps, 1 - eps); every lane of the row computes it
    float lp = 0.f;
    {
        const int choice = live ? (int)__ldg(rows.x + 2 * dr + 1) : 0;
        float logit[kMaxChoices];
        float m = -INFINITY;
#pragma unroll
        for (int j = 0; j < kMaxChoices; ++j) {
            logit[j] = (live && j < n_choices) ? lg[j] : -INFINITY;
            m = fmaxf(m, logit[j]);
        }
        float e[kMaxChoices], ssum = 0.f, ec = 0.f;
#pragma unroll
        for (int j = 0; j < kMaxChoices; ++j) {
            e[j] = (live && j < n_choices) ? expf(logit[j] - m) : 0.f;
            ssum += e[j];
            ec = (j == choice) ? e[j] : ec;
        }
        const float p = live ? ec / ssum : 0.5f;
        const float eps = 1.1920928955078125e-07f;
        lp = logf(fminf(fmaxf(p, eps), 1.0f - eps));
        if (backward) __syncwarp();   // every lane of the row has read the logits before any of them is overwritten
        if (backward && live) {
            const bool clamped = p < eps || p > 1.0f - eps;  // torch.clamp passes no gradient outside
#pragma unroll
            for (int j = 0; j < kMaxChoices; ++j)
                if (j < n_choices && (j & (kRowLanes - 1)) == sub)
                    lg[j] = clamped ? 0.f : scale * ((j == choice ? 1.0f : 0.f) - e[j] / ssum);
        }
    }
    const float mu_y = params[L.mu_y], sigma_y = params[L.sigma_y];
    const float y = live ? logf(__ldg(rows.x + 2 * dr)) : 0.f;
    float u = (y - mu_y) / sigma_y;
    float logdet = -logf(sigma_y);
    float g = 0.f;
#pragma unroll 1
    for (int k = 0; k < kTransforms; ++k) {
        if (sub == 0) u_in[wib][rw][k] = u;
        rqs_quad<false>(u, logdet, B.Q + ((size_t)k * Rp + rowc) * kQRows, base, sub, live, g, scale);
    }
    if (sub == 0 && live) B.LP[row] = lp + (-0.5f * u * u - 0.9189385332046727f) + logdet - y;
    if (!backward) return;
    __syncwarp();
    g = -u;  // d/du of the standard-normal base log-density
#pragma unroll 1
    for (int k = kTransforms - 1; k >= 0; --k) {
        float uk = u_in[wib][rw][k];
        rqs_quad<true>(uk, logdet, B.Q + ((size_t)k * Rp + rowc) * kQRows, base, sub, live, g, scale);
    }
}

// ---- 3. backward through the nets ------------------------------------------------------------
// 3a. backward-data on CUDA cores: one CTA per (row tile, net) turns d loss / d (net outputs) into
// d loss / d (hidden pre-activations), layer by layer (transposed dense products with the activation
// derivative fused into the epilogue), and writes them out for the weight-gradient GEMMs.
__global__ void __launch_bounds__(kThreads) train_backward_kernel(const float *__restrict__ params, Layout L,
                                                                  long long Rp, TrainBufs B)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    SimtSmem &S = *reinterpret_cast<SimtSmem *>(smem_raw);
    const int net = blockIdx.y;  // 0 = categorical head, 1 + k = conditioner of transform k
    const long long row0 = (long long)blockIdx.x * kTM;
    if (net > 0) {
        const int k = net - 1;
        load_rows(B.Q + (size_t)k * kQRows * Rp, kQRows, row0, kSplineOut, S.in);
        load_hidden(S.hb, B.H, Rp, net, 1, row0);
        dense<8, kMaskRelu, false, true>(params + L.fl_W3[k], nullptr, kSplineOut, kHidden, S.in, kLdIn, S.hb, kLdH, S.w,
                                         kHidden);
        save_hidden(S.hb, B.DH, Rp, net, 1, row0);
        load_hidden(S.ha, B.H, Rp, net, 0, row0);
        dense<8, kMaskRelu, false, true>(params + L.fl_W2[k], nullptr, kHidden, kHidden, S.hb, kLdH, S.ha, kLdH, S.w,
                                         kHidden);
        save_hidden(S.ha, B.DH, Rp, net, 0, row0);
    } else {
        load_rows(B.LG, kMaxChoices, row0, L.n_choices, S.in);
        load_hidden(S.ha, B.H, Rp, 0, 2, row0);
        dense<8, kMaskSigmoid, false, true>(params + L.cat_Wo, nullptr, L.n_choices, kHidden, S.in, kLdIn, S.ha, kLdH,
                                            S.w, kHidden);
        save_hidden(S.ha, B.DH, Rp, 0, 2, row0);
        load_hidden(S.hb, B.H, Rp, 0, 1, row0);
        dense<8, kMaskSigmoid, false, true>(params + L.cat_W2, nullptr, kHidden, kHidden, S.ha, kLdH, S.hb, kLdH, S.w,
                                            kHidden);
        save_hidden(S.hb, B.DH, Rp, 0, 1, row0);
        __syncthreads();  // everyone is done with the gradient in S.ha before the activations replace it
        load_hidden(S.ha, B.H, Rp, 0, 0, row0);
        dense<8, kMaskSigmoid, false, true>(params + L.cat_W1, nullptr, kHidden, kHidden, S.hb, kLdH, S.ha, kLdH, S.w,
                                            kHidden);
        save_hidden(S.ha, B.DH, Rp, 0, 0, row0);
    }
}

// 3b. weight gradients on the tensor cores.  Every layer's dW[m][n] = sum_r dY[r][m] * X[r][n] is a GEMM
// whose reduction runs over the rows of the minibatch: M, N <= 128, K = R.  One CTA owns one (layer, row
// split): per 64-row chunk, threads (c, half) of the first eight warps turn 32 rows of column c of dY into
// row c of a K-major bf16 hi / lo operand image (one 16-byte shared-memory store per 8 rows), the other
// eight warps do the same for X, and one elected thread issues the three tcgen05.mma passes (hi*hi +
// hi*lo + lo*hi, fp32 accumulation in tensor memory across all chunks).  The row splits write separate
// slices of the partial buffer: the fixed-order reduction below sums them.
struct WJob {
    const float *A;     // dY: (R, lda) row-major, M columns used
    const float *B;     // X:  (R, ldb) row-major, N columns used; nullptr = the (gathered) context rows
    int lda, ldb, M, N;     // lda / ldb = 0: the operand is stored column-major with Rp rows per column
    unsigned w_off, b_off;  // where dW (M x N, row-major) and db (M) go in a partial slice
};
constexpr int kMaxWJobs = 3 * kTransforms + 4;
struct WJobs {
    WJob j[kMaxWJobs];
};
constexpr int kWgThreads = 512;                  // 2 operands x 128 columns x 2 halves of the chunk's rows
static_assert(kWgRows == 64, "thread mapping below: 32 rows (four 8-row K groups) per thread and chunk");
// K-major images with the stride between 8-row K groups padded by 32 bytes (the UMMA descriptor's LBO is free):
// the eight lanes that share a column write four K groups at once, and without the pad those land in the same
// banks
constexpr uint32_t kWgPad = 32;
constexpr uint32_t kWgImg = (kWgRows / 8) * (128 * 16 + kWgPad);   // one 128 x kWgRows bf16 image
constexpr uint32_t kWgSmem = 4 * kWgImg + 64 + 2 * kWgRows * 8;
static_assert(4 * kWgImg >= 128 * 128 * 4, "the epilogue stages the 128 x 128 fp32 tile in the image area");

__global__ void __launch_bounds__(kWgThreads, 2) train_wgrad_tc_kernel(const __grid_constant__ WJobs jobs, TrainRows rows,
                                                                       long long Rp, int chunks_total, size_t total,
                                                                       float *__restrict__ P)
{
    using namespace tc;
    extern __shared__ __align__(1024) unsigned char smem[];
    uint64_t *bar = reinterpret_cast<uint64_t *>(smem + 4 * kWgImg);
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(smem + 4 * kWgImg + 16);
    long long *drow = reinterpret_cast<long long *>(smem + 4 * kWgImg + 64);  // [2][kWgRows] dataset row of each chunk row
    const WJob &J = jobs.j[blockIdx.x];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int c_begin = (int)((long long)chunks_total * blockIdx.y / gridDim.y);
    const int c_end = (int)((long long)chunks_total * (blockIdx.y + 1) / gridDim.y);
    const int n_pad = (J.N + 15) & ~15;  // UMMA N

    if (warp == 0) tmem_alloc<128>(tmem_slot);
    if (tid == 0) {
        mbar_init(bar, 1);
        fence_mbar_init();
    }

    // thread = (operand, half of the chunk's rows, column): 32 independent rows in flight per thread -- the
    // operands come from HBM (they do not fit L2 next to each other).  The loads of chunk c + 1 are issued
    // before the wait for the tensor core to finish chunk c, so that one chunk costs max(load, MMA) + the
    // conversion instead of their sum; the dataset rows of the gathered context operand are fetched one
    // chunk further ahead still.
    const bool is_a = tid < 256;
    const int half = (tid >> 7) & 1, col = tid & 127;
    const int img_rows = is_a ? 128 : n_pad, valid = is_a ? J.M : J.N;
    const bool is_ctx = !is_a && J.B == nullptr;
    const float *src = is_a ? J.A : J.B;
    const long long ld = is_a ? J.lda : J.ldb;
    unsigned char *img_hi = smem + (is_a ? 0u : 2u * kWgImg), *img_lo = img_hi + kWgImg;
    const int rr0 = 32 * half;  // first row of the chunk this thread converts (row-major / gathered operands)
    const bool colmajor = !is_ctx && ld == 0;
    const int wq = (tid & 255) >> 5, q = tid & 7, cs = (tid >> 3) & 3;  // column-major operands: see load_chunk
    float v[32];

    auto chunk_row = [&](int c) -> long long {  // dataset row of chunk row `tid` (tid < kWgRows)
        const long long r = (long long)c * kWgRows + tid;
        return (c < c_end && r < rows.R) ? data_row(rows, r) : 0;
    };
    auto load_chunk = [&](int c, const long long *dr) {
        const long long r0 = (long long)c * kWgRows;
        const int n_rows = (int)(rows.R - r0 < kWgRows ? rows.R - r0 : kWgRows);
        if (colmajor) {
            // column-major operand: load i of the warp covers rows [32 h, 32 h + 32) of four columns, eight
            // lanes (16 bytes each) per column = four whole 128-byte lines per request.  (One thread per
            // column with its 32 rows contiguous asked for 32 different lines per request: same bytes, but
            // the kernel then ran at 1.8 TB/s, bound by the tag stage of L1.)
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int cq = 16 * wq + 4 * (i >> 1) + cs, rr = 32 * (i & 1) + 4 * q;
                float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
                if (cq < valid && r0 + rr + 3 < Rp) t = *reinterpret_cast<const float4 *>(src + (size_t)cq * Rp + r0 + rr);
                v[4 * i + 0] = rr + 0 < n_rows ? t.x : 0.f;
                v[4 * i + 1] = rr + 1 < n_rows ? t.y : 0.f;
                v[4 * i + 2] = rr + 2 < n_rows ? t.z : 0.f;
                v[4 * i + 3] = rr + 3 < n_rows ? t.w : 0.f;
            }
        } else if (col < img_rows) {
#pragma unroll
            for (int e = 0; e < 32; ++e) {
                const int rr = rr0 + e;  // row within the chunk
                float x = 0.f;
                if (col < valid && rr < n_rows) {
                    if (!is_ctx) x = src[(size_t)(r0 + rr) * ld + col];
                    else x = col == kCond ? __ldg(rows.x + 2 * dr[rr] + 1) : __ldg(rows.cond + dr[rr] * rows.ld_cond + col);
                }
                v[e] = x;
            }
        }
    };

    long long drow_next = 0;
    if (tid < kWgRows) {
        drow[tid] = chunk_row(c_begin);
        drow_next = chunk_row(c_begin + 1);
    }
    tc_fence_before_sync();
    __syncthreads();
    tc_fence_after_sync();
    const uint32_t tmem = *tmem_slot;
    if (c_begin < c_end) load_chunk(c_begin, drow);

    float bias_acc = 0.f, bias4[4] = {0.f, 0.f, 0.f, 0.f};
    uint32_t phase = 0;
    for (int c = c_begin; c < c_end; ++c) {
        long long *dr_next = drow + (((c - c_begin) & 1) ^ 1) * kWgRows;
        if (tid < kWgRows) {
            dr_next[tid] = drow_next;  // rows of chunk c + 1: visible after the barrier below
            drow_next = chunk_row(c + 2);
        }
        if (colmajor) {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int cq = 16 * wq + 4 * (i >> 1) + cs;
                if (cq < img_rows) {
                    uint32_t hi[2], lo[2];
                    split_bf16x2(v[4 * i], v[4 * i + 1], hi[0], lo[0]);
                    split_bf16x2(v[4 * i + 2], v[4 * i + 3], hi[1], lo[1]);
                    if (is_a) bias4[i >> 1] += (v[4 * i] + v[4 * i + 1]) + (v[4 * i + 2] + v[4 * i + 3]);
                    // K group = 8 rows: rows 32 (i & 1) + 4 q .. + 3 are half q & 1 of group 4 (i & 1) + q / 2
                    const uint32_t off = (uint32_t)(4 * (i & 1) + (q >> 1)) * ((uint32_t)img_rows * 16u + kWgPad) +
                                         (uint32_t)cq * 16u + (uint32_t)(q & 1) * 8u;
                    *reinterpret_cast<uint2 *>(img_hi + off) = make_uint2(hi[0], hi[1]);
                    *reinterpret_cast<uint2 *>(img_lo + off) = make_uint2(lo[0], lo[1]);
                }
            }
        } else if (col < img_rows) {
#pragma unroll
            for (int g = 0; g < 4; ++g) {
                uint32_t hi[4], lo[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) split_bf16x2(v[8 * g + 2 * j], v[8 * g + 2 * j + 1], hi[j], lo[j]);
                if (is_a)
                    bias_acc += ((v[8 * g] + v[8 * g + 1]) + (v[8 * g + 2] + v[8 * g + 3])) +
                                ((v[8 * g + 4] + v[8 * g + 5]) + (v[8 * g + 6] + v[8 * g + 7]));
                const uint32_t off = (uint32_t)(4 * half + g) * ((uint32_t)img_rows * 16u + kWgPad) + (uint32_t)col * 16u;
                *reinterpret_cast<uint4 *>(img_hi + off) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
                *reinterpret_cast<uint4 *>(img_lo + off) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
            }
        }
        fence_proxy_async_smem();
        tc_fence_before_sync();
        __syncthreads();
        tc_fence_after_sync();
        if (warp == 0) {
            if (elect_one_sync()) {
                const uint32_t idesc = umma_idesc_bf16_f32(128, n_pad);
                const uint32_t a0 = smem_u32(smem), b0 = smem_u32(smem + 2 * kWgImg);
                const uint32_t lbo_a = 128u * 16u + kWgPad, lbo_b = (uint32_t)n_pad * 16u + kWgPad;
#pragma unroll
                for (int pass = 0; pass < 3; ++pass) {
                    const uint32_t pa = a0 + (pass == 2 ? kWgImg : 0u), pb = b0 + (pass == 1 ? kWgImg : 0u);
#pragma unroll
                    for (int ks = 0; ks < kWgRows / 16; ++ks)
                        umma_bf16(tmem, umma_desc_kmajor(pa + ks * 2 * lbo_a, lbo_a, 128),
                                  umma_desc_kmajor(pb + ks * 2 * lbo_b, lbo_b, 128), idesc,
                                  (c > c_begin) || (pass | ks) != 0);
                }
                umma_commit(bar);
            }
            __syncwarp();
        }
        if (c + 1 < c_end) load_chunk(c + 1, dr_next);  // in flight while the tensor core works
        mbar_wait(bar, phase);  // the images may be rebuilt once the tensor core has read them
        phase ^= 1;
        tc_fence_after_sync();
    }
    // the two halves of a dY column add up their bias sums (fixed order)
    float *tile = reinterpret_cast<float *>(smem);  // the images are dead
    __syncthreads();
    if (is_a && !colmajor && half == 1) tile[col] = bias_acc;
    __syncthreads();
    if (is_a && !colmajor && half == 0) bias_acc += tile[col];
    __syncthreads();
    // accumulators -> shared memory (lane m of tensor memory = row m of dW; warp w reads lane group w % 4,
    // columns 32 * (w / 4) ..; XOR swizzle against bank conflicts) -> this split's slice, coalesced
    float *Pout = P + (size_t)blockIdx.y * total;
    {
        const int m = 32 * (warp & 3) + lane, n0 = 32 * (warp >> 2);
        if (n0 < n_pad) {
            uint32_t a[32];
            if (c_end > c_begin) {
                tmem_ld32(tmem + ((uint32_t)(32 * (warp & 3)) << 16) + (uint32_t)n0, a);
                tmem_wait_ld();
            } else {
#pragma unroll
                for (int j = 0; j < 32; ++j) a[j] = 0u;
            }
#pragma unroll
            for (int j = 0; j < 32; ++j) tile[m * 128 + ((n0 + j) ^ lane)] = __uint_as_float(a[j]);
        }
        if (is_a && colmajor) {  // eight lanes share a column: fixed-order butterfly, lane q = 0 writes
#pragma unroll
            for (int cg = 0; cg < 4; ++cg) {
                float b = bias4[cg];
                b += __shfl_xor_sync(0xFFFFFFFFu, b, 1);
                b += __shfl_xor_sync(0xFFFFFFFFu, b, 2);
                b += __shfl_xor_sync(0xFFFFFFFFu, b, 4);
                const int cq = 16 * wq + 4 * cg + cs;
                if (q == 0 && cq < J.M) Pout[J.b_off + cq] = b;
            }
        } else if (tid < 128 && tid < J.M) {
            Pout[J.b_off + tid] = bias_acc;  // (tid < 128: operand A, half 0, col = tid)
        }
    }
    tc_fence_before_sync();
    __syncthreads();
    for (int m = warp; m < J.M; m += kWgThreads / 32)
        for (int n = lane; n < J.N; n += 32) Pout[J.w_off + (size_t)m * J.N + n] = tile[m * 128 + (n ^ (m & 31))];
    if (warp == 0) tmem_dealloc<128>(tmem);
}

// ---- 4. fixed-order reductions ---------------------------------------------------------------
__device__ __forceinline__ float block_sum(float v, float *red)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    float t = 0.f;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += red[w];
    return t;
}

__global__ void __launch_bounds__(kReduceThreads) train_reduce_kernel(const float *__restrict__ P, int groups,
                                                                      size_t total, size_t n_trainable,
                                                                      float *__restrict__ grad, float *__restrict__ SS)
{
    __shared__ float red[kReduceThreads / 32];
    const size_t i = (size_t)blockIdx.x * kReduceThreads + threadIdx.x;
    float g = 0.f;
    if (i < n_trainable)
        for (int s = 0; s < groups; ++s) g += P[(size_t)s * total + i];
    if (i < total) grad[i] = g;  // the log rt standardisation (tail of the buffer) is not trained
    const float t = block_sum(g * g, red);
    if (threadIdx.x == 0) SS[blockIdx.x] = t;
}

// stats[0] = loss = -mean log p, stats[1] = |grad|^2 (0 when no gradient was asked for)
__global__ void __launch_bounds__(1024) train_stats_kernel(const float *__restrict__ LP, long long R,
                                                           const float *__restrict__ SS, int n_ss,
                                                           float *__restrict__ stats)
{
    __shared__ float red[32];
    float v = 0.f;
    for (long long r = threadIdx.x; r < R; r += blockDim.x) v += LP[r];
    const float sum_lp = block_sum(v, red);
    v = 0.f;
    for (int b = threadIdx.x; b < n_ss; b += blockDim.x) v += SS[b];
    const float ss = block_sum(v, red);
    if (threadIdx.x == 0) {
        stats[0] = -sum_lp / (float)R;
        stats[1] = ss;
    }
}

// ---- 5. Adam (torch.optim.Adam defaults: no weight decay, no amsgrad) with clip_grad_norm_ ------
__global__ void __launch_bounds__(256) adam_kernel(float *__restrict__ params, const float *__restrict__ grad,
                                                   float *__restrict__ m, float *__restrict__ v, size_t n,
                                                   const float *__restrict__ stats, float lr, float beta1, float beta2,
                                                   float eps, float bc1, float bc2_sqrt, float max_norm)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float clip = 1.0f;
    if (max_norm > 0.f) {
        const float norm = sqrtf(stats[1]);
        clip = fminf(max_norm / (norm + 1e-6f), 1.0f);  // torch.nn.utils.clip_grad_norm_
    }
    const float g = grad[i] * clip;
    const float mi = beta1 * m[i] + (1.0f - beta1) * g;
    const float vi = beta2 * v[i] + (1.0f - beta2) * g * g;
    m[i] = mi;
    v[i] = vi;
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    params[i] -= (lr / bc1) * (mi / denom);
}

}  // namespace mnle

using namespace mnle;

DDM_API size_t mnle_train_workspace_floats(int n_choices, int64_t R)
{
    if (n_choices < 1 || n_choices > kMaxChoices || R <= 0) return 0;
    const Layout L = make_layout(n_choices);
    Carver ws(nullptr);
    train_workspace(ws, L, train_dims(L, R));
    return ws.floats();
}

DDM_API int mnle_train_nll_grad_f32(const float *params_dev, int n_choices, const float *x_dev, const float *cond_dev,
                                    int64_t ld_cond, const int64_t *row_index_dev, int64_t R, float *stats_dev,
                                    float *grad_dev, float *workspace_dev, int flags, void *stream)
{
    DDM_REQUIRE(n_choices >= 1 && n_choices <= kMaxChoices, "mnle_train_nll_grad_f32: n_choices=%d outside [1,%d]",
                n_choices, kMaxChoices);
    DDM_REQUIRE(R >= 1 && R <= 0x7FFFFFFFll * kTM / 2, "mnle_train_nll_grad_f32: R=%lld out of range", (long long)R);
    DDM_REQUIRE(params_dev && x_dev && cond_dev && stats_dev && workspace_dev,
                "mnle_train_nll_grad_f32: null pointer");
    DDM_REQUIRE(ld_cond >= kCond, "mnle_train_nll_grad_f32: ld_cond=%lld < 85", (long long)ld_cond);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const Layout L = make_layout(n_choices);
    const TrainDims d = train_dims(L, R);
    Carver ws(workspace_dev);
    const TrainBufs B = train_workspace(ws, L, d);
    TrainRows rows{x_dev, cond_dev, reinterpret_cast<const long long *>(row_index_dev), (long long)ld_cond, (long long)R};

    static_assert(sizeof(SimtSmem) < 113 * 1024, "two CTAs per SM");
    const int want_grad = grad_dev != nullptr;
    // the gathered context rows as fp32 columns (written by the tensor-core forward's prep kernel, read by the
    // weight-gradient GEMMs of the first layers): the flow nets keep two hidden layers, so slot 2 of net 1 is free
    float *ctx_cols = B.H + (size_t)(1 * 3 + 2) * kHidden * (size_t)d.Rp;
    if (flags & DDM_TRAIN_FP32_FORWARD) {
        DDM_CUDA_TRY(cudaFuncSetAttribute(train_forward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          (int)sizeof(SimtSmem)));
        train_forward_kernel<<<dim3(d.tiles, kNets), kThreads, sizeof(SimtSmem), st>>>(params_dev, L, rows, d.Rp, B, 1);
        DDM_CUDA_TRY(cudaGetLastError());
    } else {  // forward on the tensor cores (mnle_tc.cu), keeping logits, spline parameters and activations
        const TcTrainDump keep{B.H, B.Q, B.LG, d.Rp, nullptr, nullptr, want_grad ? ctx_cols : nullptr};
        const int rc = tc_train_forward(params_dev, L, B.pack, x_dev, cond_dev, (long long)ld_cond,
                                        reinterpret_cast<const long long *>(row_index_dev), (long long)R, keep, B.LP, st);
        if (rc != DDM_OK) return rc;
    }
    train_rows_kernel<<<(unsigned)((d.Rp + kBlockRows - 1) / kBlockRows), kRowWarps * 32, 0, st>>>(
        params_dev, L, rows, d.Rp, -1.0f / (float)R, want_grad, B);
    DDM_CUDA_TRY(cudaGetLastError());
    int n_ss = 0;
    if (want_grad) {
        DDM_CUDA_TRY(cudaFuncSetAttribute(train_backward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          (int)sizeof(SimtSmem)));
        if (flags & DDM_TRAIN_FP32_FORWARD) {  // the fp32 anchor keeps the whole chain on the CUDA cores
            train_backward_kernel<<<dim3(d.tiles, kNets), kThreads, sizeof(SimtSmem), st>>>(params_dev, L, d.Rp, B);
            DDM_CUDA_TRY(cudaGetLastError());
        } else {  // backward-data on the tensor cores (transposed weight images of the pack built above)
            const TcTrainDump bwd{B.H, B.Q, B.LG, d.Rp, B.DH, nullptr};
            const int rc = tc_train_backward(L, B.pack, (long long)R, bwd, st);
            if (rc != DDM_OK) return rc;
        }
        // weight-gradient GEMMs: (dY, X) of every layer
        WJobs jobs;
        int nj = 0;
        const size_t hs = (size_t)d.Rp * kHidden;  // one [Rp][128] activation block
        auto H = [&](int net, int slot) { return B.H + ((size_t)net * 3 + slot) * hs; };
        auto DH = [&](int net, int slot) { return B.DH + ((size_t)net * 3 + slot) * hs; };
        auto add = [&](const float *A, int lda, int M, const float *Bm, int ldb, int N, size_t w_off, size_t b_off) {
            jobs.j[nj++] = WJob{A, Bm, lda, ldb, M, N, (unsigned)w_off, (unsigned)b_off};
        };
        add(B.LG, kMaxChoices, n_choices, H(0, 2), 0, kHidden, L.cat_Wo, L.cat_bo);
        add(DH(0, 2), 0, kHidden, H(0, 1), 0, kHidden, L.cat_W2, L.cat_b2);
        add(DH(0, 1), 0, kHidden, H(0, 0), 0, kHidden, L.cat_W1, L.cat_b1);
        const float *ctx_x = (flags & DDM_TRAIN_FP32_FORWARD) ? nullptr : ctx_cols;  // nullptr: gather from the dataset
        add(DH(0, 0), 0, kHidden, ctx_x, 0, kCond, L.cat_W0, L.cat_b0);
        for (int k = 0; k < kTransforms; ++k) {
            const int net = 1 + k;
            add(B.Q + (size_t)k * kQRows * d.Rp, kQRows, kSplineOut, H(net, 1), 0, kHidden, L.fl_W3[k], L.fl_b3[k]);
            add(DH(net, 1), 0, kHidden, H(net, 0), 0, kHidden, L.fl_W2[k], L.fl_b2[k]);
            add(DH(net, 0), 0, kHidden, ctx_x, 0, kCtx, L.fl_W1[k], L.fl_b1[k]);
        }
        DDM_CUDA_TRY(cudaFuncSetAttribute(train_wgrad_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kWgSmem));
        train_wgrad_tc_kernel<<<dim3(nj, d.groups), kWgThreads, kWgSmem, st>>>(jobs, rows, d.Rp, (int)((R + kWgRows - 1) / kWgRows), L.total,
                                                                             B.P);
        DDM_CUDA_TRY(cudaGetLastError());
        train_reduce_kernel<<<d.reduce_blocks, kReduceThreads, 0, st>>>(B.P, d.groups, L.total, L.mu_y, grad_dev, B.SS);
        DDM_CUDA_TRY(cudaGetLastError());
        n_ss = d.reduce_blocks;
    }
    train_stats_kernel<<<1, 1024, 0, st>>>(B.LP, (long long)R, B.SS, n_ss, stats_dev);
    DDM_CUDA_TRY(cudaGetLastError());
    return DDM_OK;
}

DDM_API int mnle_train_adam_f32(float *params_dev, const float *grad_dev, float *m_dev, float *v_dev, int n_choices,
                                const float *stats_dev, float lr, float beta1, float beta2, float eps, int64_t step,
                                float max_grad_norm, void *stream)
{
    DDM_REQUIRE(n_choices >= 1 && n_choices <= kMaxChoices, "mnle_train_adam_f32: n_choices=%d outside [1,%d]",
                n_choices, kMaxChoices);
    DDM_REQUIRE(params_dev && grad_dev && m_dev && v_dev, "mnle_train_adam_f32: null pointer");
    DDM_REQUIRE(step >= 1, "mnle_train_adam_f32: step counts from 1, got %lld", (long long)step);
    DDM_REQUIRE(max_grad_norm <= 0.f || stats_dev != nullptr, "mnle_train_adam_f32: clipping needs stats_dev");
    const Layout L = make_layout(n_choices);
    const size_t n = L.mu_y;  // everything before the (fixed) log rt standardisation
    const float bc1 = 1.0f - powf(beta1, (float)step);
    const float bc2_sqrt = sqrtf(1.0f - powf(beta2, (float)step));
    adam_kernel<<<(unsigned)((n + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        params_dev, grad_dev, m_dev, v_dev, n, stats_dev, lr, beta1, beta2, eps, bc1, bc2_sqrt, max_grad_norm);
    DDM_CUDA_TRY(cudaGetLastError());
    return DDM_OK;
}

// ---- potential: value and d/d theta in reverse mode on the tensor cores (row f2) ------------------------
// What autograd does for the reference's NUTS (potentials.py:112 with track_gradients=True), with the training
// step's kernels: the (T*C, 85) rows of the reference's expansion (row r = t*C + c) go through the tcgen05
// forward (activations kept), the per-row spline sweep leaves d log p / d (spline parameters, logits), the
// tcgen05 backward-data pass turns them into d log p / d (first-layer pre-activations), and only the five theta
// columns of every first layer are contracted: grad[c][i] = sum_t sum_net sum_j DH[net][0][j][t*C+c] W1_net[j][i].
namespace mnle {

// Ragged sessions (offsets != null, D + 1 entries): t is the flat trial, and its rows take the chains of its session,
// theta row session_of(t) * C + c.
__global__ void __launch_bounds__(256) potential_rows_kernel(const float *__restrict__ theta, long long ld_theta,
                                                             const float *__restrict__ x, const float *__restrict__ pulses,
                                                             long long ld_pulses, int T, int C, float *__restrict__ cond,
                                                             float *__restrict__ xr, const long long *__restrict__ offsets = nullptr,
                                                             int D = 1)
{
    const long long total = (long long)T * C * kCond;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const long long r = idx / kCond;
        const int j = (int)(idx - r * kCond);
        const int t = (int)(r / C), c = (int)(r - (long long)t * C);
        if (j < 5) {
            const long long th_row = offsets != nullptr ? (long long)session_of(offsets, D, t) * C + c : c;
            cond[idx] = __ldg(theta + th_row * ld_theta + j);
        } else {
            cond[idx] = __ldg(pulses + (long long)t * ld_pulses + (j - 5));
        }
        if (j < 2) xr[2 * r + j] = __ldg(x + 2 * t + j);
    }
}

// the five theta columns of every first layer, [kNets][128][8] (three zeros of padding): what the backward kernel's
// last epilogue contracts the first-layer derivatives with
__global__ void __launch_bounds__(128) potential_w1_kernel(const float *__restrict__ params, Layout L, float *__restrict__ w1t)
{
    const int net = blockIdx.x, j = threadIdx.x;
    const int K = net == 0 ? kCond : kCtx;
    const float *W = params + (net == 0 ? L.cat_W0 : L.fl_W1[net - 1]);
#pragma unroll
    for (int i = 0; i < 8; ++i) w1t[((size_t)net * kHidden + j) * 8 + i] = i < 5 ? __ldg(W + (size_t)j * K + i) : 0.f;
}

constexpr int kGradPlanes = kNets * 2;   // (net, column half) partial gradients per row, written by the backward kernel

// grid (chain blocks of 128, planes): part[(plane * C + c) * 5 + i] = sum_t GP[plane][i][t * C + c]  (fixed order)
__global__ void __launch_bounds__(128) potential_grad_partial_kernel(const float *__restrict__ GP, long long Rp, int T, int C,
                                                                     float *__restrict__ part)
{
    const int plane = blockIdx.y, c = blockIdx.x * 128 + threadIdx.x;
    if (c >= C) return;
    const float *src = GP + (size_t)plane * 5 * (size_t)Rp + c;
    float acc[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
    for (int t = 0; t < T; ++t) {
#pragma unroll
        for (int i = 0; i < 5; ++i) acc[i] += __ldcg(src + (size_t)i * Rp + (size_t)t * C);
    }
    float *dst = part + ((size_t)plane * C + c) * 5;
#pragma unroll
    for (int i = 0; i < 5; ++i) dst[i] = acc[i];
}

__global__ void __launch_bounds__(128) potential_grad_final_kernel(const float *__restrict__ part, const float *__restrict__ LP, int T,
                                                                   int C, float *__restrict__ out, float *__restrict__ grad)
{
    const int c = blockIdx.x * 128 + threadIdx.x;
    if (c >= C) return;
    float acc[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
    for (int s = 0; s < kGradPlanes; ++s)
#pragma unroll
        for (int i = 0; i < 5; ++i) acc[i] += part[((size_t)s * C + c) * 5 + i];
#pragma unroll
    for (int i = 0; i < 5; ++i) grad[(size_t)c * 5 + i] = acc[i];
    float sum = 0.f;
    for (int t = 0; t < T; ++t) sum += LP[(size_t)t * C + c];
    out[c] = sum;
}

// Only what the passes above read or write: no DH (the backward pass keeps no derivatives), no weight-gradient
// partials, and activations of the categorical net's three sigmoid layers alone (the ReLU layers keep sign masks).
struct PotentialGradBufs {
    TrainBufs t;   // pack, Q, LG, LP; H, DH, P and SS stay null (train_rows_kernel reads only Q, LG and LP)
    float *cond, *xr, *w1t, *gp, *part;
    uint32_t *HM;  // [kNets][3][4][Rp] sign masks of the ReLU layers
    float *H;      // [3][128][Rp] activations of the categorical net (net 0 of TcTrainDump::H)
};

static PotentialGradBufs potential_grad_workspace(Carver &ws, const Layout &L, const TrainDims &d, long long C)
{
    PotentialGradBufs b{};
    b.t.pack = ws.take<unsigned char>(tc_train_pack_bytes(L.n_choices, d.R));
    b.t.Q = ws.take((size_t)kTransforms * kQRows * d.Rp);
    b.t.LG = ws.take((size_t)kMaxChoices * d.Rp);
    b.t.LP = ws.take(d.Rp);
    b.cond = ws.take((size_t)d.R * kCond);            // the expanded rows
    b.xr = ws.take(2 * (size_t)d.R);
    b.w1t = ws.take((size_t)kNets * kHidden * 8);       // theta columns of the first layers
    b.gp = ws.take((size_t)kGradPlanes * 5 * (size_t)d.Rp);  // per-row partial gradients
    b.part = ws.take((size_t)kGradPlanes * (size_t)C * 5);   // per-chain partial gradients
    b.HM = ws.take<uint32_t>((size_t)kNets * 3 * 4 * (size_t)d.Rp);
    // H last: the kernels address it as TcTrainDump::H, whose slots span all eleven nets, and only net 0's are carved.
    // The ReLU nets keep sign masks in HM instead and the backward pass never reads their slots; were that wrong, their
    // writes would land past the end of the workspace, where a guard band after the caller's buffer shows them.
    b.H = ws.take((size_t)3 * kHidden * d.Rp);
    return b;
}

// The argument checks and empty cases of the potentials over expanded (trial, chain) rows.  *H is set when there
// are rows to evaluate; otherwise the return value is final: an error, or DDM_OK when C == 0, or when T == 0 once out_dev
// (n_sets * C: one sum per dataset and chain) and (want_grad) grad_dev are zeroed.
static int expanded_rows_prologue(const char *entry, Handle **H, void *handle, const float *theta_dev, int64_t ld_theta,
                                  const float *x_dev, const float *pulses_dev, int64_t ld_pulses, int64_t T, int64_t C,
                                  float *out_dev, bool want_grad, float *grad_dev, const float *workspace_dev,
                                  cudaStream_t st, int64_t n_sets = 1)
{
    *H = nullptr;
    Handle *h = live_handle(handle, entry);
    if (h == nullptr) return DDM_ERR_STATE;
    DDM_REQUIRE(T >= 0 && C >= 0 && T * C <= 8000000ll, "%s: T=%lld x C=%lld rows (at most 8e6 per call)", entry, (long long)T,
                (long long)C);
    if (C == 0) return DDM_OK;
    DDM_REQUIRE(out_dev && (grad_dev || !want_grad), "%s: null output", entry);
    if (T == 0) {
        DDM_CUDA_TRY(cudaMemsetAsync(out_dev, 0, (size_t)n_sets * (size_t)C * sizeof(float), st));
        if (want_grad) DDM_CUDA_TRY(cudaMemsetAsync(grad_dev, 0, (size_t)C * 5 * sizeof(float), st));
        return DDM_OK;
    }
    DDM_REQUIRE(theta_dev && x_dev && pulses_dev && workspace_dev, "%s: null pointer", entry);
    DDM_REQUIRE(ld_theta >= 5 && ld_pulses >= kCond - 5, "%s: ld_theta=%lld ld_pulses=%lld too small", entry, (long long)ld_theta,
                (long long)ld_pulses);
    DDM_REQUIRE((reinterpret_cast<uintptr_t>(workspace_dev) & 255u) == 0, "%s: workspace must be 256-byte aligned", entry);
    *H = h;
    return DDM_OK;
}

}  // namespace mnle

DDM_API size_t mnle_loglik_grad_tc_workspace_floats(int n_choices, int64_t T, int64_t C)
{
    if (n_choices < 1 || n_choices > kMaxChoices || T <= 0 || C <= 0) return 0;
    const Layout L = make_layout(n_choices);
    Carver ws(nullptr);
    potential_grad_workspace(ws, L, train_dims(L, T * C), C);
    return ws.floats();
}

DDM_API int mnle_loglik_sum_grad_tc_f32(void *handle, const float *theta_dev, int64_t ld_theta, const float *x_dev,
                                        const float *pulses_dev, int64_t ld_pulses, int64_t T, int64_t C, float *out_dev,
                                        float *grad_dev, float *workspace_dev, void *stream)
{
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    Handle *H;
    int rc = expanded_rows_prologue("mnle_loglik_sum_grad_tc_f32", &H, handle, theta_dev, ld_theta, x_dev, pulses_dev, ld_pulses,
                                    T, C, out_dev, true, grad_dev, workspace_dev, st);
    if (H == nullptr) return rc;
    const Layout &L = H->layout;
    const long long R = T * C;
    const TrainDims d = train_dims(L, R);
    Carver ws(workspace_dev);
    const PotentialGradBufs B = potential_grad_workspace(ws, L, d, C);
    potential_w1_kernel<<<kNets, kHidden, 0, st>>>(H->params, L, B.w1t);
    DDM_CUDA_TRY(cudaGetLastError());
    potential_rows_kernel<<<(unsigned)std::min<long long>((R * kCond + 255) / 256, 148 * 16), 256, 0, st>>>(
        theta_dev, ld_theta, x_dev, pulses_dev, ld_pulses, (int)T, (int)C, B.cond, B.xr);
    DDM_CUDA_TRY(cudaGetLastError());
    TrainRows rows{B.xr, B.cond, nullptr, (long long)kCond, R};
    const TcTrainDump keep{B.H, B.t.Q, B.t.LG, d.Rp, nullptr, nullptr, nullptr, nullptr, nullptr, B.HM};
    rc = tc_train_forward(H->params, L, B.t.pack, B.xr, B.cond, (long long)kCond, nullptr, R, keep, B.t.LP, st);
    if (rc != DDM_OK) return rc;
    // scale = +1: the "loss" is the sum of the rows' log-probabilities
    train_rows_kernel<<<(unsigned)((d.Rp + kBlockRows - 1) / kBlockRows), kRowWarps * 32, 0, st>>>(H->params, L, rows, d.Rp, 1.0f, 1, B.t);
    DDM_CUDA_TRY(cudaGetLastError());
    // backward-data on tcgen05 without keeping the derivatives: the last epilogue of every net contracts d log p /
    // d (first-layer pre-activations) with the five theta columns of that layer and leaves five numbers per row
    const TcTrainDump bwd{B.H, B.t.Q, B.t.LG, d.Rp, nullptr, nullptr, nullptr, B.gp, B.w1t, B.HM};
    rc = tc_train_backward(L, B.t.pack, R, bwd, st);
    if (rc != DDM_OK) return rc;
    const unsigned cb = (unsigned)((C + 127) / 128);
    potential_grad_partial_kernel<<<dim3(cb, kGradPlanes), 128, 0, st>>>(B.gp, d.Rp, (int)T, (int)C, B.part);
    DDM_CUDA_TRY(cudaGetLastError());
    potential_grad_final_kernel<<<cb, 128, 0, st>>>(B.part, B.t.LP, (int)T, (int)C, out_dev, grad_dev);
    DDM_CUDA_TRY(cudaGetLastError());
    return DDM_OK;
}


// ---- potential: networks on the tensor cores, spline chain in fp64 ("tc64") ----------------------------
// On a trained estimator the fp32 rounding of the spline arithmetic, not of the networks, is what separates an
// fp32 evaluation from exact arithmetic (mnle_common.cuh::rqs_forward).  Here the tcgen05 rows-mode forward
// writes the raw spline parameters and choice logits of every (trial, chain) row, and one thread per row runs
// the ten splines, the categorical head and the final sum in fp64; the trials of a chain are added in fp64 in a
// fixed order.
namespace mnle {

// Four lanes per row, six bins per lane, like train_rows_kernel -- in fp64 and forward only: a lane evaluates 12 of a
// transform's 48 exponentials instead of all of them, and four times as many threads hide the latency of the fp64 chain.
__device__ __forceinline__ double quad_max(double v)
{
    v = fmax(v, __shfl_xor_sync(kFull, v, 1));
    return fmax(v, __shfl_xor_sync(kFull, v, 2));
}
__device__ __forceinline__ double pick6(const double (&v)[kLaneBins], int i)
{
    double r = v[0];
#pragma unroll
    for (int j = 1; j < kLaneBins; ++j) r = (i == j) ? v[j] : r;
    return r;
}
// knot edges lo / hi of the lane's six bins from the row's 24 logits (fp64 softmax and cumulative sum)
__device__ __forceinline__ void knots6_f64(const float (&logit)[kLaneBins], int base, int sub, double (&lo)[kLaneBins],
                                           double (&hi)[kLaneBins])
{
    const double inv_sqrt_h = 0.08838834764831844055, span = 1.0 - 1e-3 * kBins, tail = (double)kTail;
    double a[kLaneBins], m = -INFINITY;
#pragma unroll
    for (int i = 0; i < kLaneBins; ++i) {
        a[i] = (double)logit[i] * inv_sqrt_h;
        m = fmax(m, a[i]);
    }
    m = quad_max(m);
    double pre[kLaneBins], run = 0.0;
#pragma unroll
    for (int i = 0; i < kLaneBins; ++i) {
        run += exp(a[i] - m);
        pre[i] = run;
    }
    const double t0 = quad_get(run, base, 0), t1 = quad_get(run, base, 1), t2 = quad_get(run, base, 2), t3 = quad_get(run, base, 3);
    const double off = (sub > 0 ? t0 : 0.0) + (sub > 1 ? t1 : 0.0) + (sub > 2 ? t2 : 0.0);
    const double inv_s = 1.0 / (((t0 + t1) + t2) + t3);
#pragma unroll
    for (int i = 0; i < kLaneBins; ++i) {
        const int j = kLaneBins * sub + i;
        const double inc = (off + pre[i]) * inv_s;
        hi[i] = (j >= kBins - 1) ? tail : 2.0 * tail * (1e-3 * (double)(j + 1) + span * inc) - tail;
    }
    const double up = __shfl_up_sync(kFull, hi[kLaneBins - 1], 1);
    lo[0] = (sub == 0) ? -tail : up;
#pragma unroll
    for (int i = 1; i < kLaneBins; ++i) lo[i] = hi[i - 1];
}

// INVERSE (the sampler): u <- spline^-1(u), the bin located on the height knots and the rational quadratic solved for
// the position in the bin (nflows' rational_quadratic_spline(inverse=True)); logdet is not touched.
template <bool INVERSE = false>
__device__ __forceinline__ void rqs_quad_f64(double &u, double &logdet, const float *q, int base, int sub, bool live)
{
    const double tail = (double)kTail;
    const bool inside = (u >= -tail && u <= tail);
    const double ui = inside ? u : 0.0;
    float qw[kLaneBins], qh[kLaneBins], qd[kLaneBins];
    {
        const float2 *pw = reinterpret_cast<const float2 *>(q + kLaneBins * sub);
        const float2 *ph = reinterpret_cast<const float2 *>(q + kBins + kLaneBins * sub);
        const float2 *pd = reinterpret_cast<const float2 *>(q + 2 * kBins + kLaneBins * sub);
#pragma unroll
        for (int i = 0; i < kLaneBins / 2; ++i) {
            const float2 w2 = live ? pw[i] : make_float2(0.f, 0.f), h2 = live ? ph[i] : make_float2(0.f, 0.f);
            const float2 d2 = live ? pd[i] : make_float2(0.f, 0.f);
            qw[2 * i] = w2.x, qw[2 * i + 1] = w2.y, qh[2 * i] = h2.x, qh[2 * i + 1] = h2.y, qd[2 * i] = d2.x, qd[2 * i + 1] = d2.y;
        }
    }
    double wlo[kLaneBins], whi[kLaneBins], hlo[kLaneBins], hhi[kLaneBins];
    knots6_f64(qw, base, sub, wlo, whi);
    knots6_f64(qh, base, sub, hlo, hhi);
    int cnt = 0;
#pragma unroll
    for (int i = 0; i < kLaneBins; ++i) cnt += (ui >= (INVERSE ? hlo[i] : wlo[i])) ? 1 : 0;
    const int b = quad_sum(cnt) - 1;
    const int sb = (b >= kLaneBins ? 1 : 0) + (b >= 2 * kLaneBins ? 1 : 0) + (b >= 3 * kLaneBins ? 1 : 0), ib = b - kLaneBins * sb;
    const double left = quad_get(pick6(wlo, ib), base, sb), right = quad_get(pick6(whi, ib), base, sb);
    const double bottom = quad_get(pick6(hlo, ib), base, sb), top = quad_get(pick6(hhi, ib), base, sb);
    const int bm = b > 0 ? b - 1 : 0;
    const int sm = (bm >= kLaneBins ? 1 : 0) + (bm >= 2 * kLaneBins ? 1 : 0) + (bm >= 3 * kLaneBins ? 1 : 0), im = bm - kLaneBins * sm;
    const float qd0 = quad_get(pick6(qd, im), base, sm), qd1 = quad_get(pick6(qd, ib), base, sb);
    const double d0 = (b == 0) ? 1.0 : 1e-3 + softplus_f((double)qd0);
    const double d1 = (b == kBins - 1) ? 1.0 : 1e-3 + softplus_f((double)qd1);
    const double w = right - left, h = top - bottom;
    const double delta = h / w;
    if (INVERSE) {
        // a th^2 + b th + c = 0 for the position th in the bin; the root in [0, 1] in the cancellation-free form
        const double i1 = d0 + d1 - 2.0 * delta, i2 = ui - bottom, i3 = i2 * i1;
        const double qa = h * (delta - d0) + i3, qb = h * d0 - i3, qc = -delta * i2;
        const double disc = fmax(qb * qb - 4.0 * qa * qc, 0.0);
        const double root = (2.0 * qc) / (-qb - sqrt(disc));
        if (inside) u = root * w + left;
        return;
    }
    const double th = (ui - left) / w;
    const double t1 = th * (1.0 - th);
    const double den = delta + (d0 + d1 - 2.0 * delta) * t1;
    const double out = bottom + h * (delta * th * th + d0 * t1) / den;
    const double dnum = delta * delta * (d1 * th * th + 2.0 * delta * t1 + d0 * (1.0 - th) * (1.0 - th));
    if (inside) {
        logdet += log(dnum) - 2.0 * log(den);
        u = out;
    }
}

__global__ void __launch_bounds__(kRowWarps * 32) precise_rows_kernel(const float *__restrict__ Q, const float *__restrict__ LG, long long Rp,
                                                                      const float *__restrict__ xr, long long R, int n_choices, float mu_y,
                                                                      float sigma_y, double *__restrict__ LP)
{
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int sub = lane & (kRowLanes - 1), base = lane & ~(kRowLanes - 1), rw = lane / kRowLanes;
    const long long row = ((long long)blockIdx.x * kRowWarps + wib) * kWarpRows + rw;
    const bool live = row < R;
    const long long rowc = live ? row : 0;
    const float rt = live ? __ldg(xr + 2 * rowc) : 1.0f;
    const int choice = live ? (int)__ldg(xr + 2 * rowc + 1) : 0;
    const double y = log((double)rt);
    double u = (y - (double)mu_y) / (double)sigma_y, logdet = -log((double)sigma_y);
#pragma unroll 1
    for (int k = 0; k < kTransforms; ++k) rqs_quad_f64(u, logdet, Q + ((size_t)k * Rp + rowc) * kQRows, base, sub, live);
    if (sub == 0 && live) {
        const double lp = categorical_logp<double>(LG + (size_t)row * kMaxChoices, 1, n_choices, choice);
        LP[row] = lp + (-0.5 * u * u - 0.91893853320467274178) + logdet - y;
    }
}

// grid (chain blocks of 128, D): out[d * C + c] = the fp64 sum over the T_d trials of dataset d, in trial order.  One
// dataset of T trials (offsets == null, D = 1), or ragged sessions, session d owning trials [offsets[d], offsets[d + 1]).
__global__ void __launch_bounds__(128) precise_sum_kernel(const double *__restrict__ LP, const long long *__restrict__ offsets,
                                                          int T, int C, float *__restrict__ out)
{
    const int c = blockIdx.x * 128 + threadIdx.x, d = blockIdx.y;
    if (c >= C) return;
    const long long first = offsets != nullptr ? offsets[d] : 0;
    const int Td = offsets != nullptr ? (int)(offsets[d + 1] - first) : T;
    const double *col = LP + (size_t)first * C + c;
    double sum = 0.0;
    for (int t = 0; t < Td; ++t) sum += col[(size_t)t * C];
    out[(size_t)d * C + c] = (float)sum;
}

struct Tc64Bufs {
    unsigned char *pack;
    float *Q, *LG;
    float *lp32;  // the forward kernel's own fp32 log-prob slot (unused here)
    float *cond, *xr;
    double *LP;
};

static Tc64Bufs tc64_workspace(Carver &ws, const Layout &L, const TrainDims &d)
{
    Tc64Bufs b;
    b.pack = ws.take<unsigned char>(tc_train_pack_bytes(L.n_choices, d.R));
    b.Q = ws.take((size_t)kTransforms * kQRows * d.Rp);
    b.LG = ws.take((size_t)kMaxChoices * d.Rp);
    b.lp32 = ws.take(d.Rp);
    b.cond = ws.take((size_t)d.R * kCond);
    b.xr = ws.take(2 * (size_t)d.R);
    b.LP = ws.take<double>(d.Rp);
    return b;
}

}  // namespace mnle

DDM_API size_t mnle_loglik_tc64_workspace_floats(int n_choices, int64_t T, int64_t C)
{
    if (n_choices < 1 || n_choices > kMaxChoices || T <= 0 || C <= 0) return 0;
    const Layout L = make_layout(n_choices);
    Carver ws(nullptr);
    tc64_workspace(ws, L, train_dims(L, T * C));
    return ws.floats();
}

namespace mnle {

// tc64 over N flat trials: one dataset (trial_offsets == null, N = T) or D ragged sessions (see precise_sum_kernel).
static int tc64_loglik_sum(const char *entry, void *handle, const float *theta_dev, int64_t ld_theta, const float *x_dev,
                           const float *pulses_dev, int64_t ld_pulses, const int64_t *trial_offsets_dev, int64_t D, int64_t N,
                           int64_t C, float *out_dev, float *workspace_dev, cudaStream_t st)
{
    Handle *H;
    int rc = expanded_rows_prologue(entry, &H, handle, theta_dev, ld_theta, x_dev, pulses_dev, ld_pulses, N, C, out_dev, false,
                                    nullptr, workspace_dev, st, D);
    if (H == nullptr) return rc;
    const Layout &L = H->layout;
    const long long R = N * C;
    const TrainDims d = train_dims(L, R);
    Carver ws(workspace_dev);
    const Tc64Bufs B = tc64_workspace(ws, L, d);
    const long long *offsets = reinterpret_cast<const long long *>(trial_offsets_dev);
    potential_rows_kernel<<<(unsigned)std::min<long long>((R * kCond + 255) / 256, 148 * 16), 256, 0, st>>>(
        theta_dev, ld_theta, x_dev, pulses_dev, ld_pulses, (int)N, (int)C, B.cond, B.xr, offsets, (int)D);
    DDM_CUDA_TRY(cudaGetLastError());
    const TcTrainDump keep{nullptr, B.Q, B.LG, d.Rp, nullptr, nullptr, nullptr};
    rc = tc_train_forward(H->params, L, B.pack, B.xr, B.cond, (long long)kCond, nullptr, R, keep, B.lp32, st);
    if (rc != DDM_OK) return rc;
    precise_rows_kernel<<<(unsigned)((R + kBlockRows - 1) / kBlockRows), kRowWarps * 32, 0, st>>>(B.Q, B.LG, d.Rp, B.xr, R, L.n_choices,
                                                                                                  H->mu_y, H->sigma_y, B.LP);
    DDM_CUDA_TRY(cudaGetLastError());
    precise_sum_kernel<<<dim3((unsigned)((C + 127) / 128), (unsigned)D), 128, 0, st>>>(B.LP, offsets, (int)N, (int)C, out_dev);
    DDM_CUDA_TRY(cudaGetLastError());
    return DDM_OK;
}

}  // namespace mnle

DDM_API int mnle_loglik_sum_tc64_f32(void *handle, const float *theta_dev, int64_t ld_theta, const float *x_dev,
                                     const float *pulses_dev, int64_t ld_pulses, int64_t T, int64_t C, float *out_dev,
                                     float *workspace_dev, void *stream)
{
    return tc64_loglik_sum("mnle_loglik_sum_tc64_f32", handle, theta_dev, ld_theta, x_dev, pulses_dev, ld_pulses, nullptr, 1, T,
                           C, out_dev, workspace_dev, static_cast<cudaStream_t>(stream));
}

DDM_API size_t mnle_loglik_sessions_tc64_workspace_floats(int n_choices, int64_t D, int64_t N, int64_t C)
{
    return D <= 0 ? 0 : mnle_loglik_tc64_workspace_floats(n_choices, N, C);
}

DDM_API int mnle_loglik_sum_sessions_tc64_f32(void *handle, const float *theta_dev, int64_t ld_theta, const float *x_dev,
                                              const float *pulses_dev, int64_t ld_pulses, const int64_t *trial_offsets_dev,
                                              int64_t D, int64_t N, int64_t C, float *out_dev, float *workspace_dev, void *stream)
{
    DDM_REQUIRE(D >= 0 && D <= 65535, "mnle_loglik_sum_sessions_tc64_f32: D=%lld sessions (at most 65535 per call)", (long long)D);
    if (D == 0) return DDM_OK;
    DDM_REQUIRE(trial_offsets_dev != nullptr, "mnle_loglik_sum_sessions_tc64_f32: null trial_offsets");
    return tc64_loglik_sum("mnle_loglik_sum_sessions_tc64_f32", handle, theta_dev, ld_theta, x_dev, pulses_dev, ld_pulses,
                           trial_offsets_dev, D, N, C, out_dev, workspace_dev, static_cast<cudaStream_t>(stream));
}

// ---- estimator.sample: the choice from the categorical net, then log rt from the flow run in inverse --------------
// sbi's MixedDensityEstimator.sample draws the choice first and then log rt from the spline flow conditioned on it.
// Here: the S x B condition rows are expanded (row r = s * B + b), the tcgen05 rows-mode forward runs the categorical
// net alone and keeps the logits, one thread per row draws the choice in fp64 and writes it into the context column,
// the forward runs the ten conditioners on the new context and keeps the raw spline parameters, and four lanes per row
// draw u from N(0, 1) and walk the ten splines backwards in fp64 (the same arithmetic as the tc64 potential).
namespace mnle {

constexpr uint32_t kSampleTag = 0x4D4E4C45u;  // counter word 3 of the sampler's Philox blocks (the simulator's is 0 or 1)

__global__ void __launch_bounds__(256) sample_rows_kernel(const float *__restrict__ cond_in, long long ld_cond, long long B,
                                                          long long R, float *__restrict__ cond, float *__restrict__ xr)
{
    const long long total = R * kCond;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const long long r = idx / kCond;
        const int j = (int)(idx - r * kCond);
        cond[idx] = __ldg(cond_in + (r % B) * ld_cond + j);
        if (j < 2) xr[2 * r + j] = j == 0 ? 1.0f : 0.0f;  // rt is not read by the forward; the choice starts at 0
    }
}

// One Philox block per row (see the header): u_c from word 0, the normal from words 1-3 by Box-Muller in fp64.
// draws != null: row r takes [u_c, n] = draws[2 r], draws[2 r + 1] instead.
__global__ void __launch_bounds__(256) sample_choice_kernel(const float *__restrict__ LG, long long R, long long B, int n_choices,
                                                            const ddm::PhiloxKey key, unsigned long long sample_offset,
                                                            const float *__restrict__ draws, float *__restrict__ xr,
                                                            double *__restrict__ normal)
{
    const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= R) return;
    double uc, n;
    if (draws != nullptr) {
        uc = (double)__ldg(draws + 2 * r);
        n = (double)__ldg(draws + 2 * r + 1);
    } else {
        const unsigned long long s = sample_offset + (unsigned long long)(r / B);
        const uint32_t b = (uint32_t)(r % B);
        uint32_t w[4];
        ddm::philox4x32_10((uint32_t)s, (uint32_t)(s >> 32), b, kSampleTag, key, w);
        uc = ((double)w[0] + 0.5) * 0x1p-32;
        const double u1 = ((double)(((unsigned long long)(w[1] >> 5) << 26) | (w[2] >> 6)) + 0.5) * 0x1p-53;
        n = sqrt(-2.0 * log(u1)) * cospi(((double)w[3] + 0.5) * 0x1p-31);
    }
    const float *lg = LG + (size_t)r * kMaxChoices;
    double m = -INFINITY;
    for (int j = 0; j < n_choices; ++j) m = fmax(m, (double)lg[j]);
    double s = 0.0;
    for (int j = 0; j < n_choices; ++j) s += exp((double)lg[j] - m);
    int c = n_choices - 1;  // also when rounding leaves u_c at or above the last cumulative probability
    double cum = 0.0;
    for (int j = 0; j < n_choices - 1; ++j) {
        cum += exp((double)lg[j] - m) / s;
        if (uc < cum) {
            c = j;
            break;
        }
    }
    xr[2 * r + 1] = (float)c;
    normal[r] = n;
}

// (__maxnreg__: with only the launch bound ptxas settles on 64 registers and spills; 80 keeps three blocks per SM)
__global__ void __maxnreg__(80) sample_chain_kernel(const float *__restrict__ Q, long long Rp, const float *__restrict__ xr,
                                                                      const double *__restrict__ normal, long long R, float mu_y,
                                                                      float sigma_y, float *__restrict__ x_out)
{
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int sub = lane & (kRowLanes - 1), base = lane & ~(kRowLanes - 1), rw = lane / kRowLanes;
    const long long row = ((long long)blockIdx.x * kRowWarps + wib) * kWarpRows + rw;
    const bool live = row < R;
    const long long rowc = live ? row : 0;
    double u = live ? normal[rowc] : 0.0, unused = 0.0;
#pragma unroll 1
    for (int k = kTransforms - 1; k >= 0; --k) rqs_quad_f64<true>(u, unused, Q + ((size_t)k * Rp + rowc) * kQRows, base, sub, live);
    if (sub == 0 && live) {
        x_out[2 * row] = (float)exp((double)mu_y + (double)sigma_y * u);
        x_out[2 * row + 1] = __ldg(xr + 2 * row + 1);
    }
}

struct SampleBufs {
    unsigned char *pack;
    float *Q, *LG;
    float *cond, *xr;  // expanded condition rows, x rows
    double *normal;
};

static SampleBufs sample_workspace(Carver &ws, const Layout &L, const TrainDims &d)
{
    SampleBufs b;
    b.pack = ws.take<unsigned char>(tc_train_pack_bytes(L.n_choices, d.R));
    b.Q = ws.take((size_t)kTransforms * kQRows * d.Rp);
    b.LG = ws.take((size_t)kMaxChoices * d.Rp);
    b.cond = ws.take((size_t)d.R * kCond);
    b.xr = ws.take(2 * (size_t)d.R);
    b.normal = ws.take<double>(d.Rp);
    return b;
}

}  // namespace mnle

DDM_API size_t mnle_sample_tc_workspace_floats(int n_choices, int64_t B, int64_t S)
{
    if (n_choices < 1 || n_choices > kMaxChoices || B <= 0 || S <= 0 || B * S > 8000000ll) return 0;
    const Layout L = make_layout(n_choices);
    Carver ws(nullptr);
    sample_workspace(ws, L, train_dims(L, B * S));
    return ws.floats();
}

DDM_API int mnle_sample_tc_f32(void *handle, const float *cond_dev, int64_t ld_cond, int64_t B, int64_t S, uint64_t seed,
                               uint64_t sample_offset, const float *draws_dev, float *x_out_dev, float *workspace_dev, void *stream)
{
    DDM_REQUIRE(B >= 0 && S >= 0, "mnle_sample_tc_f32: B=%lld S=%lld must not be negative", (long long)B, (long long)S);
    DDM_REQUIRE(B == 0 || S <= 8000000ll / B, "mnle_sample_tc_f32: B=%lld x S=%lld rows (at most 8e6 per call)", (long long)B,
                (long long)S);
    DDM_REQUIRE(ld_cond >= kCond, "mnle_sample_tc_f32: ld_cond=%lld < 85", (long long)ld_cond);
    const long long R = B * S;
    if (R > 0) {
        DDM_REQUIRE(cond_dev && x_out_dev && workspace_dev, "mnle_sample_tc_f32: null pointer");
        DDM_REQUIRE((reinterpret_cast<uintptr_t>(workspace_dev) & 255u) == 0, "mnle_sample_tc_f32: workspace must be 256-byte aligned");
    }
    Handle *H = live_handle(handle, "mnle_sample_tc_f32");
    if (H == nullptr) return DDM_ERR_STATE;
    if (R == 0) return DDM_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const Layout &L = H->layout;
    const TrainDims d = train_dims(L, R);
    Carver ws(workspace_dev);
    const SampleBufs W = sample_workspace(ws, L, d);
    sample_rows_kernel<<<(unsigned)std::min<long long>((R * kCond + 255) / 256, 148 * 16), 256, 0, st>>>(cond_dev, (long long)ld_cond,
                                                                                                        (long long)B, R, W.cond, W.xr);
    DDM_CUDA_TRY(cudaGetLastError());
    TcTrainDump keep{nullptr, W.Q, W.LG, d.Rp, nullptr, nullptr, nullptr};
    keep.net0 = 0;
    keep.nets = 1;  // the categorical net: logits
    int rc = tc_train_forward(H->params, L, W.pack, W.xr, W.cond, (long long)kCond, nullptr, R, keep, nullptr, st);
    if (rc != DDM_OK) return rc;
    sample_choice_kernel<<<(unsigned)((R + 255) / 256), 256, 0, st>>>(W.LG, R, (long long)B, L.n_choices, ddm::make_philox_key(seed),
                                                                     (unsigned long long)sample_offset, draws_dev, W.xr, W.normal);
    DDM_CUDA_TRY(cudaGetLastError());
    keep.net0 = 1;
    keep.nets = kTransforms;  // the conditioners on [condition, sampled choice]: raw spline parameters
    rc = tc_train_forward(H->params, L, W.pack, W.xr, W.cond, (long long)kCond, nullptr, R, keep, nullptr, st);
    if (rc != DDM_OK) return rc;
    sample_chain_kernel<<<(unsigned)((R + kBlockRows - 1) / kBlockRows), kRowWarps * 32, 0, st>>>(W.Q, d.Rp, W.xr, W.normal, R, H->mu_y,
                                                                                                   H->sigma_y, x_out_dev);
    DDM_CUDA_TRY(cudaGetLastError());
    return DDM_OK;
}
