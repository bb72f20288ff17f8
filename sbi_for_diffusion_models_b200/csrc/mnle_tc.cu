// MNLE log-likelihood on the 5th-generation tensor cores (tcgen05.mma, TMEM accumulators).
//
// The 128x128 and 128x71 layers of the categorical net and of the ten spline conditioners are
// dense GEMMs over (trial, chain) rows -- the only tensor-core-shaped work on this path.  fp32
// accuracy (sums within 1e-4 relative, north_star) is kept by splitting every operand into
// bf16 hi + lo and issuing three MMAs per product (hi*hi + hi*lo + lo*hi, fp32 accumulate in
// TMEM): 16 mantissa bits per operand at 3/2 of the cost of a tf32 product.
//
// This file: the operand layout / descriptor self-test (mnle_tc_selftest) and the fused kernel.
#include "mnle_common.cuh"
#include "tc_ptx.cuh"

namespace mnle {

using namespace tc;

// Shared-memory image of a K-major bf16 operand tile [R rows][K]: for every group of 8 k's
// (16 bytes) all R rows are contiguous.  offset(r, k) = (k/8) * R*16 + r*16 + (k%8)*2 bytes.
//   => SBO (next 8-row group) = 128 B, LBO (next 8-k group) = R*16 B.
__host__ __device__ constexpr uint32_t tile_offset(int R, int r, int k) { return (uint32_t)((k >> 3) * R * 16 + r * 16 + (k & 7) * 2); }

// ------------------------------------------------------------------------------ self-test ---
// D (128 x N) = A (128 x 128) * B (N x 128)^T through exactly the building blocks of the fused
// kernel.  passes = 1: bf16(A) * bf16(B) only; passes = 3: hi/lo split.  lbo / sbo can be
// overridden (0 = the layout's own values) to probe descriptor conventions on hardware.
__global__ void __launch_bounds__(128) tc_selftest_kernel(const float *__restrict__ A, const float *__restrict__ B, int N,
                                                          int passes, uint32_t lbo_a, uint32_t lbo_b, uint32_t sbo,
                                                          float *__restrict__ D)
{
    extern __shared__ __align__(1024) unsigned char smem[];
    unsigned char *a_hi = smem;                 // 128 x 128 bf16 = 32 KB
    unsigned char *a_lo = smem + 32768;
    unsigned char *b_hi = smem + 65536;         // up to 128 x 128 bf16
    unsigned char *b_lo = smem + 98304;
    uint64_t *bar = reinterpret_cast<uint64_t *>(smem + 131072);
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(smem + 131072 + 16);

    const int tid = threadIdx.x, warp = tid >> 5;
    const bool a_in_tmem = (passes % 100) > 10 && passes < 100 || passes >= 200;
    if (a_in_tmem && passes < 100) passes -= 10;
    if (warp == 0) tmem_alloc<256>(tmem_slot);
    if (tid == 0) {
        mbar_init(bar, 1);
        fence_mbar_init();
    }
    tc_fence_before_sync();
    __syncthreads();
    tc_fence_after_sync();
    if (a_in_tmem) {
        // A hi -> TMEM columns [128, 192), A lo -> [192, 256): lane = row, column j = k pair (2j, 2j+1)
        const uint32_t tm = *tmem_slot + ((uint32_t)(warp * 32) << 16);
        for (int j0 = 0; j0 < 64; j0 += 16) {
            uint32_t hi[16], lo[16];
#pragma unroll
            for (int j = 0; j < 16; ++j)
                split_bf16x2(A[tid * 128 + 2 * (j0 + j)], A[tid * 128 + 2 * (j0 + j) + 1], hi[j], lo[j]);
            tmem_st16(tm + 128u + (uint32_t)j0, hi);
            tmem_st16(tm + 192u + (uint32_t)j0, lo);
        }
        tmem_wait_st();
    }
    // operands -> smem images (thread r owns row r of A and, if r < N, row r of B)
    for (int kg = 0; kg < 16; ++kg) {
        uint16_t hi[8], lo[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) split_bf16(A[tid * 128 + kg * 8 + j], hi[j], lo[j]);
        uint4 vh = make_uint4(hi[0] | (hi[1] << 16), hi[2] | (hi[3] << 16), hi[4] | (hi[5] << 16), hi[6] | (hi[7] << 16));
        uint4 vl = make_uint4(lo[0] | (lo[1] << 16), lo[2] | (lo[3] << 16), lo[4] | (lo[5] << 16), lo[6] | (lo[7] << 16));
        *reinterpret_cast<uint4 *>(a_hi + tile_offset(128, tid, kg * 8)) = vh;
        *reinterpret_cast<uint4 *>(a_lo + tile_offset(128, tid, kg * 8)) = vl;
        if (tid < N) {
#pragma unroll
            for (int j = 0; j < 8; ++j) split_bf16(B[tid * 128 + kg * 8 + j], hi[j], lo[j]);
            vh = make_uint4(hi[0] | (hi[1] << 16), hi[2] | (hi[3] << 16), hi[4] | (hi[5] << 16), hi[6] | (hi[7] << 16));
            vl = make_uint4(lo[0] | (lo[1] << 16), lo[2] | (lo[3] << 16), lo[4] | (lo[5] << 16), lo[6] | (lo[7] << 16));
            *reinterpret_cast<uint4 *>(b_hi + tile_offset(N, tid, kg * 8)) = vh;
            *reinterpret_cast<uint4 *>(b_lo + tile_offset(N, tid, kg * 8)) = vl;
        }
    }
    fence_proxy_async_smem();
    tc_fence_before_sync();
    __syncthreads();
    tc_fence_after_sync();
    const uint32_t tmem = *tmem_slot;

    // passes >= 100: throughput probe -- (passes % 100) rounds of the 24-MMA stage sequence back to
    // back, D[0] = clock cycles from the first issue to the commit's arrival
    const int reps = passes >= 100 ? passes % 100 : 0;
    if (reps) passes = 3;
    long long t_start = 0;
    if (warp == 0 && elect_one_sync()) {
        const uint32_t idesc = umma_idesc_bf16_f32(128, N);
        const uint32_t la = lbo_a ? lbo_a : 128u * 16u, lb = lbo_b ? lbo_b : (uint32_t)N * 16u, sb = sbo ? sbo : 128u;
        uint32_t acc = 0;
        t_start = clock64();
        for (int rep = 0; rep < max(reps, 1); ++rep)
        for (int pass = 0; pass < passes; ++pass) {
            const unsigned char *pa = (pass == 2) ? a_lo : a_hi;
            const unsigned char *pb = (pass == 1) ? b_lo : b_hi;
#pragma unroll
            for (int ks = 0; ks < 8; ++ks) {
                const uint64_t da = umma_desc_kmajor(smem_u32(pa) + ks * 2 * 128 * 16, la, sb);
                const uint64_t db = umma_desc_kmajor(smem_u32(pb) + ks * 2 * N * 16, lb, sb);
                if (a_in_tmem)
                    umma_bf16_ts(tmem, tmem + (pass == 2 ? 192u : 128u) + (uint32_t)ks * 8u, db, idesc, acc);
                else
                    umma_bf16(tmem, da, db, idesc, acc);
                acc = 1;
            }
        }
        umma_commit(bar);
    }
    mbar_wait(bar, 0);
    tc_fence_after_sync();
    const long long t_end = clock64();
    if (reps) {
        t_start = __shfl_sync(0xFFFFFFFFu, t_start, 0);  // (any lane may have been elected)
        if (tid == 0) D[0] = (float)(t_end - t_start);
        tc_fence_before_sync();
        __syncthreads();
        if (warp == 0) tmem_dealloc<256>(tmem);
        return;
    }
    // thread (warp w, lane l) reads TMEM lane 32 w + l = output row
    for (int c0 = 0; c0 < N; c0 += 16) {
        uint32_t r[16];
        tmem_ld16(tmem + ((uint32_t)(warp * 32) << 16) + (uint32_t)c0, r);
        tmem_wait_ld();
#pragma unroll
        for (int j = 0; j < 16; ++j) D[tid * N + c0 + j] = __uint_as_float(r[j]);
    }
    tc_fence_before_sync();
    __syncthreads();
    if (warp == 0) tmem_dealloc<256>(tmem);
}


// ---------------------------------------------------------------- per-trial first layer ---
// hoist[t][net][j] = b1[j] + sum_i W1[j][5 + i] * pulses[t][i] (+ W1[j][85] * choice[t] for the
// spline conditioners): the part of every first layer that does not depend on the chain.
// grid = (nets, ceil(T / 8)): the 128 x 81 weight block is staged in shared memory once per block
// and reused for 8 trials.  Block (0, 0) also clears the per-chain-block arrival counters of the
// fused kernel's final reduction.
// SESS, ragged sessions (offsets: D + 1 entries, T = offsets[D] flat trials): the net-0 blocks also
// write the session of each of their trials to sess[] (one binary search per trial instead of one per
// tile and thread in the fused kernel), and write the C zeros of the empty sessions d = y (mod grid y)
// -- such a session has no tile that could write them.
constexpr int kHoistTrials = 8;
constexpr int kHoistK = kCtx - 5;  // 81
template <bool SESS>
__global__ void __launch_bounds__(kHidden) mnle_hoist_kernel(const float *__restrict__ params, Layout L,
                                                            const float *__restrict__ x,
                                                            const float *__restrict__ pulses, long long ld_pulses, int T,
                                                            float *__restrict__ hoist, unsigned int *__restrict__ counters,
                                                            int n_counters, const long long *__restrict__ offsets, int D,
                                                            int C, int *__restrict__ sess, float *__restrict__ out)
{
    __shared__ float w_s[kHidden * kHoistK];
    __shared__ float in_s[kHoistTrials][kHoistK + 3];
    const int net = blockIdx.x, t0 = blockIdx.y * kHoistTrials, j = threadIdx.x;
    if (blockIdx.x == 0 && blockIdx.y == 0)
        for (int i = j; i < n_counters; i += kHidden) counters[i] = 0u;
    if (SESS && blockIdx.x == 0) {
        if (j < kHoistTrials && t0 + j < T) sess[t0 + j] = session_of(offsets, D, t0 + j);
        for (int d = blockIdx.y; d < D; d += gridDim.y)
            if (__ldg(offsets + d + 1) == __ldg(offsets + d))
                for (int c = j; c < C; c += kHidden) out[(size_t)d * C + c] = 0.f;
    }
    const int K = net == 0 ? kCond : kCtx;
    const float *W = params + (net == 0 ? L.cat_W0 : L.fl_W1[net - 1]);
    // 81 independent loads per thread in flight (fully unrolled): the block is latency-bound
#pragma unroll
    for (int it = 0; it < kHoistK; ++it) {
        const int idx = it * kHidden + j;
        const int row = idx / kHoistK, i = idx - row * kHoistK;
        w_s[idx] = (5 + i < K) ? __ldg(W + (size_t)row * K + 5 + i) : 0.f;
    }
    for (int idx = j; idx < kHoistTrials * kHoistK; idx += kHidden) {
        const int tr = idx / kHoistK, i = idx - tr * kHoistK, t = t0 + tr;
        float v = 0.f;
        if (t < T) v = (i < kCond - 5) ? __ldg(pulses + (long long)t * ld_pulses + i) : __ldg(x + 2 * t + 1);
        in_s[tr][i] = v;
    }
    __syncthreads();
    const float b = __ldg(params + (net == 0 ? L.cat_b0 : L.fl_b1[net - 1]) + j);
    float acc[kHoistTrials];
#pragma unroll
    for (int tr = 0; tr < kHoistTrials; ++tr) acc[tr] = b;
#pragma unroll 3
    for (int i = 0; i < kHoistK; ++i) {
        const float w = w_s[j * kHoistK + i];
#pragma unroll
        for (int tr = 0; tr < kHoistTrials; ++tr) acc[tr] = fmaf(w, in_s[tr][i], acc[tr]);
    }
#pragma unroll
    for (int tr = 0; tr < kHoistTrials; ++tr)
        if (t0 + tr < T) hoist[((size_t)(t0 + tr) * kNets + net) * kHidden + j] = acc[tr];
}

// ------------------------------------------------------------------------ fused kernel ---
// One CTA = two row tiles of 128 (trial, chain) rows in ping-pong: while the tensor core runs a
// stage of one tile, the four epilogue warps of the other tile turn its accumulators into the
// next A operand.  Activations never leave tensor memory: D (128 fp32 columns) -> registers ->
// bias, activation, bf16 hi/lo split -> A_hi / A_lo (64 + 64 packed columns) of the same tile,
// which the next stage's tcgen05.mma reads as its A operand.  2 x 256 columns = all of TMEM.
// Shared memory holds only the streamed weight blobs (3 slots) and the theta-stage A images.
constexpr int kTcM = 128;                        // rows per tile = UMMA M
constexpr int kTcTiles = 2;                      // tiles per CTA
constexpr int kTcEpiWarps = 16;                  // warp w: lane quarter w & 3, tile (w >> 2) & 1, column half w >> 3
constexpr int kTcEpiThreads = kTcEpiWarps * 32;
constexpr int kTcIssuers = 2;                    // issuer warps: warp kTcEpiWarps + i owns stages s = i (mod 2)
constexpr int kTcThreads = kTcEpiThreads + 32 * kTcIssuers;
constexpr uint32_t kImgBytes = kTcM * 256;       // one bf16 image of 128 rows x 128 k
constexpr uint32_t kKGroupBytes = kTcM * 16;     // 8 k's of all 128 rows
constexpr uint32_t kAThBytes = kTcM * 64;        // theta-stage A image: 128 rows x 32 k
constexpr uint32_t kCtxImgBytes = kTcM * kInputK * 2;          // rows mode: 128 rows x 96 k of context, one bf16 term
constexpr uint32_t kSlotBytes = 2 * kImgBytes + kHidden * 4;   // largest blob; theta blobs are 8 KB + 2 biases
// Shared memory.  Potential mode: theta-stage A images of the two tiles, then a ring of 3 weight slots
// (prefetch two stages ahead).  Rows mode: the 86-wide context of both tiles as bf16 hi / lo A images
// (4 x 24 KB; tensor memory is full with two tiles), then 2 weight slots (prefetch one stage ahead).
template <bool ROWS>
struct TcSmem {
    static constexpr int kSlots = ROWS ? 2 : 3;
    static constexpr uint32_t kA = 0;
    static constexpr uint32_t kSlot0 = ROWS ? kTcTiles * 2 * kCtxImgBytes : kTcTiles * kAThBytes;
    static constexpr uint32_t kBars = kSlot0 + kSlots * kSlotBytes;
    static constexpr uint32_t kBytes = kBars + 128;
    static_assert(kBytes <= 227 * 1024, "tiles do not fit shared memory");
};
constexpr uint32_t kTmemD = 0, kTmemAHi = 128, kTmemALo = 192, kTmemTile = 256;  // columns

// ncols accumulator columns + bias -> activation -> packed bf16 hi / lo columns of the A operand.
// The CUDA-core side of this kernel is bound by the half-rate ALU pipe (min/max, selects,
// conversions, logic), so the arithmetic is phrased for the FMA pipe wherever possible.
// `keep` (training forward): the activations of this row also go to global memory, COLUMN-major (element
// (row, col) at keep[col * keep_ld], keep pointing at the row): a lane holds one row, so the 32 lanes of a
// store instruction write 32 consecutive rows of one column = one 128-byte line.
// `keep_m` (potential gradient, ReLU layers): instead of the activations only the SIGNS of the pre-activations are
// kept, one 32-bit word per 32 columns (bit 31 - j: column c0 + j negative), words keep_ld apart.  (A pre-activation
// of exactly +0 counts as active here and as inactive in torch's ReLU: it carries no gradient either way unless the
// upstream gradient is non-zero at a measure-zero point.)
template <int EPI>
__device__ __forceinline__ void tc_epilogue_act(uint32_t trow, int col0, int ncols, const float *bias,
                                                float *keep = nullptr, size_t keep_ld = 0, uint32_t *keep_m = nullptr)
{
#pragma unroll 1
    for (int c0 = col0; c0 < col0 + ncols; c0 += 32) {
        uint32_t v[32];
        tmem_ld32(trow + kTmemD + (uint32_t)c0, v);
        tmem_wait_ld();
        uint32_t hi[16], lo[16];
        uint32_t neg = 0u;
#pragma unroll
        for (int g = 0; g < 8; ++g) {
            const float4 b = *reinterpret_cast<const float4 *>(bias + c0 + 4 * g);
            float f[4] = {__uint_as_float(v[4 * g + 0]), __uint_as_float(v[4 * g + 1]), __uint_as_float(v[4 * g + 2]),
                          __uint_as_float(v[4 * g + 3])};
            add_f32x2(f[0], f[1], b.x, b.y);
            add_f32x2(f[2], f[3], b.z, b.w);
            if (EPI == kEpiSigmoid) {
#pragma unroll
                for (int j = 0; j < 4; ++j) f[j] = fast_rcp(1.0f + fast_ex2(-1.4426950408889634f * f[j]));
            }
            if (EPI == kEpiRelu && keep_m != nullptr) {
#pragma unroll
                for (int j = 0; j < 4; ++j) neg = __funnelshift_l(__float_as_uint(f[j]), neg, 1);   // shift the sign bit in
            }
            split_relu_bf16x2(f[0], f[1], hi[2 * g], lo[2 * g]);
            split_relu_bf16x2(f[2], f[3], hi[2 * g + 1], lo[2 * g + 1]);
            if (keep != nullptr) {  // (the ReLU is fused into the conversions above)
#pragma unroll
                for (int j = 0; j < 4; ++j) keep[(size_t)(c0 + 4 * g + j) * keep_ld] = EPI == kEpiRelu ? fmaxf(f[j], 0.f) : f[j];
            }
        }
        if (EPI == kEpiRelu && keep_m != nullptr) keep_m[(size_t)((c0 - col0) >> 5) * keep_ld] = neg;
        tmem_st16(trow + kTmemAHi + (uint32_t)(c0 >> 1), hi);
        tmem_st16(trow + kTmemALo + (uint32_t)(c0 >> 1), lo);
    }
    tmem_wait_st();
}

// Backward-data epilogue: ncols accumulator columns (d loss / d activations) times the derivative of the
// activation whose output h sits in global memory -> d loss / d pre-activations, written to global memory
// and, when another stage follows, split into the bf16 hi / lo A operand of that stage.
// d_row may be null (potential gradient: the derivatives are not kept); w1s (shared memory, [128][8], may be null): the
// five theta columns of this net's first layer -- acc5[i] += sum_j d[j] * w1s[j][i] over this thread's columns.
// POT (the potential's gradient): ReLU layers read sign masks (m_row) instead of activations, nothing is written to
// d_row, and the last stage contracts with w1s.  !POT (the training step): activations in, derivatives out.
template <int EPI, bool POT>
__device__ __forceinline__ void tc_epilogue_mask(uint32_t trow, int col0, int ncols, const float *h_row, float *d_row, size_t ld,
                                                 bool have, bool feeds_next, uint64_t *dfull, uint32_t parity,
                                                 const float *w1s = nullptr, float *acc5 = nullptr, const uint32_t *m_row = nullptr)
{
#pragma unroll 1
    for (int c0 = col0; c0 < col0 + ncols; c0 += 32) {
        float h[32];  // column-major storage: every load / store below is one 128-byte line per warp
        constexpr bool masks = POT && EPI == kEpiRelu;   // sign masks of the pre-activations instead of activations
        uint32_t neg = 0xFFFFFFFFu;
        if (masks) {
            if (have) neg = m_row[(size_t)((c0 - col0) >> 5) * ld];
        } else {
#pragma unroll
            for (int j = 0; j < 32; ++j) h[j] = have ? h_row[(size_t)(c0 + j) * ld] : 0.f;
        }
        if (c0 == col0) {  // the kept activations do not depend on the MMAs: their latency hides behind the wait
            mbar_wait(dfull, parity);
            tc_fence_after_sync();
        }
        uint32_t v[32];
        tmem_ld32(trow + kTmemD + (uint32_t)c0, v);
        tmem_wait_ld();
#pragma unroll
        for (int j = 0; j < 32; ++j) {  // h <- d loss / d pre-activation, in place
            const float x = __uint_as_float(v[j]);
            if (masks) h[j] = (neg & (0x80000000u >> j)) ? 0.f : x;
            else h[j] = EPI == kEpiRelu ? (h[j] > 0.f ? x : 0.f) : x * h[j] * (1.0f - h[j]);
        }
        if (feeds_next) {
            uint32_t hi[16], lo[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) split_bf16x2(h[2 * j], h[2 * j + 1], hi[j], lo[j]);
            tmem_st16(trow + kTmemAHi + (uint32_t)(c0 >> 1), hi);
            tmem_st16(trow + kTmemALo + (uint32_t)(c0 >> 1), lo);
        }
        if (!POT && have) {
#pragma unroll
            for (int j = 0; j < 32; ++j) d_row[(size_t)(c0 + j) * ld] = h[j];
        }
        if (POT && w1s != nullptr) {
#pragma unroll
            for (int j = 0; j < 32; ++j) {
                const float4 wa = *reinterpret_cast<const float4 *>(w1s + (c0 + j) * 8);   // same address in every lane: broadcast
                const float wb = w1s[(c0 + j) * 8 + 4];
                acc5[0] = fmaf(h[j], wa.x, acc5[0]);
                acc5[1] = fmaf(h[j], wa.y, acc5[1]);
                acc5[2] = fmaf(h[j], wa.z, acc5[2]);
                acc5[3] = fmaf(h[j], wa.w, acc5[3]);
                acc5[4] = fmaf(h[j], wb, acc5[4]);
            }
        }
    }
    tmem_wait_st();
}

// softmax numerators of one 24-bin block held in registers: e[j] = exp((q[j] - max q) / sqrt(128));
// returns 1 / sum e.
__device__ __forceinline__ float rqs_softmax(const float (&q)[kBins], float (&e)[kBins])
{
    const float c = 0.08838834764831845f * 1.4426950408889634f;  // log2(e) / sqrt(128)
    float m = fmaxf(fmaxf(q[0], q[1]), q[2]);
#pragma unroll
    for (int j = 3; j < kBins; j += 3) m = fmaxf(fmaxf(m, q[j]), fmaxf(q[j + 1], q[j + 2]));
    const float mc = m * c;
    float s0 = 0.f, s1 = 0.f;
#pragma unroll
    for (int j = 0; j < kBins; j += 2) {
        e[j] = fast_ex2(fmaf(q[j], c, -mc));
        e[j + 1] = fast_ex2(fmaf(q[j + 1], c, -mc));
        s0 += e[j];
        s1 += e[j + 1];
    }
    return fast_rcp(s0 + s1);
}

// One rational-quadratic spline transform (Durkan et al. 2019, linear tails) of row `trow`.
// The 71 parameters are pulled from the accumulator columns in three 24-column blocks (widths,
// derivatives, heights).  The bin is located without selects: p_j = [u >= knot_j] (one FSET per
// knot) gives the one-hot ind_j = p_j - p_{j+1}, and every per-bin quantity is a dot product with
// ind on the FMA pipe (exact: ind is 0 or 1).  The tile's aready barrier is released as soon as
// the last block is in registers.
__device__ __forceinline__ void tc_epilogue_spline(uint32_t trow, const float *bias, float &u, float &logdet,
                                                   uint64_t *aready)
{
    uint32_t vw[kBins], vd[kBins];
    tmem_ld_n<kBins>(trow + kTmemD, vw);
    tmem_ld_n<kBins>(trow + kTmemD + 2 * kBins, vd);  // 23 derivatives + 1 padding column
    tmem_wait_ld();
    const bool inside = (u >= -kTail && u <= kTail);
    const float uc = fminf(fmaxf(u, -kTail), kTail);  // (outside rows are computed and discarded)
    float q[kBins], e[kBins], ind[kBins];
    const float span = 2.0f * kTail * (1.0f - kMinBin * kBins), floor20 = 2.0f * kTail * kMinBin;
#pragma unroll
    for (int j = 0; j < kBins; ++j) q[j] = __uint_as_float(vw[j]) + bias[j];
    float sc = span * rqs_softmax(q, e);
    float knot = -kTail, pprev = 1.0f, left = 0.f, wid = 0.f;
#pragma unroll
    for (int j = 0; j < kBins; ++j) {
        const float w20 = (j == kBins - 1) ? kTail - knot : fmaf(sc, e[j], floor20);
        const float next = (j == kBins - 1) ? kTail : knot + w20;
        const float pnext = (j == kBins - 1) ? 0.0f : (uc >= next ? 1.0f : 0.0f);
        ind[j] = pprev - pnext;
        left = fmaf(ind[j], knot, left);
        wid = fmaf(ind[j], w20, wid);
        pprev = pnext;
        knot = next;
    }
    float r0 = 0.f, r1 = 0.f;  // derivative logits at the bin's two knots (interior knots only)
#pragma unroll
    for (int j = 0; j < kBins - 1; ++j) {
        const float dj = __uint_as_float(vd[j]) + bias[2 * kBins + j];
        r0 = fmaf(ind[j + 1], dj, r0);
        r1 = fmaf(ind[j], dj, r1);
    }
    uint32_t vh[kBins];
    tmem_ld_n<kBins>(trow + kTmemD + kBins, vh);
    tmem_wait_ld();
    // bias is part of the weight slot, which may be refilled once this tile has arrived: read it first
#pragma unroll
    for (int j = 0; j < kBins; ++j) q[j] = __uint_as_float(vh[j]) + bias[kBins + j];
    tc_fence_before_sync();
    mbar_arrive(aready);  // D and the slot are free: the next stage's MMA runs while the spline finishes
    sc = span * rqs_softmax(q, e);
    knot = -kTail;
    float bottom = 0.f, hgt = 0.f;
#pragma unroll
    for (int j = 0; j < kBins; ++j) {
        const float h20 = (j == kBins - 1) ? kTail - knot : fmaf(sc, e[j], floor20);
        bottom = fmaf(ind[j], knot, bottom);
        hgt = fmaf(ind[j], h20, hgt);
        knot += h20;
    }
    if (!inside) return;  // identity outside the tail bound
    // softplus(r) = log(1 + exp(r)); the boundary knots have derivative exactly 1
    const float l2e = 1.4426950408889634f, ln2 = 0.6931471805599453f;
    const float sp0 = r0 > 20.0f ? r0 : ln2 * fast_lg2(1.0f + fast_ex2(r0 * l2e));
    const float sp1 = r1 > 20.0f ? r1 : ln2 * fast_lg2(1.0f + fast_ex2(r1 * l2e));
    const float d0 = ind[0] > 0.5f ? 1.0f : kMinDeriv + sp0;
    const float d1 = ind[kBins - 1] > 0.5f ? 1.0f : kMinDeriv + sp1;
    const float rw = fast_rcp(wid);
    const float delta = hgt * rw;
    const float th = (uc - left) * rw;
    const float om = 1.0f - th;
    const float t1 = th * om;
    const float den = fmaf(d0 + d1 - 2.0f * delta, t1, delta);
    const float rden = fast_rcp(den);
    const float dnum = delta * delta * (d1 * th * th + 2.0f * delta * t1 + d0 * om * om);
    logdet = fmaf(ln2, fast_lg2(dnum * rden * rden), logdet);
    u = fmaf(hgt * (delta * th * th + d0 * t1), rden, bottom);
}

// tile = ((d * T + t) * CB + chain block), chain block fastest; grid: tc_grid().
// D independent datasets (own x, pulses and C chains each) share one launch.  SESS, ragged sessions
// (a template flag, so that the uniform path's code is what it was): tile = (flat trial * CB + chain block), session d = sess[flat trial] (written by
// mnle_hoist_kernel), whose T_d trials start at trial_offsets[d].
// Launch shape of the potential kernel: whole waves of two-tile CTAs (one CTA per SM), and the tiles that
// are left over once the last FULL wave of pairs is placed go one per CTA when that fits a single wave --
// a half-empty wave of pairs costs a whole pair time (400 tiles on 148 SMs: 148 pairs + 104 singles
// instead of 200 pairs in two waves).  CTAs are scheduled in index order, so the singles run last.
static void tc_grid(long long n_tiles, int sms, int *n_pairs, long long *grid)
{
    const long long per_wave = 2ll * sms;
    const long long rem = n_tiles % per_wave;
    long long pairs = n_tiles / 2, singles = n_tiles & 1;
    if (n_tiles > per_wave && rem > 0 && rem <= sms) {
        pairs = (n_tiles - rem) / 2;
        singles = rem;
    }
    *n_pairs = (int)pairs;
    *grid = pairs + singles;
}

// Launch shape of the training kernels, per net (grid = (11 nets, *grid)): a 4 096-row minibatch is 32 tiles
// x 11 nets = 176 two-tile CTAs on 148 SMs, i.e. a second wave that is 19 % full and costs a whole pair time.
// When the pairs that do not fit whole waves can run as ONE wave of one-tile CTAs instead, they do (13 pairs
// + 6 singles per net: 143 + 66 CTAs; a single takes about 0.6 of a pair time).
static void train_grid(long long n_tiles, int sms, int *n_pairs, long long *grid, int nets = kNets)
{
    long long pairs = n_tiles / 2;
    const long long all = pairs * nets, rem = all % sms;
    if (all > sms && rem > 0) {
        const long long fewer = (all - rem) / nets;
        if ((n_tiles - 2 * fewer) * nets <= sms) pairs = fewer;
    }
    *n_pairs = (int)pairs;
    *grid = pairs + (n_tiles - 2 * pairs);
}

// ROWS: estimator.log_prob over arbitrary rows -- `theta` is the (R, 85) condition matrix (row stride
// ld_theta), x is (R, 2), C = R; the 86-wide context of each tile sits in shared memory as bf16 hi / lo
// A images and every net's first layer is a K = 96 stage with both operands from shared memory (the
// other stages take A from tensor memory as in potential mode); out[row] = log-prob.
// KEEP (rows mode only, the training forward): minibatch row c reads dataset row row_index[c] (null:
// identity), and the hidden activations, raw spline parameters and choice logits of every row below
// keep.Rp are written out for the backward pass (TcTrainDump).
// BWD (rows layout, the training backward-data pass): the A image of a net's first stage holds the
// gradient rows (d loss / d spline parameters or logits), the weight images are the transposed ones, and
// every epilogue multiplies by the activation derivative (tc_epilogue_mask) and writes keep.DH.
template <bool ROWS, bool KEEP = false, bool BWD = false, bool POT = false, bool SESS = false>
__global__ void __launch_bounds__(kTcThreads, 1)
    mnle_tc_kernel(const unsigned char *__restrict__ pack, const __grid_constant__ TcPlan plan,
                   const float *__restrict__ theta, long long ld_theta, const float *__restrict__ x,
                   const float *__restrict__ hoist, int D, int T, int C, int n_pairs, float mu_y, float sigma_y,
                   int n_choices,
                   float *__restrict__ partial, unsigned int *__restrict__ counters, float *__restrict__ out,
                   long long *__restrict__ trace, const long long *__restrict__ row_index = nullptr,
                   TcTrainDump keep = TcTrainDump{}, const int *__restrict__ sess = nullptr,
                   const long long *__restrict__ trial_offsets = nullptr)
{
    static_assert(ROWS || !KEEP, "only the rows-mode kernel keeps activations");
    static_assert(!BWD || (ROWS && !KEEP), "the backward pass uses the rows-mode layout");
    static_assert(!POT || BWD, "POT selects the potential-gradient flavour of the backward pass");
    static_assert(!SESS || !ROWS, "ragged sessions are a potential-mode layout");
    extern __shared__ __align__(1024) unsigned char smem[];
    using SM = TcSmem<ROWS>;
    constexpr int kTcSlots = SM::kSlots;
    constexpr uint32_t kSmemSlot0 = SM::kSlot0, kSmemBars = SM::kBars, kSmemATh = SM::kA;
    uint64_t *wfull = reinterpret_cast<uint64_t *>(smem + kSmemBars);  // [kTcSlots]
    uint64_t *dfull = wfull + 3;                                       // [kTcTiles]
    uint64_t *aready = dfull + kTcTiles;                               // [kTcTiles]
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(smem + kSmemBars + 96);
    // turn[X]: phase s completes when the issuer of stage s has consumed its aready[X] phase (issuers only)
    uint64_t *turn = aready + kTcTiles;                                // [kTcTiles]
    uint64_t *cfull = turn + kTcTiles;                                 // [kTcTiles] KEEP: context images landed
    // dth[X]: accumulators of a THETA stage are complete.  Theta stages have a barrier of their own because only
    // the hf = 1 warps take part in them: were they counted on dfull, an hf = 0 warp still in the tail of the
    // previous spline could find dfull TWO phases ahead (theta stage and the next layer both committed), take
    // the parity of the newer phase for the one it waits for and block for good -- a deadlock seen once in
    // ~1e7 tiles.  Every thread waits for every phase of the barriers it uses; phases are counted per barrier.
    uint64_t *dth = reinterpret_cast<uint64_t *>(smem + kSmemBars + 104);  // [kTcTiles]

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int CB = (C + kTcM - 1) / kTcM;
    // The training forward (KEEP) does not chain the splines (the per-row kernel does), so the eleven nets
    // are independent: blockIdx.x picks one net and the CTA runs only that net's 3 or 4 stages -- 11 x
    // more CTAs for a minibatch that is only a few dozen row tiles.  Barrier phases count local stages.
    // Training grids are (net, CTA of the net): CTAs are scheduled x-fastest, so every net's two-tile CTAs
    // start before any one-tile CTA does (see train_grid()).
    const int net_id = KEEP ? keep.net0 + (int)blockIdx.x : (BWD ? (int)blockIdx.x : 0);
    const int s_off = KEEP ? (net_id == 0 ? 0 : 4 + 3 * (net_id - 1)) : (BWD ? (net_id == 0 ? 0 : 3 + 2 * (net_id - 1)) : 0);
    const int n_st = KEEP ? (net_id == 0 ? 4 : 3) : (BWD ? (net_id == 0 ? 3 : 2) : kTcStages);
    // CTAs [0, n_pairs) take two tiles each, the rest one tile each (see tc_grid())
    const int bx = (KEEP || BWD) ? (int)blockIdx.y : (int)blockIdx.x;
    const int tile0 = bx >= n_pairs ? 2 * n_pairs + (bx - n_pairs) : bx * kTcTiles;
    const int n_active = bx >= n_pairs ? 1 : kTcTiles;

    // potential gradient: the theta columns of this net's first layer, [128][8] floats, in the unused tail of tile 0's
    // first A image (the backward pass fills K groups 0..9 of an image, this is groups 10 and 11)
    float *w1s = reinterpret_cast<float *>(smem + kSmemATh + 10u * kKGroupBytes);
    if (BWD && POT)
        for (int i = tid; i < kHidden * 8; i += kTcThreads) w1s[i] = __ldg(keep.W1T + (size_t)net_id * kHidden * 8 + i);
    if (warp == kTcEpiWarps) tmem_alloc<512>(tmem_slot);
    if (tid == 0) {
        for (int i = 0; i < kTcTiles; ++i) mbar_init(&turn[i], 1);
        for (int i = 0; i < kTcTiles; ++i) mbar_init(&cfull[i], 1);
        for (int i = 0; i < kTcTiles; ++i) mbar_init(&dth[i], 1);
        for (int i = 0; i < kTcSlots; ++i) mbar_init(&wfull[i], 1);
        for (int i = 0; i < kTcTiles; ++i) {
            mbar_init(&dfull[i], 1);
            mbar_init(&aready[i], kTcEpiThreads / kTcTiles);
        }
        fence_mbar_init();
    }
    tc_fence_before_sync();
    __syncthreads();
    tc_fence_after_sync();
    const uint32_t tmem = *tmem_slot;

    if (warp >= kTcEpiWarps) {
        // ================= issuers: bulk copies of the stage blobs + every tcgen05.mma =========
        // The whole warp walks the (uniform) stage loop; one elected lane issues.  Two issuer warps take
        // alternate stages.  Per stage an issuer spends ~700 cycles building the sixteen operand
        // descriptors on the uniform datapath, ~220 in the commit and 300-500 issuing the next bulk copies
        // (measured with the clock64 trace); a single issuer did that with the tensor pipe idle between
        // stages.  Now one warp prepares stage s + 1 while the other is blocked in the MMA queue of stage s.
        // A stage's MMAs wait for its A operand (aready), which exists only after the previous stage's
        // accumulators were committed and drained; the only extra ordering is `turn` (below).
        const int iw = warp - kTcEpiWarps;
        const uint32_t tmem_u = __shfl_sync(0xFFFFFFFFu, tmem, 0);
        const int t_of[2] = {tile0 / CB, (tile0 + 1) / CB};
        auto load = [&](int s) {
            const TcStage &st = plan.st[s_off + s];
            unsigned char *slot = smem + kSmemSlot0 + (uint32_t)(s % kTcSlots) * kSlotBytes;
            uint64_t *bar = &wfull[s % kTcSlots];
            if (elect_one_sync()) {
                mbar_expect_tx(bar, st.bytes + (st.kind != kStageTheta ? 0u : (uint32_t)n_active * kHidden * 4u));
                bulk_g2s(slot, pack + st.off, st.bytes, bar);
                if (st.kind == kStageTheta) {
                    bulk_g2s(slot + st.bytes, hoist + ((size_t)t_of[0] * kNets + st.net) * kHidden, kHidden * 4, bar);
                    if (n_active > 1)
                        bulk_g2s(slot + st.bytes + kHidden * 4, hoist + ((size_t)t_of[1] * kNets + st.net) * kHidden,
                                 kHidden * 4, bar);
                }
            }
            __syncwarp();
        };
        // the ring is kTcSlots deep: stage s + kTcSlots - 1 is fetched while stage s runs
        for (int g = iw; g < kTcSlots - 1; g += kTcIssuers) load(g);
#pragma unroll 1
        for (int s = iw; s < n_st; s += kTcIssuers) {
            const TcStage &st = plan.st[s_off + s];
            const uint32_t slot = smem_u32(smem + kSmemSlot0 + (uint32_t)(s % kTcSlots) * kSlotBytes);
            const uint32_t n = st.n, idesc = umma_idesc_bf16_f32(kTcM, (int)n);
#pragma unroll 1
            for (int X = 0; X < n_active; ++X) {
                if (trace && blockIdx.x == 0 && lane == 0) trace[(s * 2 + X) * 8 + 5] = clock64();
                // A parity wait cannot tell phase s from phase s - 2: first make sure the other issuer has
                // consumed phase s - 1 (then aready is in phase s or s + 1 and its parity is unambiguous;
                // turn itself is unambiguous because this warp completed its phase s - 2)
                if (s > 0) mbar_wait(&turn[X], (s - 1) & 1);
                mbar_wait(&aready[X], s & 1);  // A operand of this stage written, D drained
                if (elect_one_sync()) mbar_arrive(&turn[X]);
                __syncwarp();
                tc_fence_after_sync();
                if (trace && blockIdx.x == 0 && lane == 0) trace[(s * 2 + X) * 8 + 0] = clock64();
                if (X == 0) mbar_wait(&wfull[s % kTcSlots], (s / kTcSlots) & 1);
                if (trace && blockIdx.x == 0 && lane == 0) trace[(s * 2 + X) * 8 + 1] = clock64();
                const uint32_t tm = tmem_u + (uint32_t)X * kTmemTile;
                if (elect_one_sync()) {
                    if (st.kind == kStageInput) {
                        // K of the operand images: the 96 context columns, or (BWD) what the plan says
                        const int ksteps = BWD ? (int)(st.pad >> 8) : kInputK / 16;
                        const uint32_t w_img = kHidden * (uint32_t)ksteps * 32u;
                        const uint32_t ctx = smem_u32(smem + kSmemATh + (uint32_t)X * 2u * kCtxImgBytes);
#pragma unroll
                        for (int pass = 0; pass < 3; ++pass) {
                            const uint32_t a = ctx + (pass == 2 ? kCtxImgBytes : 0u);
                            const uint32_t w = slot + (pass == 1 ? w_img : 0u);
#pragma unroll 1
                            for (int ks = 0; ks < ksteps; ++ks)
                                umma_bf16(tm + kTmemD, umma_desc_kmajor(a + ks * 2 * kKGroupBytes, kKGroupBytes, 128),
                                          umma_desc_kmajor(w + ks * 2 * kKGroupBytes, kKGroupBytes, 128), idesc,
                                          (pass | ks) != 0);
                        }
                    } else if (st.kind == kStageTheta) {
                        const uint32_t a = smem_u32(smem + kSmemATh + (uint32_t)X * kAThBytes);
#pragma unroll
                        for (int ks = 0; ks < 2; ++ks)
                            umma_bf16(tm + kTmemD, umma_desc_kmajor(a + ks * 2 * kKGroupBytes, kKGroupBytes, 128),
                                      umma_desc_kmajor(slot + ks * 2 * kKGroupBytes, kKGroupBytes, 128), idesc, ks);
                    } else {
                        const uint32_t w_img = n * 256u, w_kg = n * 16u;
#pragma unroll
                        for (int pass = 0; pass < 3; ++pass) {
                            const uint32_t a = tm + (pass == 2 ? kTmemALo : kTmemAHi);
                            const uint32_t w = slot + (pass == 1 ? w_img : 0u);
#pragma unroll
                            for (int ks = 0; ks < 8; ++ks)
                                umma_bf16_ts(tm + kTmemD, a + (uint32_t)ks * 8u,
                                             umma_desc_kmajor(w + ks * 2 * w_kg, w_kg, 128), idesc, (pass | ks) != 0);
                        }
                    }
                    if (trace && blockIdx.x == 0) trace[(s * 2 + X) * 8 + 4] = clock64();
                    umma_commit(st.kind == kStageTheta ? &dth[X] : &dfull[X]);
                }
                __syncwarp();
                // every tile is past stage s-1, so its slot can take the next stage to fetch (issued after
                // the MMAs: the copy has a whole stage of slack, the MMA issue is on the critical path)
                if (X == n_active - 1 && s + kTcSlots - 1 < n_st) load(s + kTcSlots - 1);
                if (trace && blockIdx.x == 0 && lane == 0) trace[(s * 2 + X) * 8 + 6] = clock64();
            }
        }
    } else if (((warp >> 2) & 1) < n_active) {
        // ====== epilogue warps: tile X, lane quarter q (thread = row), column half hf ==========
        const int X = (warp >> 2) & 1, q = warp & 3, hf = warp >> 3, r = 32 * q + lane;
        // t = flattened (dataset, trial) index, c = chain within the dataset
        const int tile = tile0 + X, t = tile / CB, cb = tile - t * CB, c = cb * kTcM + r;
        const int d = SESS ? __ldg(sess + t) : t / T;
        const bool live = c < C;
        const long long c_glob = (long long)d * C + c;
        const uint32_t trow = tmem + (uint32_t)X * kTmemTile + ((uint32_t)(32 * q) << 16);
        if (BWD) {
            // gradient row of this net's outputs -> bf16 hi / lo A images (K-major): 71 spline parameters in
            // K = 80 (this thread: 40 of them), or the choice logits in K = 16 (8 each)
            unsigned char *img_hi = smem + kSmemATh + (uint32_t)X * 2u * kCtxImgBytes, *img_lo = img_hi + kCtxImgBytes;
            const int net = net_id;
            const bool have = c_glob < keep.Rp;
            const float *grow = net == 0 ? keep.LG + (size_t)(have ? c_glob : 0) * kMaxChoices
                                         : keep.Q + ((size_t)(net - 1) * (size_t)keep.Rp + (size_t)(have ? c_glob : 0)) * 72;
            // all loads first (ten 16-byte loads of a spline-parameter row, 288-byte row stride), then the split
            float gv[40];
            int n_groups;
            if (net == 0) {
                n_groups = 1;
#pragma unroll
                for (int j = 0; j < 8; ++j) gv[j] = (have && hf == 0 && j < n_choices) ? grow[j] : 0.f;
            } else {
                n_groups = 5;
                const float4 *g4 = reinterpret_cast<const float4 *>(grow + 40 * hf);
#pragma unroll
                for (int j = 0; j < 10; ++j) {
                    const float4 t = have ? g4[j] : make_float4(0.f, 0.f, 0.f, 0.f);
                    gv[4 * j + 0] = t.x;
                    gv[4 * j + 1] = t.y;
                    gv[4 * j + 2] = t.z;
                    gv[4 * j + 3] = (40 * hf + 4 * j + 3 < kSplineOut) ? t.w : 0.f;  // column 71 of the row is padding
                }
            }
            const int kg0 = (net == 0 ? 1 : 5) * hf;
#pragma unroll
            for (int g = 0; g < 5; ++g) {
                if (g < n_groups) {
                    uint32_t hi[4], lo[4];
#pragma unroll
                    for (int j = 0; j < 4; ++j) split_bf16x2(gv[8 * g + 2 * j], gv[8 * g + 2 * j + 1], hi[j], lo[j]);
                    const uint32_t off = (uint32_t)(kg0 + g) * kKGroupBytes + (uint32_t)r * 16u;
                    *reinterpret_cast<uint4 *>(img_hi + off) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
                    *reinterpret_cast<uint4 *>(img_lo + off) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
                }
            }
        } else if (KEEP) {
            // the tile's context images were built by tc_prep_kernel (tc_ctx_tile): one bulk copy, everybody waits for it
            unsigned char *img_hi = smem + kSmemATh + (uint32_t)X * 2u * kCtxImgBytes;
            if (q == 0 && hf == 0 && lane == 0) {
                mbar_expect_tx(&cfull[X], 2u * kCtxImgBytes);
                bulk_g2s(img_hi, keep.ctx + (size_t)tile * 2u * kCtxImgBytes, 2u * kCtxImgBytes, &cfull[X]);
            }
            mbar_wait(&cfull[X], 0);
        } else if (ROWS) {
            // context row [cond (85), choice, 0...] -> bf16 hi / lo A images of this tile (K-major, like the
            // weights); this thread: k in [48 hf, 48 hf + 48)
            unsigned char *img_hi = smem + kSmemATh + (uint32_t)X * 2u * kCtxImgBytes, *img_lo = img_hi + kCtxImgBytes;
            const long long drow = (KEEP && row_index != nullptr && live) ? row_index[c_glob] : c_glob;
            const float *crow = theta + drow * ld_theta;
            const float ch = live ? __ldg(x + 2 * drow + 1) : 0.f;
#pragma unroll 1
            for (int k0 = 48 * hf; k0 < 48 * hf + 48; k0 += 8) {
                uint32_t hi[4], lo[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    float v[2];
#pragma unroll
                    for (int e = 0; e < 2; ++e) {
                        const int k = k0 + 2 * j + e;
                        v[e] = !live ? 0.f : (k < kCond ? __ldg(crow + k) : (k == kCond ? ch : 0.f));
                    }
                    split_bf16x2(v[0], v[1], hi[j], lo[j]);
                }
                const uint32_t off = (uint32_t)(k0 >> 3) * kKGroupBytes + (uint32_t)r * 16u;
                *reinterpret_cast<uint4 *>(img_hi + off) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
                *reinterpret_cast<uint4 *>(img_lo + off) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
            }
        } else {   // A image of the theta stage: k = term * 5 + i, terms t1 t1 t2 t1 t2 t3 (pairs with tc_pack_job's theta image)
            unsigned char *a_th = smem + kSmemATh + (uint32_t)X * kAThBytes;
            uint16_t tt[5][3];
#pragma unroll
            for (int i = 0; i < 5; ++i) split3_bf16(live ? __ldg(theta + c_glob * ld_theta + i) : 0.f, tt[i]);
            const int aterm[6] = {0, 0, 1, 0, 1, 2};
            uint16_t kv[32];
#pragma unroll
            for (int k = 0; k < 32; ++k) kv[k] = (k < 30) ? tt[k % 5][aterm[k / 5]] : (uint16_t)0;
#pragma unroll
            for (int g = 0; g < 4; ++g) {
                if ((g >> 1) != hf) continue;
                uint4 v;
                v.x = kv[8 * g + 0] | ((uint32_t)kv[8 * g + 1] << 16);
                v.y = kv[8 * g + 2] | ((uint32_t)kv[8 * g + 3] << 16);
                v.z = kv[8 * g + 4] | ((uint32_t)kv[8 * g + 5] << 16);
                v.w = kv[8 * g + 6] | ((uint32_t)kv[8 * g + 7] << 16);
                *reinterpret_cast<uint4 *>(a_th + (uint32_t)g * kKGroupBytes + (uint32_t)r * 16u) = v;
            }
        }
        fence_proxy_async_smem();
        mbar_arrive(&aready[X]);

        const long long xi = ROWS ? (live ? ((KEEP && row_index != nullptr) ? row_index[c_glob] : c_glob) : 0) : t;
        const bool kept = KEEP && c_glob < keep.Rp;  // padding rows up to Rp get defined values too
        // (the training kernels evaluate neither the splines nor the choice probability: train_rows_kernel does)
        const float rt = (BWD || KEEP) ? 1.0f : __ldg(x + 2 * xi);
        const int choice = (BWD || KEEP) ? 0 : (int)__ldg(x + 2 * xi + 1);
        const float y = logf(rt);
        // training forward: `hoist` points at (mu_y, sigma_y) in the parameter buffer (no host round trip)
        const float mu = KEEP ? __ldg(hoist) : mu_y, sigma = KEEP ? __ldg(hoist + 1) : sigma_y;
        float u = (y - mu) / sigma, logdet = -logf(sigma), lp = 0.f;
        uint32_t ph_d = 0u, ph_t = 0u;  // phases of dfull[X] / dth[X] this thread has waited for

#pragma unroll 1
        for (int s = 0; s < n_st; ++s) {
            const TcStage &st = plan.st[s_off + s];
            if (BWD) {
                const bool have = c_glob < keep.Rp;
                const size_t at = ((size_t)st.net * 3 + ((st.pad & 0xFF) - 1)) * kHidden * (size_t)keep.Rp + (size_t)(have ? c_glob : 0);
                float *d_row = POT ? nullptr : keep.DH + at;
                const bool last = !(s + 1 < n_st);
                const float *wsel = (POT && last) ? w1s : nullptr;   // the last stage ends at the first layer
                float acc5[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
                const uint32_t *m_row = !POT ? nullptr
                                        : keep.HM + (((size_t)st.net * 3 + ((st.pad & 0xFF) - 1)) * 4 + 2 * hf) * (size_t)keep.Rp +
                                              (size_t)(have ? c_glob : 0);
                if (st.epi == kEpiRelu)
                    tc_epilogue_mask<kEpiRelu, POT>(trow, 64 * hf, 64, keep.H + at, d_row, (size_t)keep.Rp, have, !last,
                                                    &dfull[X], ph_d & 1u, wsel, acc5, m_row);
                else
                    tc_epilogue_mask<kEpiSigmoid, POT>(trow, 64 * hf, 64, keep.H + at, d_row, (size_t)keep.Rp, have, !last,
                                                       &dfull[X], ph_d & 1u, wsel, acc5);
                if (POT && wsel != nullptr && have) {
#pragma unroll
                    for (int i = 0; i < 5; ++i)   // [net][hf][i][row]: a warp writes 32 consecutive rows of one plane
                        keep.GP[(((size_t)net_id * 2 + hf) * 5 + i) * (size_t)keep.Rp + (size_t)c_glob] = acc5[i];
                }
                ++ph_d;
                tc_fence_before_sync();
                mbar_arrive(&aready[X]);
                continue;
            }
            if (st.epi >= kEpiSpline && hf != 0) {  // row-wise epilogues are done by the hf = 0 thread of the row
                mbar_wait(&dfull[X], ph_d++ & 1u);  // (never arrive twice within one phase of aready)
                mbar_arrive(&aready[X]);
                continue;
            }
            if (st.kind == kStageTheta && hf == 0) {
                // theta stages belong to the hf = 1 warps (all 128 columns, arriving for both halves):
                // the stage follows a spline, whose tail the hf = 0 warps are still computing.  They do not
                // touch dth at all (see its declaration).
                continue;
            }
            mbar_wait(&wfull[s % kTcSlots], (s / kTcSlots) & 1);  // the bias travelled with the stage blob
            const float *bias = reinterpret_cast<const float *>(smem + kSmemSlot0 + (uint32_t)(s % kTcSlots) * kSlotBytes +
                                                                st.bias_off + (st.kind != kStageTheta ? 0u : (uint32_t)X * kHidden * 4u));
            if (st.kind == kStageTheta) mbar_wait(&dth[X], ph_t++ & 1u);
            else mbar_wait(&dfull[X], ph_d++ & 1u);
            tc_fence_after_sync();
            const bool tracer = trace && blockIdx.x == 0 && q == 0 && lane == 0 && hf == (st.kind != kStageTheta ? 0 : 1);
            if (tracer) trace[(s * 2 + X) * 8 + 2] = clock64();
            if (st.kind == kStageTheta) {
                if (st.epi == kEpiRelu) tc_epilogue_act<kEpiRelu>(trow, 0, kHidden, bias);
                else tc_epilogue_act<kEpiSigmoid>(trow, 0, kHidden, bias);
                tc_fence_before_sync();
                mbar_arrive_n(&aready[X], 2);
                if (tracer) trace[(s * 2 + X) * 8 + 3] = clock64();
                continue;
            }
            float *keep_h = nullptr;
            uint32_t *keep_m = nullptr;
            if (KEEP && kept && st.pad != 0) {
                if (keep.HM != nullptr && st.epi == kEpiRelu)   // potential gradient: sign masks instead of activations
                    keep_m = keep.HM + (((size_t)st.net * 3 + (st.pad - 1)) * 4 + 2 * hf) * (size_t)keep.Rp + (size_t)c_glob;
                else if (keep.H != nullptr)                      // (H == null: only logits and spline parameters are kept)
                    keep_h = keep.H + ((size_t)st.net * 3 + (st.pad - 1)) * kHidden * (size_t)keep.Rp + (size_t)c_glob;
            }
            if (st.epi == kEpiRelu) {
                tc_epilogue_act<kEpiRelu>(trow, 64 * hf, 64, bias, keep_h, (size_t)keep.Rp, keep_m);
            } else if (st.epi == kEpiSigmoid) {
                tc_epilogue_act<kEpiSigmoid>(trow, 64 * hf, 64, bias, keep_h, (size_t)keep.Rp);
            } else if (st.epi == kEpiSpline) {
                if (KEEP) {  // the splines are evaluated by the per-row kernel: only keep the raw parameters
                    float *dst = keep.Q + ((size_t)(st.net - 1) * (size_t)keep.Rp + (size_t)(kept ? c_glob : 0)) * 72;
#pragma unroll 1
                    for (int c0 = 0; c0 < kSplineN; c0 += 16) {  // 71 parameters in five 16-column blocks
                        uint32_t v[16];
                        tmem_ld16(trow + kTmemD + (uint32_t)c0, v);
                        tmem_wait_ld();
                        if (kept) {
#pragma unroll
                            for (int j = 0; j < 16; j += 4) {
                                if (c0 + j + 3 < kSplineOut) {
                                    *reinterpret_cast<float4 *>(dst + c0 + j) = make_float4(
                                        __uint_as_float(v[j]) + bias[c0 + j], __uint_as_float(v[j + 1]) + bias[c0 + j + 1],
                                        __uint_as_float(v[j + 2]) + bias[c0 + j + 2], __uint_as_float(v[j + 3]) + bias[c0 + j + 3]);
                                } else {
#pragma unroll
                                    for (int e = 0; e < 4; ++e)
                                        if (c0 + j + e < kSplineOut) dst[c0 + j + e] = __uint_as_float(v[j + e]) + bias[c0 + j + e];
                                }
                            }
                        }
                    }
                    tc_fence_before_sync();
                    mbar_arrive(&aready[X]);
                } else {
                    tc_epilogue_spline(trow, bias, u, logdet, &aready[X]);
                }
                if (tracer) trace[(s * 2 + X) * 8 + 3] = clock64();
                continue;
            } else {
                uint32_t v[16];
                tmem_ld16(trow + kTmemD, v);
                tmem_wait_ld();
                float lg[kMaxChoices];
#pragma unroll
                for (int j = 0; j < kMaxChoices; ++j) lg[j] = __uint_as_float(v[j]) + bias[j];
                if (KEEP && kept) {
#pragma unroll
                    for (int j = 0; j < kMaxChoices; ++j)
                        if (j < n_choices) keep.LG[(size_t)c_glob * kMaxChoices + j] = lg[j];
                }
                float m = -INFINITY;
#pragma unroll
                for (int j = 0; j < kMaxChoices; ++j)
                    if (j < n_choices) m = fmaxf(m, lg[j]);
                float sum = 0.f, pc = 0.f;
#pragma unroll
                for (int j = 0; j < kMaxChoices; ++j)
                    if (j < n_choices) {
                        const float ex = expf(lg[j] - m);
                        sum += ex;
                        if (j == choice) pc = ex;
                    }
                const float eps = 1.1920928955078125e-07f;
                lp = logf(fminf(fmaxf(pc / sum, eps), 1.0f - eps));
            }
            tc_fence_before_sync();
            mbar_arrive(&aready[X]);
            if (tracer) trace[(s * 2 + X) * 8 + 3] = clock64();
        }
        if (ROWS) {
            if (!KEEP && !BWD && hf == 0 && live) out[c_glob] = lp + (-0.5f * u * u - 0.9189385332046727f) + logdet - y;
        } else if (hf == 0) {
            // ---- sum over trials, fixed order: the tile that arrives last at its chain block adds
            // the T_d partial rows of its session (every run gives the same bits whichever tile that is)
            if (live) partial[(size_t)t * C + c] = lp + (-0.5f * u * u - 0.9189385332046727f) + logdet - y;
            const long long first = SESS ? __ldg(trial_offsets + d) : (long long)d * T;
            const int Td = SESS ? (int)(__ldg(trial_offsets + d + 1) - first) : T;
            uint32_t *last_s = tmem_slot + 1 + X;
            __threadfence();
            asm volatile("bar.sync %0, 128;" ::"r"(1 + X) : "memory");
            if (q == 0 && lane == 0) *last_s = (atomicAdd(&counters[d * CB + cb], 1u) == (unsigned)(Td - 1));
            asm volatile("bar.sync %0, 128;" ::"r"(1 + X) : "memory");
            if (*last_s && live) {
                __threadfence();
                const float *col = partial + (size_t)first * C + c;
                float sum = 0.f;
#pragma unroll 10
                for (int tt = 0; tt < Td; ++tt) sum += __ldcg(col + (size_t)tt * C);
                out[c_glob] = sum;
            }
        }
    }
    tc_fence_before_sync();
    __syncthreads();
    if (warp == kTcEpiWarps) tmem_dealloc<512>(tmem);
}

// ------------------------------------------------------------------------ operand packs ---
// Every operand pack is written on the device from the packed fp32 parameters (tc_prep_kernel), one pack job
// per stage blob: the handle's pack once, when mnle_create has copied the parameters, and the training pack
// every optimisation step, because the parameters change.
enum PackKind : uint16_t {
    kPackDense = 0,       // image row = row of W, k = column of W: hi image, lo image, bias
    kPackTransposed = 1,  // image row = column of W, k = row of W: hi image, lo image (backward-data stages)
    kPackTheta = 2,       // theta image of W's first five columns (tc_pack_job): one image, no bias
};
struct PackJob {
    uint32_t w_off, b_off;      // weight / bias position in the packed parameters (floats)
    uint32_t dst, img_bytes;    // blob position in the pack, bytes of one image (hi; lo follows)
    uint16_t n_valid, k_valid;  // W is [n_valid][k_valid] row-major
    uint16_t n_img, kind;       // rows of the image (UMMA N); PackKind
};
constexpr int kTrainStages = kTcStages + 3 + 2 * kTransforms;  // forward stages + backward-data stages
struct PackJobs {
    PackJob j[kTrainStages];  // (the training pack has the most jobs)
    int n;
};

constexpr int kPackSplit = 8;  // CTAs per pack job

// One launch prepares everything the tensor-core kernels read: CTAs [0, jobs.n * kPackSplit) write the
// operand pack from the current parameters -- every byte of it, padding rows / columns and padding biases
// included, so the caller's workspace needs no clearing --, the others build the context images of one row
// tile each (tc_ctx_tile below).
__device__ __forceinline__ void tc_pack_job(const float *__restrict__ params, const PackJob &J, int part,
                                            unsigned char *__restrict__ pack)
{
    const int n_img = J.n_img, k_img = (int)(J.img_bytes / (2u * J.n_img));
    const int total = n_img * k_img;
    for (int idx = part * blockDim.x + threadIdx.x; idx < total; idx += kPackSplit * blockDim.x) {
        if (J.kind == kPackTheta) {
            // [n_img][32]: k = term * 5 + i holds term {0, 1, 0, 2, 1, 0}[term] of the three-term split of W[r][i],
            // paired with the A terms t1 t1 t2 t1 t2 t3 mnle_tc_kernel builds (all products of order <= 4); k = 30, 31: 0
            const int r = idx / k_img, k = idx - r * k_img, term = k / 5;
            uint16_t t[3] = {0, 0, 0};
            if (k < 30) split3_bf16(params[J.w_off + r * J.k_valid + (k - 5 * term)], t);
            *reinterpret_cast<uint16_t *>(pack + J.dst + tile_offset(n_img, r, k)) =
                term == 3 ? t[2] : (term == 1 || term == 4) ? t[1] : t[0];
            continue;
        }
        int r, k;  // image row, k; consecutive threads read consecutive parameters
        float v = 0.f;
        if (J.kind == kPackDense) {
            r = idx / k_img;
            k = idx - r * k_img;
            if (r < J.n_valid && k < J.k_valid) v = params[J.w_off + r * J.k_valid + k];
        } else {  // image row = column of W, k = row of W
            k = idx / n_img;
            r = idx - k * n_img;
            if (k < J.n_valid && r < J.k_valid) v = params[J.w_off + k * J.k_valid + r];
        }
        uint16_t hi, lo;
        split_bf16(v, hi, lo);
        const uint32_t off = J.dst + tile_offset(n_img, r, k);
        *reinterpret_cast<uint16_t *>(pack + off) = hi;
        *reinterpret_cast<uint16_t *>(pack + off + J.img_bytes) = lo;
    }
    if (part == 0 && J.kind == kPackDense)
        for (int n = threadIdx.x; n < n_img; n += blockDim.x)
            reinterpret_cast<float *>(pack + J.dst + 2 * J.img_bytes)[n] = n < J.n_valid ? params[J.b_off + n] : 0.f;
}

// Stage plans and pack jobs of the two operand packs (null outputs are skipped); returns the pack's bytes.
// Both packs start with the forward stages, in `plan` (the rows-mode plan): cat (first layer, W1, W2, Wo),
// then flow 0..9 (first layer, W2, W3), every first layer a K = 96 stage.  The training pack (theta = false)
// continues with the backward-data stages, in `tail` in the order of the backward pass; the handle's pack
// (theta = true) with one theta stage per net, net i's in tail->st[i].
static size_t pack_plan(const Layout &L, bool theta, TcPlan *plan, TcPlan *tail, PackJobs *jobs)
{
    size_t bytes = 0;
    int s = 0;
    if (jobs) jobs->n = 0;
    auto stage = [&](size_t W, size_t b, int n_valid, int k_valid, int n_img, int k_img, int kind, int epi, int net, int slot) {
        const uint32_t img = (uint32_t)n_img * (uint32_t)k_img * 2u;
        if (plan) {
            TcStage &st = plan->st[s];
            st.off = (uint32_t)bytes;
            st.bytes = 2u * img + (uint32_t)n_img * 4u;
            st.bias_off = 2u * img;
            st.n = (uint16_t)n_img;
            st.kind = (uint8_t)kind;
            st.epi = (uint8_t)epi;
            st.net = (uint16_t)net;
            st.pad = (uint16_t)slot;
        }
        if (jobs)
            jobs->j[jobs->n++] = PackJob{(uint32_t)W, (uint32_t)b, (uint32_t)bytes, img, (uint16_t)n_valid,
                                         (uint16_t)k_valid, (uint16_t)n_img, kPackDense};
        bytes += 2u * img + (uint32_t)n_img * 4u;
        ++s;
    };
    stage(L.cat_W0, L.cat_b0, kHidden, kCond, kHidden, kInputK, kStageInput, kEpiSigmoid, 0, 1);
    stage(L.cat_W1, L.cat_b1, kHidden, kHidden, kHidden, kHidden, kStageK128, kEpiSigmoid, 0, 2);
    stage(L.cat_W2, L.cat_b2, kHidden, kHidden, kHidden, kHidden, kStageK128, kEpiSigmoid, 0, 3);
    stage(L.cat_Wo, L.cat_bo, L.n_choices, kHidden, 16, kHidden, kStageK128, kEpiCategorical, 0, 0);
    for (int k = 0; k < kTransforms; ++k) {
        stage(L.fl_W1[k], L.fl_b1[k], kHidden, kCtx, kHidden, kInputK, kStageInput, kEpiRelu, 1 + k, 1);
        stage(L.fl_W2[k], L.fl_b2[k], kHidden, kHidden, kHidden, kHidden, kStageK128, kEpiRelu, 1 + k, 2);
        stage(L.fl_W3[k], L.fl_b3[k], kSplineOut, kHidden, kSplineN, kHidden, kStageK128, kEpiSpline, 1 + k, 0);
    }
    if (theta) {
        // theta stage: the image alone; its bias is the net's per-trial first-layer sum (mnle_hoist_kernel),
        // which the potential kernel stages right behind the image
        auto tstage = [&](size_t W, int ldw, int epi, int net) {
            const uint32_t img = (uint32_t)kHidden * 32u * 2u;
            if (tail)
                tail->st[net] = TcStage{(uint32_t)bytes, img, img, (uint16_t)kHidden, (uint8_t)kStageTheta, (uint8_t)epi,
                                        (uint16_t)net, 0};
            if (jobs)
                jobs->j[jobs->n++] = PackJob{(uint32_t)W, 0u, (uint32_t)bytes, img, (uint16_t)kHidden, (uint16_t)ldw,
                                             (uint16_t)kHidden, kPackTheta};
            bytes += img;
        };
        tstage(L.cat_W0, kCond, kEpiSigmoid, 0);
        for (int k = 0; k < kTransforms; ++k) tstage(L.fl_W1[k], kCtx, kEpiRelu, 1 + k);
        return bytes;
    }
    // backward-data: out[row][in] = sum_out g[row][out] W[out][in]  ->  B image = W transposed ([in][out], K = out)
    int bs = 0;
    auto bstage = [&](size_t W, int n_out, int n_in, int k_img, int kind, int epi, int net, int mask_slot) {
        const uint32_t img = (uint32_t)kHidden * (uint32_t)k_img * 2u;  // n_in = 128 rows everywhere
        if (tail) {
            TcStage &st = tail->st[bs];
            st.off = (uint32_t)bytes;
            st.bytes = 2u * img;
            st.bias_off = 2u * img;
            st.n = (uint16_t)kHidden;
            st.kind = (uint8_t)kind;
            st.epi = (uint8_t)epi;
            st.net = (uint16_t)net;
            st.pad = (uint16_t)((mask_slot + 1) | ((k_img / 16) << 8));
        }
        if (jobs)
            jobs->j[jobs->n++] = PackJob{(uint32_t)W, 0u, (uint32_t)bytes, img, (uint16_t)n_out, (uint16_t)n_in,
                                         (uint16_t)kHidden, kPackTransposed};
        bytes += 2u * img;
        ++bs;
    };
    bstage(L.cat_Wo, L.n_choices, kHidden, 16, kStageInput, kEpiSigmoid, 0, 2);
    bstage(L.cat_W2, kHidden, kHidden, kHidden, kStageK128, kEpiSigmoid, 0, 1);
    bstage(L.cat_W1, kHidden, kHidden, kHidden, kStageK128, kEpiSigmoid, 0, 0);
    for (int k = 0; k < kTransforms; ++k) {
        bstage(L.fl_W3[k], kSplineOut, kHidden, kSplineN, kStageInput, kEpiRelu, 1 + k, 1);
        bstage(L.fl_W2[k], kHidden, kHidden, kHidden, kStageK128, kEpiRelu, 1 + k, 0);
    }
    return bytes;
}

// The eleven nets of a row tile all start from the same 86-wide context.  Instead of every CTA gathering
// and splitting its tile's rows itself (27 k cycles before its first MMA, eleven times per tile), the
// bf16 hi / lo A images of every tile are built once per step and the CTAs fetch them with one bulk copy.
// grid = tiles, 384 threads: thread = (row, third of the 96 k's).
__device__ __forceinline__ void tc_ctx_tile(int tile, const float *__restrict__ x, const float *__restrict__ cond,
                                            long long ld_cond, const long long *__restrict__ row_index, long long R,
                                            unsigned char *__restrict__ out, float *__restrict__ cx, long long Rp)
{
    const int r = threadIdx.x & 127, part = threadIdx.x >> 7;
    const long long row = (long long)tile * kTcM + r;
    const bool live = row < R;
    const long long drow = live ? (row_index ? row_index[row] : row) : 0;
    const float *crow = cond + drow * ld_cond;
    unsigned char *img_hi = out + (size_t)tile * 2u * kCtxImgBytes, *img_lo = img_hi + kCtxImgBytes;
    float v[32];
#pragma unroll
    for (int e = 0; e < 32; ++e) {
        const int k = 32 * part + e;
        v[e] = !live ? 0.f : (k < kCond ? __ldg(crow + k) : (k == kCond ? __ldg(x + 2 * drow + 1) : 0.f));
    }
    if (cx != nullptr && row < Rp) {  // fp32 copy for the weight-gradient GEMMs: lanes = consecutive rows of a column
#pragma unroll
        for (int e = 0; e < 32; ++e)
            if (32 * part + e <= kCond) cx[(size_t)(32 * part + e) * (size_t)Rp + (size_t)row] = v[e];
    }
#pragma unroll
    for (int g = 0; g < 4; ++g) {
        uint32_t hi[4], lo[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) split_bf16x2(v[8 * g + 2 * j], v[8 * g + 2 * j + 1], hi[j], lo[j]);
        const uint32_t off = (uint32_t)(4 * part + g) * kKGroupBytes + (uint32_t)r * 16u;
        *reinterpret_cast<uint4 *>(img_hi + off) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
        *reinterpret_cast<uint4 *>(img_lo + off) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
    }
}

__global__ void __launch_bounds__(384) tc_prep_kernel(const float *__restrict__ params, const __grid_constant__ PackJobs jobs,
                                                      unsigned char *__restrict__ pack, const float *__restrict__ x,
                                                      const float *__restrict__ cond, long long ld_cond,
                                                      const long long *__restrict__ row_index, long long R,
                                                      unsigned char *__restrict__ ctx, float *__restrict__ cx, long long Rp)
{
    const int pack_ctas = jobs.n * kPackSplit;
    if ((int)blockIdx.x < pack_ctas) tc_pack_job(params, jobs.j[blockIdx.x / kPackSplit], (int)blockIdx.x % kPackSplit, pack);
    else tc_ctx_tile((int)blockIdx.x - pack_ctas, x, cond, ld_cond, row_index, R, ctx, cx, Rp);
}

// The handle's pack from the parameters mnle_create copied to the device (legacy default stream, waited for):
// tc_rows_plan is the forward plan, tc_plan the same with every first layer replaced by the net's theta stage.
int tc_handle_pack(Handle *H)
{
    TcPlan theta;
    PackJobs jobs;
    const size_t bytes = pack_plan(H->layout, true, &H->tc_rows_plan, &theta, &jobs);
    H->tc_plan = H->tc_rows_plan;
    for (TcStage &st : H->tc_plan.st)
        if (st.kind == kStageInput) st = theta.st[st.net];
    DDM_CUDA_TRY(cudaMalloc(&H->tc_pack, bytes));
    tc_prep_kernel<<<(unsigned)(jobs.n * kPackSplit), 384>>>(H->params, jobs, static_cast<unsigned char *>(H->tc_pack), nullptr,
                                                             nullptr, 0, nullptr, 0, nullptr, nullptr, 0);
    DDM_CUDA_TRY(cudaGetLastError());
    DDM_CUDA_TRY(cudaStreamSynchronize(0));
    return DDM_OK;
}

static size_t train_pack_only_bytes(const Layout &L)
{
    return (pack_plan(L, false, nullptr, nullptr, nullptr) + 127) / 128 * 128;
}

size_t tc_train_pack_bytes(int n_choices, long long R)
{
    return train_pack_only_bytes(make_layout(n_choices)) + (size_t)((R + kTcM - 1) / kTcM) * 2u * kCtxImgBytes;
}

int tc_train_forward(const float *params_dev, const Layout &L, void *pack_dev, const float *x_dev, const float *cond_dev,
                     long long ld_cond, const long long *row_index_dev, long long R, const TcTrainDump &dump,
                     float *lp_dev, cudaStream_t st)
{
    TcPlan plan;
    PackJobs jobs;
    pack_plan(L, false, &plan, nullptr, &jobs);
    DDM_REQUIRE((reinterpret_cast<uintptr_t>(pack_dev) & 15u) == 0, "tc_train_forward: pack must be 16-byte aligned");
    DDM_REQUIRE(dump.net0 >= 0 && dump.nets >= 1 && dump.net0 + dump.nets <= kNets, "tc_train_forward: bad net range");
    if (dump.net0 > 0) jobs.n = 0;  // the pack was written by this call's launch from net 0: context images only
    unsigned char *ctx_dev = static_cast<unsigned char *>(pack_dev) + train_pack_only_bytes(L);
    tc_prep_kernel<<<(unsigned)(jobs.n * kPackSplit + (R + kTcM - 1) / kTcM), 384, 0, st>>>(
        params_dev, jobs, static_cast<unsigned char *>(pack_dev), x_dev, cond_dev, ld_cond, row_index_dev, R, ctx_dev, dump.CX,
        dump.Rp);
    DDM_CUDA_TRY(cudaGetLastError());
    TcTrainDump keep = dump;
    keep.ctx = ctx_dev;
    int dev = 0, sms = 0, n_pairs = 0;
    long long grid = 0;
    DDM_CUDA_TRY(cudaGetDevice(&dev));
    DDM_CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    train_grid((R + kTcM - 1) / kTcM, sms, &n_pairs, &grid, dump.nets);
    DDM_REQUIRE(grid <= 65535, "training minibatch too large for one launch (at most ~8e6 rows)");
    DDM_CUDA_TRY(cudaFuncSetAttribute(mnle_tc_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)TcSmem<true>::kBytes));
    // (mu_y, sigma_y) sit at the tail of the parameter buffer: the kernel reads them through `hoist`
    mnle_tc_kernel<true, true><<<dim3((unsigned)dump.nets, (unsigned)grid), kTcThreads, TcSmem<true>::kBytes, st>>>(
        static_cast<const unsigned char *>(pack_dev), plan, cond_dev, ld_cond, x_dev, params_dev + L.mu_y, 1, 1, (int)R,
        n_pairs, 0.f, 1.f, L.n_choices, nullptr, nullptr, lp_dev, nullptr, row_index_dev, keep);
    DDM_CUDA_TRY(cudaGetLastError());
    return DDM_OK;
}

int tc_train_backward(const Layout &L, const void *pack_dev, long long R, const TcTrainDump &dump, cudaStream_t st)
{
    TcPlan bplan;
    pack_plan(L, false, nullptr, &bplan, nullptr);
    int dev = 0, sms = 0, n_pairs = 0;
    long long grid = 0;
    DDM_CUDA_TRY(cudaGetDevice(&dev));
    DDM_CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    train_grid((R + kTcM - 1) / kTcM, sms, &n_pairs, &grid);
    DDM_REQUIRE(grid <= 65535, "training minibatch too large for one launch (at most ~8e6 rows)");
    if (dump.GP != nullptr) {   // the potential's gradient: sign masks in, five numbers per row out
        DDM_REQUIRE(dump.HM != nullptr && dump.W1T != nullptr, "tc_train_backward: potential mode needs HM and W1T");
        DDM_CUDA_TRY(cudaFuncSetAttribute(mnle_tc_kernel<true, false, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          (int)TcSmem<true>::kBytes));
        mnle_tc_kernel<true, false, true, true><<<dim3(kNets, (unsigned)grid), kTcThreads, TcSmem<true>::kBytes, st>>>(
            static_cast<const unsigned char *>(pack_dev), bplan, nullptr, 0, nullptr, nullptr, 1, 1, (int)R, n_pairs, 0.f, 1.f,
            L.n_choices, nullptr, nullptr, nullptr, nullptr, nullptr, dump);
    } else {
        DDM_CUDA_TRY(cudaFuncSetAttribute(mnle_tc_kernel<true, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          (int)TcSmem<true>::kBytes));
        mnle_tc_kernel<true, false, true><<<dim3(kNets, (unsigned)grid), kTcThreads, TcSmem<true>::kBytes, st>>>(
            static_cast<const unsigned char *>(pack_dev), bplan, nullptr, 0, nullptr, nullptr, 1, 1, (int)R, n_pairs, 0.f, 1.f,
            L.n_choices, nullptr, nullptr, nullptr, nullptr, nullptr, dump);
    }
    DDM_CUDA_TRY(cudaGetLastError());
    return DDM_OK;
}

}  // namespace mnle

using namespace mnle;

DDM_API int mnle_tc_selftest(const float *a_dev, const float *b_dev, int N, int passes, uint32_t lbo_a, uint32_t lbo_b,
                             uint32_t sbo, float *d_dev, void *stream)
{
    DDM_REQUIRE(a_dev && b_dev && d_dev, "mnle_tc_selftest: null pointer");
    DDM_REQUIRE(N >= 16 && N <= 128 && N % 16 == 0, "mnle_tc_selftest: N=%d must be a multiple of 16 in [16,128]", N);
    DDM_REQUIRE(passes == 1 || passes == 3 || passes == 11 || passes == 13 || (passes > 100 && passes < 300),
                "mnle_tc_selftest: passes must be 1 or 3 (+10: A operand from TMEM; 100 + r / 200 + r: timing probe)");
    const int smem = 131072 + 64;
    DDM_CUDA_TRY(cudaFuncSetAttribute(tc_selftest_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    tc_selftest_kernel<<<1, 128, smem, static_cast<cudaStream_t>(stream)>>>(a_dev, b_dev, N, passes, lbo_a, lbo_b, sbo, d_dev);
    DDM_CUDA_TRY(cudaGetLastError());
    return DDM_OK;
}

// Debug aid (tools/trace_mnle_tc.py): device buffer of kTcStages * 2 * 8 clock64 stamps written by
// CTA 0 -- per (stage, tile): [0] issuer saw the A operand, [1] issuer had the weights, [2] epilogue saw
// the accumulators, [3] epilogue finished, [4] MMAs issued, [5] issuer reached the stage, [6] next bulk
// copies issued.  nullptr (default) = off.
static long long *g_tc_trace = nullptr;
DDM_API int mnle_tc_set_trace(long long *trace_dev)
{
    g_tc_trace = trace_dev;
    return DDM_OK;
}

// Workspace of the fused potential over N flat trials of D datasets / sessions, in floats: the per-trial first
// layers, the per-row partial sums, the arrival counters and (ragged sessions) the session of every trial.
static size_t tc_sum_workspace(float *base, long long D, long long N, long long C, bool sessions, float **hoist,
                               float **partial, unsigned int **counters, int **sess)
{
    const size_t n_hoist = (size_t)N * kNets * kHidden, n_partial = (size_t)N * (size_t)C;
    const size_t n_counters = (size_t)D * (size_t)((C + kTcM - 1) / kTcM);
    if (base != nullptr) {
        *hoist = base;
        *partial = base + n_hoist;
        *counters = reinterpret_cast<unsigned int *>(*partial + n_partial);
        *sess = sessions ? reinterpret_cast<int *>(base + n_hoist + n_partial + n_counters) : nullptr;
    }
    return n_hoist + n_partial + n_counters + (sessions ? (size_t)N : 0);
}

// The fused potential over N flat trials: D datasets of T trials each (trial_offsets == null, N = D * T), or D
// ragged sessions, session d owning flat trials [trial_offsets[d], trial_offsets[d + 1]) (T unused).
static int tc_loglik_sum(const char *entry, void *handle, const float *theta_dev, int64_t ld_theta, const float *x_dev,
                         const float *pulses_dev, int64_t ld_pulses, const int64_t *trial_offsets_dev, int64_t D, int64_t T,
                         int64_t N, int64_t C, float *out_dev, float *workspace_dev, void *stream)
{
    Handle *H = live_handle(handle, entry, true);
    if (H == nullptr) return DDM_ERR_STATE;
    DDM_REQUIRE(D >= 0 && T >= 0 && N >= 0 && C >= 0 && D <= 0x7FFFFFFFll && T <= 0x7FFFFFFFll && C <= 0x7FFFFFFFll - kTcM,
                "%s: D=%lld T=%lld N=%lld C=%lld out of range", entry, (long long)D, (long long)T, (long long)N, (long long)C);
    if (C == 0 || D == 0) return DDM_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    DDM_REQUIRE(out_dev != nullptr, "%s: null output", entry);
    if (N == 0) {
        DDM_CUDA_TRY(cudaMemsetAsync(out_dev, 0, (size_t)D * (size_t)C * sizeof(float), st));
        return DDM_OK;
    }
    DDM_REQUIRE(theta_dev && x_dev && pulses_dev && workspace_dev, "%s: null pointer", entry);
    DDM_REQUIRE(ld_theta >= 5 && ld_pulses >= kCond - 5, "%s: ld_theta=%lld ld_pulses=%lld too small", entry,
                (long long)ld_theta, (long long)ld_pulses);
    DDM_REQUIRE((reinterpret_cast<uintptr_t>(workspace_dev) & 15u) == 0, "%s: workspace must be 16-byte aligned", entry);
    const long long CB = (C + kTcM - 1) / kTcM;
    const long long n_tiles = N * CB;
    DDM_REQUIRE(N <= 0x7FFFFFFFll / kHoistTrials && n_tiles <= 0x7FFFFFFFll && D * CB <= 0x7FFFFFFFll,
                "%s: N * ceil(C / 128) = %lld tiles is too many", entry, n_tiles);
    float *hoist, *partial;
    unsigned int *counters;
    int *sess;
    tc_sum_workspace(workspace_dev, D, N, C, trial_offsets_dev != nullptr, &hoist, &partial, &counters, &sess);
    const long long hoist_blocks = (N + kHoistTrials - 1) / kHoistTrials;
    DDM_REQUIRE(hoist_blocks <= 65535, "%s: %lld trials is too many for one call", entry, (long long)N);
    const long long *offsets = reinterpret_cast<const long long *>(trial_offsets_dev);
    auto hoist_kernel = offsets != nullptr ? mnle_hoist_kernel<true> : mnle_hoist_kernel<false>;
    hoist_kernel<<<dim3(kNets, (unsigned)hoist_blocks), kHidden, 0, st>>>(H->params, H->layout, x_dev, pulses_dev, ld_pulses, (int)N,
                                                                       hoist, counters, (int)(D * CB), offsets, (int)D, (int)C, sess,
                                                                       out_dev);
    DDM_CUDA_TRY(cudaGetLastError());
    auto kernel = offsets != nullptr ? mnle_tc_kernel<false, false, false, false, true> : mnle_tc_kernel<false>;
    DDM_CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TcSmem<false>::kBytes));
    int sms = 0, n_pairs = 0;
    long long grid = 0;
    DDM_CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, H->device));
    tc_grid(n_tiles, sms, &n_pairs, &grid);
    kernel<<<(unsigned)grid, kTcThreads, TcSmem<false>::kBytes, st>>>(
        static_cast<const unsigned char *>(H->tc_pack), H->tc_plan, theta_dev, ld_theta, x_dev, hoist, (int)D, (int)T, (int)C,
        n_pairs, H->mu_y, H->sigma_y, H->layout.n_choices, partial, counters, out_dev, g_tc_trace, nullptr, TcTrainDump{}, sess,
        offsets);
    DDM_CUDA_TRY(cudaGetLastError());
    return DDM_OK;
}

DDM_API size_t mnle_loglik_batched_tc_workspace_floats(int64_t D, int64_t T, int64_t C)
{
    if (D <= 0 || T <= 0 || C <= 0) return 0;
    return tc_sum_workspace(nullptr, D, D * T, C, false, nullptr, nullptr, nullptr, nullptr);
}

DDM_API size_t mnle_loglik_tc_workspace_floats(int64_t T, int64_t C)
{
    return mnle_loglik_batched_tc_workspace_floats(1, T, C);
}

DDM_API size_t mnle_loglik_sessions_tc_workspace_floats(int64_t D, int64_t N, int64_t C)
{
    if (D <= 0 || N <= 0 || C <= 0) return 0;
    return tc_sum_workspace(nullptr, D, N, C, true, nullptr, nullptr, nullptr, nullptr);
}

DDM_API int mnle_loglik_sum_batched_tc_f32(void *handle, const float *theta_dev, int64_t ld_theta, const float *x_dev,
                                           const float *pulses_dev, int64_t ld_pulses, int64_t D, int64_t T, int64_t C,
                                           float *out_dev, float *workspace_dev, void *stream)
{
    const bool in_range = D >= 0 && T >= 0 && D <= 0x7FFFFFFFll && T <= 0x7FFFFFFFll;   // (N = -1 is reported as out of range)
    return tc_loglik_sum("mnle_loglik_sum_tc", handle, theta_dev, ld_theta, x_dev, pulses_dev, ld_pulses, nullptr, D, T,
                         in_range ? D * T : -1, C, out_dev, workspace_dev, stream);
}

DDM_API int mnle_loglik_sum_tc_f32(void *handle, const float *theta_dev, int64_t ld_theta, const float *x_dev,
                                   const float *pulses_dev, int64_t ld_pulses, int64_t T, int64_t C, float *out_dev,
                                   float *workspace_dev, void *stream)
{
    return mnle_loglik_sum_batched_tc_f32(handle, theta_dev, ld_theta, x_dev, pulses_dev, ld_pulses, 1, T, C, out_dev,
                                          workspace_dev, stream);
}

DDM_API int mnle_loglik_sum_sessions_tc_f32(void *handle, const float *theta_dev, int64_t ld_theta, const float *x_dev,
                                            const float *pulses_dev, int64_t ld_pulses, const int64_t *trial_offsets_dev,
                                            int64_t D, int64_t N, int64_t C, float *out_dev, float *workspace_dev, void *stream)
{
    DDM_REQUIRE(trial_offsets_dev != nullptr || D == 0, "mnle_loglik_sum_sessions_tc_f32: null trial_offsets");
    return tc_loglik_sum("mnle_loglik_sum_sessions_tc_f32", handle, theta_dev, ld_theta, x_dev, pulses_dev, ld_pulses,
                         trial_offsets_dev, D, 0, N, C, out_dev, workspace_dev, stream);
}

DDM_API int mnle_log_prob_rows_tc_f32(void *handle, const float *x_dev, const float *cond_dev, int64_t ld_cond, int64_t R,
                                      float *out_dev, void *stream)
{
    Handle *H = live_handle(handle, "mnle_log_prob_rows_tc_f32", true);
    if (H == nullptr) return DDM_ERR_STATE;
    DDM_REQUIRE(R >= 0 && R <= 0x7FFFFFFFll - kTcM, "mnle_log_prob_rows_tc_f32: bad R");
    if (R == 0) return DDM_OK;
    DDM_REQUIRE(x_dev && cond_dev && out_dev, "mnle_log_prob_rows_tc_f32: null pointer");
    DDM_REQUIRE(ld_cond >= kCond, "mnle_log_prob_rows_tc_f32: ld_cond=%lld < 85", (long long)ld_cond);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    DDM_CUDA_TRY(cudaFuncSetAttribute(mnle_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)TcSmem<true>::kBytes));
    int sms = 0, n_pairs = 0;
    long long grid = 0;
    DDM_CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, H->device));
    tc_grid((R + kTcM - 1) / kTcM, sms, &n_pairs, &grid);
    mnle_tc_kernel<true><<<(unsigned)grid, kTcThreads, TcSmem<true>::kBytes, st>>>(
        static_cast<const unsigned char *>(H->tc_pack), H->tc_rows_plan, cond_dev, ld_cond, x_dev, nullptr, 1, 1, (int)R,
        n_pairs, H->mu_y, H->sigma_y, H->layout.n_choices, nullptr, nullptr, out_dev, nullptr);
    DDM_CUDA_TRY(cudaGetLastError());
    return DDM_OK;
}
