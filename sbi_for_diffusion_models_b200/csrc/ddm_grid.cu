// The pulse DDM's own likelihood: its first-passage law by density propagation on a grid.
//
// The scheme is the one oracle/ddm_grid_spec.py defines in float64 (read its docstring first): M cells of width
// h = B / M over (0, B), each cell's mass at its centre, one Euler step = the truncated Gaussian of mean
// c (1 - lam dt) + kick and variance s^2 - h^2 / 12 integrated over every cell, tails beyond 0 and B absorbed.
//
// One CTA of 512 threads per row; the two density buffers live in shared memory (2 x 8192 fp32 = 64 KB).  ptxas
// (CUDA 12.9, sm_100a): 58 registers, no spills, so two CTAs per SM.
// A thread owns runs of kRun consecutive target cells and gathers over the contiguous range of sources that can
// reach them (c (1 - lam dt) is monotone in the cell index, so that range follows from the run's ends).  With the
// leak, source j's mean sits (j + 1/2) lam dt cells below its centre: the stencil is not Toeplitz, so every
// (source, edge) value of the Gaussian CDF is evaluated, with erfcf, and the kRun + 1 edges of a run share them.
// Tabulating the CDF on a fine grid and interpolating would save the erfcf but adds an interpolation error the
// float64 spec would have to reproduce, and the table would depend on h / s, which differs from row to row.
//
// Arithmetic is fp32 with fp32 accumulation: every weight and every mass is positive, so sums do not cancel.  A
// weight is the truncated-normal mass between two edges taken from the two smaller tails, never as a difference of
// numbers close to 1.  Positions are kept as an exact integer cell offset plus a small fraction, so that an edge's
// distance from a source is not rounded at the scale of the cell index.  Reductions run in a fixed order inside the
// CTA, so a row gives the same bits in any batch.
#include "ddm_common.cuh"

#include <math.h>

namespace ddm {

constexpr int kGridMaxCells = 8192;
constexpr int kGridThreads = 512;
constexpr int kRun = 4;                 // target cells per thread and pass
constexpr double kGridSigmas = 6.0;     // oracle/ddm_grid_spec.py SIGMAS
constexpr int kModeLaw = 0, kModeLoglik = 1;

struct GridArgs {
    const float *theta;
    long long ld_theta;
    const float *pulses;
    long long ld_pulses;
    const float *x;
    long long N;
    long long C;                        // > 0: row r = t * C + c (theta row c, x / pulse row t); 0: row r everywhere
    int n_max, spp;
    float dt, t_max, t_nd_hi, noise_scale;
    double cells_per_sigma;
    float tail_r, tail_norm;            // truncation: tail = max(0.5 erfc(z) - tail_r, 0) * tail_norm
    int mode;
    float *law;                         // (N, 2, n_max)
    float *survive;                     // (N,)
    int *cells;                         // NULL or (N,)
    float *out;                         // (N,) log-likelihood
};

struct RowScal {
    int M, W, target, side;             // side: 0 / 1 / 2 for loglik rows
    float g;                            // h / (sigma_eff sqrt 2): cell distance -> erfc argument
    float ldt;                          // lam dt
    float gain_cells;                   // gain / h
    double p0;                          // start after the first decay, in cells
    bool bad;
};

__device__ __forceinline__ float tail_mass(float x_cells, float g, float tail_r, float tail_norm)
{
    const float t = 0.5f * erfcf(fabsf(x_cells) * g) - tail_r;
    return fmaxf(t, 0.0f) * tail_norm;
}

// mass between edges xa < xb (in cells, relative to the source) from the two smaller tails ta, tb
__device__ __forceinline__ float cell_mass(float xa, float xb, float ta, float tb)
{
    return xb <= 0.0f ? tb - ta : (xa >= 0.0f ? ta - tb : (1.0f - ta) - tb);
}

__device__ __forceinline__ float lower_mass(float x, float t) { return x <= 0.0f ? t : 1.0f - t; }

// Fixed-order block sum of two values; every thread gets the totals.
__device__ __forceinline__ float2 block_sum2(float a, float b, float2 *red)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        a += __shfl_down_sync(0xFFFFFFFFu, a, o);
        b += __shfl_down_sync(0xFFFFFFFFu, b, o);
    }
    const int w = threadIdx.x >> 5;
    if ((threadIdx.x & 31) == 0) red[w] = make_float2(a, b);
    __syncthreads();
    float2 s = make_float2(0.0f, 0.0f);
    for (int i = 0; i < kGridThreads / 32; ++i) {
        s.x += red[i].x;
        s.y += red[i].y;
    }
    __syncthreads();
    return s;
}

__device__ RowScal row_scalars(const GridArgs &a, const float *th, const float *x)
{
    RowScal r;
    const float a0f = fminf(fmaxf(th[0], 0.0f), 1.0f);
    const float lam = th[1];
    const float gain = fabsf(th[2]);
    float B = fabsf(th[3]);
    if (B < 1e-6f) B = 1e-6f;
    const float t_nd = fminf(fmaxf(th[4], 0.0f), a.t_nd_hi);
    const float win = floorf((a.t_max - t_nd) / a.dt);   // the simulator's window, in fp32
    r.W = (win != win) ? 0 : (int)fminf(fmaxf(win, 0.0f), (float)a.n_max);
    const double s = (double)a.noise_scale;
    const double cells = ceil((double)B * a.cells_per_sigma / s);
    r.M = (int)fmin(fmax(cells, 1.0), (double)kGridMaxCells);
    const double h = (double)B / r.M;
    const double sig = sqrt(fmax(s * s - h * h / 12.0, 0.25 * s * s));
    r.g = (float)(h / (sig * 1.4142135623730951));
    r.ldt = lam * a.dt;
    const double decay = 1.0 - (double)lam * (double)a.dt;
    r.gain_cells = (float)((double)gain / h);
    r.p0 = (double)a0f * (double)B / h * decay;
    r.bad = !(decay > 0.0) || !isfinite(th[0]) || !isfinite(lam) || !isfinite(gain) || !isfinite(th[3]) ||
            !isfinite(th[4]);
    r.target = r.W;
    r.side = 2;
    if (a.mode == kModeLoglik) {
        const float c = x[1];
        r.side = c == 0.0f ? 0 : (c == 1.0f ? 1 : 2);
        if (r.side < 2) r.target = (int)rintf((x[0] - t_nd) / a.dt);   // k = round((rt - t_nd) / dt)
    }
    return r;
}

__global__ void __launch_bounds__(kGridThreads) grid_kernel(GridArgs a)
{
    extern __shared__ float smem[];
    __shared__ float2 red[kGridThreads / 32];
    float *cur = smem, *nxt = smem + kGridMaxCells;

    const long long row = blockIdx.x;
    const long long ti = a.C > 0 ? row % a.C : row;
    const long long xi = a.C > 0 ? row / a.C : row;
    const float *th = a.theta + ti * a.ld_theta;
    const float *pl = a.pulses + xi * a.ld_pulses;
    const RowScal r = row_scalars(a, th, a.x + 2 * xi);
    const int M = r.M;
    const float g = r.g, tr = a.tail_r, tn = a.tail_norm;
    const int tid = threadIdx.x;
    const float dt_log = logf(a.dt);

    if (a.mode == kModeLaw) {
        float *law = a.law + row * 2ll * a.n_max;
        for (int k = tid; k < 2 * a.n_max; k += kGridThreads) law[k] = 0.0f;
        if (a.cells && tid == 0) a.cells[row] = M;
        __syncthreads();
        if (r.bad) {
            for (int k = tid; k < 2 * a.n_max; k += kGridThreads) law[k] = NAN;
            if (tid == 0) a.survive[row] = NAN;
            return;
        }
    } else {
        float res = 0.0f;
        bool done = false;
        if (r.bad) res = NAN, done = true;
        else if (r.side < 2 && (r.target < 1 || r.target > r.W)) res = -INFINITY, done = true;
        else if (r.side == 2 && r.W == 0) res = 0.0f, done = true;
        if (done) {
            if (tid == 0) a.out[row] = res;
            return;
        }
    }
    const int n_steps = r.target;           // W for the law and for choice 2, the observed step otherwise
    const bool law_mode = a.mode == kModeLaw;
    if (n_steps == 0) {                      // law with W = 0: everything survives
        if (tid == 0) a.survive[row] = 1.0f;
        return;
    }

    for (int k = 0; k < n_steps; ++k) {
        float kick = 0.0f;
        if (k % a.spp == 0) kick = r.gain_cells * pl[k / a.spp];
        // beyond the domain plus the Gaussian's reach the kick's size no longer matters
        const float kick_lim = 2.0f * (float)M + 8.0f * (float)kGridSigmas / g + 8.0f;
        kick = fminf(fmaxf(kick, -kick_lim), kick_lim);
        const bool last = k == n_steps - 1;
        const bool want_abs = law_mode || last;
        const bool want_next = law_mode || !last || r.side == 2;

        if (k == 0) {
            // the exact start point: position p = pi + pf in cells, pi integer
            const double p = r.p0 + (double)kick;
            const double pi = floor(p);
            const float pf = (float)(p - pi);
            const long long pii = (long long)pi;
            if (want_abs && tid == 0) {
                const float xb = (float)(0ll - pii) - pf, xt = (float)(pii - M) + pf;
                const float bot = lower_mass(xb, tail_mass(xb, g, tr, tn));
                const float top = lower_mass(xt, tail_mass(xt, g, tr, tn));
                if (law_mode) {
                    a.law[row * 2ll * a.n_max + 0] = bot;
                    a.law[row * 2ll * a.n_max + a.n_max] = top;
                } else if (last && r.side < 2) {
                    const float pr = r.side == 0 ? bot : top;
                    a.out[row] = logf(pr) - dt_log;
                }
            }
            if (want_next)
                for (int i = tid; i < M; i += kGridThreads) {
                    const float xa = (float)(i - pii) - pf, xb = xa + 1.0f;
                    cur[i] = cell_mass(xa, xb, tail_mass(xa, g, tr, tn), tail_mass(xb, g, tr, tn));
                }
            __syncthreads();
            continue;
        }

        // sources: p_j = (j + 1/2)(1 - lam dt) + kick = j + ki - off_j with ki = rint(kick) and
        // off_j = (j + 1/2) lam dt - 1/2 - (kick - ki); an edge e is at e - p_j = (e - j - ki) + off_j
        const float ki_f = rintf(kick);
        const int ki = (int)ki_f;
        const float kf = kick - ki_f;
        if (want_abs) {
            float bot = 0.0f, top = 0.0f;
            for (int j = tid; j < M; j += kGridThreads) {
                const float m = cur[j];
                const float off = fmaf((float)j + 0.5f, r.ldt, -0.5f - kf);
                const float xb = (float)(-j - ki) + off;              // edge 0
                const float xt = (float)(j + ki - M) - off;           // p_j - B: mass above B
                bot = fmaf(m, lower_mass(xb, tail_mass(xb, g, tr, tn)), bot);
                top = fmaf(m, lower_mass(xt, tail_mass(xt, g, tr, tn)), top);
            }
            const float2 s = block_sum2(bot, top, red);
            if (tid == 0) {
                if (law_mode) {
                    a.law[row * 2ll * a.n_max + k] = s.x;
                    a.law[row * 2ll * a.n_max + a.n_max + k] = s.y;
                } else if (last && r.side < 2) {
                    a.out[row] = logf(r.side == 0 ? s.x : s.y) - dt_log;
                }
            }
        }
        if (!want_next) break;

        const float reach = (float)kGridSigmas / (g * 1.4142135623730951f) + 2.0f;   // cells
        const float inv_decay = 1.0f / (1.0f - r.ldt);
        for (int i0 = tid * kRun; i0 < M; i0 += kGridThreads * kRun) {
            float acc[kRun];
#pragma unroll
            for (int q = 0; q < kRun; ++q) acc[q] = 0.0f;
            const float lo = ((float)i0 - reach - kick) * inv_decay - 1.5f;
            const float hi = ((float)(i0 + kRun) + reach - kick) * inv_decay + 1.5f;
            const int jlo = (int)fmaxf(floorf(lo), 0.0f);
            const int jhi = (int)fminf(ceilf(hi), (float)(M - 1));
            for (int j = jlo; j <= jhi; ++j) {
                const float m = cur[j];
                const float off = fmaf((float)j + 0.5f, r.ldt, -0.5f - kf);
                float xe[kRun + 1], te[kRun + 1];
#pragma unroll
                for (int q = 0; q <= kRun; ++q) {
                    xe[q] = (float)(i0 + q - j - ki) + off;
                    te[q] = tail_mass(xe[q], g, tr, tn);
                }
#pragma unroll
                for (int q = 0; q < kRun; ++q) acc[q] = fmaf(m, cell_mass(xe[q], xe[q + 1], te[q], te[q + 1]), acc[q]);
            }
#pragma unroll
            for (int q = 0; q < kRun; ++q)
                if (i0 + q < M) nxt[i0 + q] = acc[q];
        }
        __syncthreads();
        float *t = cur;
        cur = nxt;
        nxt = t;
    }

    if (law_mode || r.side == 2) {
        float part = 0.0f;
        for (int j = tid; j < M; j += kGridThreads) part += cur[j];
        const float2 s = block_sum2(part, 0.0f, red);
        if (tid == 0) {
            if (law_mode) a.survive[row] = s.x;
            else a.out[row] = logf(s.x);
        }
    }
}

__global__ void grid_chain_sum_kernel(const float *ws, long long T, long long C, float *out)
{
    const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    double s = 0.0;
    for (long long t = 0; t < T; ++t) s += (double)ws[t * C + c];
    out[c] = (float)s;
}

static int grid_launch(GridArgs a, int64_t P, const char *what, void *stream)
{
    DDM_REQUIRE(a.N >= 0, "%s: N must be >= 0", what);
    DDM_REQUIRE(a.n_max >= 0 && a.n_max <= (1 << 24), "%s: n_max out of range", what);
    DDM_REQUIRE(a.spp >= 1, "%s: steps_per_pulse must be >= 1", what);
    DDM_REQUIRE(a.dt > 0.0f && isfinite(a.dt) && a.noise_scale > 0.0f && isfinite(a.noise_scale) && isfinite(a.t_max),
                "%s: bad schedule scalars", what);
    DDM_REQUIRE(a.cells_per_sigma > 0.0 && a.cells_per_sigma <= 64.0, "%s: cells_per_sigma must be in (0, 64]", what);
    if (a.N == 0) return DDM_OK;
    DDM_REQUIRE(a.theta && a.pulses, "%s: null input", what);
    DDM_REQUIRE(a.ld_theta >= 5, "%s: ld_theta must be >= 5", what);
    const int64_t need = (a.n_max + a.spp - 1) / a.spp;
    DDM_REQUIRE(P >= need, "%s: pulses have %lld columns, the schedule needs %lld", what, (long long)P,
                (long long)need);
    DDM_REQUIRE(a.ld_pulses >= P, "%s: ld_pulses must be >= P", what);
    DDM_REQUIRE(a.N <= 0x7FFFFFFFll, "%s: at most 2^31 - 1 rows per call", what);
    const double tr = 0.5 * erfc(kGridSigmas / 1.4142135623730951);
    a.tail_r = (float)tr;
    a.tail_norm = (float)(1.0 / (1.0 - 2.0 * tr));
    const size_t smem = 2u * kGridMaxCells * sizeof(float);
    DDM_CUDA_TRY(cudaFuncSetAttribute(grid_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    grid_kernel<<<(unsigned)a.N, kGridThreads, smem, static_cast<cudaStream_t>(stream)>>>(a);
    DDM_CUDA_TRY(cudaGetLastError());
    return DDM_OK;
}

static GridArgs grid_args(const float *theta, int64_t ld_theta, const float *pulses, int64_t ld_pulses, int64_t N,
                          int64_t n_max, int64_t spp, float dt, float t_max, float t_nd_hi, float noise_scale,
                          float cells_per_sigma)
{
    GridArgs a = {};
    a.theta = theta;
    a.ld_theta = ld_theta;
    a.pulses = pulses;
    a.ld_pulses = ld_pulses;
    a.N = N;
    a.n_max = (int)(n_max > (1 << 24) || n_max < 0 ? -1 : n_max);
    a.spp = (int)(spp > (1 << 24) ? 0 : spp);
    a.dt = dt;
    a.t_max = t_max;
    a.t_nd_hi = t_nd_hi;
    a.noise_scale = noise_scale;
    a.cells_per_sigma = (double)cells_per_sigma;
    return a;
}

}  // namespace ddm

using namespace ddm;

DDM_API int ddm_grid_max_cells(void) { return kGridMaxCells; }

DDM_API int ddm_grid_law_f32(const float *theta_dev, int64_t ld_theta, const float *pulses_dev, int64_t ld_pulses,
                             int64_t N, int64_t P, int64_t n_max, int64_t steps_per_pulse, float dt, float t_max,
                             float t_nd_hi, float noise_scale, float cells_per_sigma, float *law_out_dev,
                             float *survive_out_dev, int32_t *cells_out_dev, void *stream)
{
    GridArgs a = grid_args(theta_dev, ld_theta, pulses_dev, ld_pulses, N, n_max, steps_per_pulse, dt, t_max, t_nd_hi,
                           noise_scale, cells_per_sigma);
    a.mode = kModeLaw;
    a.law = law_out_dev;
    a.survive = survive_out_dev;
    a.cells = cells_out_dev;
    DDM_REQUIRE(N == 0 || (law_out_dev && survive_out_dev), "ddm_grid_law_f32: null output");
    return grid_launch(a, P, "ddm_grid_law_f32", stream);
}

DDM_API int ddm_grid_loglik_f32(const float *theta_dev, int64_t ld_theta, const float *x_dev, const float *pulses_dev,
                                int64_t ld_pulses, int64_t N, int64_t P, int64_t n_max, int64_t steps_per_pulse,
                                float dt, float t_max, float t_nd_hi, float noise_scale, float cells_per_sigma,
                                float *out_dev, void *stream)
{
    GridArgs a = grid_args(theta_dev, ld_theta, pulses_dev, ld_pulses, N, n_max, steps_per_pulse, dt, t_max, t_nd_hi,
                           noise_scale, cells_per_sigma);
    a.mode = kModeLoglik;
    a.x = x_dev;
    a.out = out_dev;
    DDM_REQUIRE(N == 0 || (x_dev && out_dev), "ddm_grid_loglik_f32: null x / output");
    return grid_launch(a, P, "ddm_grid_loglik_f32", stream);
}

DDM_API size_t ddm_grid_loglik_sum_workspace_floats(int64_t T, int64_t C)
{
    return (T > 0 && C > 0) ? (size_t)T * (size_t)C : 0;
}

DDM_API int ddm_grid_loglik_sum_f32(const float *theta_dev, int64_t ld_theta, const float *x_dev,
                                    const float *pulses_dev, int64_t ld_pulses, int64_t T, int64_t C, int64_t P,
                                    int64_t n_max, int64_t steps_per_pulse, float dt, float t_max, float t_nd_hi,
                                    float noise_scale, float cells_per_sigma, float *out_dev, float *workspace_dev,
                                    void *stream)
{
    DDM_REQUIRE(T >= 0 && C >= 0, "ddm_grid_loglik_sum_f32: T and C must be >= 0");
    DDM_REQUIRE(T * C <= 0x7FFFFFFFll, "ddm_grid_loglik_sum_f32: T * C must be < 2^31");
    if (C == 0) return DDM_OK;
    DDM_REQUIRE(out_dev != nullptr, "ddm_grid_loglik_sum_f32: null output");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (T == 0) {
        DDM_CUDA_TRY(cudaMemsetAsync(out_dev, 0, (size_t)C * sizeof(float), st));
        return DDM_OK;
    }
    DDM_REQUIRE(workspace_dev != nullptr && x_dev != nullptr, "ddm_grid_loglik_sum_f32: null workspace / x");
    GridArgs a = grid_args(theta_dev, ld_theta, pulses_dev, ld_pulses, T * C, n_max, steps_per_pulse, dt, t_max,
                           t_nd_hi, noise_scale, cells_per_sigma);
    a.mode = kModeLoglik;
    a.C = C;
    a.x = x_dev;
    a.out = workspace_dev;
    const int rc = grid_launch(a, P, "ddm_grid_loglik_sum_f32", stream);
    if (rc != DDM_OK) return rc;
    grid_chain_sum_kernel<<<(unsigned)((C + 255) / 256), 256, 0, st>>>(workspace_dev, T, C, out_dev);
    DDM_CUDA_TRY(cudaGetLastError());
    return DDM_OK;
}
