// The pulse DDM's own likelihood: its first-passage law by density propagation on a grid.
//
// The scheme is the one oracle/ddm_grid_spec.py defines in float64 (read its docstring first): M cells of width
// h = B / M over (0, B), each cell's mass at its centre, one Euler step = the truncated Gaussian of mean
// c (1 - lam dt) + kick and variance s^2 - h^2 / 12 integrated over every cell, tails beyond 0 and B absorbed.
//
// One CTA of 512 threads per row; the two density buffers live in shared memory (2 x 8192 fp32 = 64 KB).  ptxas
// (CUDA 12.9, sm_100a): 57 registers, no spills, so two CTAs per SM.
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

#include <algorithm>

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

// The helpers below round every product on its own (no fma contraction), so that the row kernel and the batched
// potential, which inline them at different call sites, compute the same fp32 numbers.
__device__ __forceinline__ float tail_mass(float x_cells, float g, float tail_r, float tail_norm)
{
    const float t = __fsub_rn(__fmul_rn(0.5f, erfcf(__fmul_rn(fabsf(x_cells), g))), tail_r);
    return __fmul_rn(fmaxf(t, 0.0f), tail_norm);
}

// mass between edges xa < xb (in cells, relative to the source) from the two smaller tails ta, tb
__device__ __forceinline__ float cell_mass(float xa, float xb, float ta, float tb)
{
    return xb <= 0.0f ? tb - ta : (xa >= 0.0f ? ta - tb : (1.0f - ta) - tb);
}

__device__ __forceinline__ float lower_mass(float x, float t) { return x <= 0.0f ? t : 1.0f - t; }

// The sources that can reach target cells i0 .. i0 + kRun - 1: c (1 - lam dt) + kick is monotone in the cell index.
__device__ __forceinline__ int2 source_range(int i0, float reach, float kick, float inv_decay, int M)
{
    const float lo = __fsub_rn(__fmul_rn(__fsub_rn(__fsub_rn((float)i0, reach), kick), inv_decay), 1.5f);
    const float hi = __fadd_rn(__fmul_rn(__fsub_rn(__fadd_rn((float)(i0 + kRun), reach), kick), inv_decay), 1.5f);
    return make_int2((int)fmaxf(floorf(lo), 0.0f), (int)fminf(ceilf(hi), (float)(M - 1)));
}

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

// ---- the pieces of one step that the row kernel and the batched potential share ----
// Cell i of a density buffer lives at buf[ix(i)]: the row kernel stores cells densely, the potential with one pad
// word after every 32 cells, so that the 32 threads of a warp, whose source cells are about kRun apart, read 32
// different banks.
struct DenseCells {
    __device__ __forceinline__ int operator()(int i) const { return i; }
};
struct PaddedCells {
    __device__ __forceinline__ int operator()(int i) const { return i + (i >> 5); }
};

// beyond the domain plus the Gaussian's reach the kick's size no longer matters
__device__ __forceinline__ float clamp_kick(float kick, int M, float g)
{
    const float kick_lim = 2.0f * (float)M + 8.0f * (float)kGridSigmas / g + 8.0f;
    return fminf(fmaxf(kick, -kick_lim), kick_lim);
}

// step 0 from the exact start point: position p = pi + pf in cells, pi integer
struct StartPoint {
    long long pii;
    float pf;
};

__device__ __forceinline__ StartPoint start_point(double p0, float kick)
{
    const double p = p0 + (double)kick;
    const double pi = floor(p);
    return StartPoint{(long long)pi, (float)(p - pi)};
}

// step 0's absorptions (bottom, top)
__device__ __forceinline__ float2 start_absorb(StartPoint sp, int M, float g, float tr, float tn)
{
    const float xb = (float)(0ll - sp.pii) - sp.pf, xt = (float)(sp.pii - M) + sp.pf;
    return make_float2(lower_mass(xb, tail_mass(xb, g, tr, tn)), lower_mass(xt, tail_mass(xt, g, tr, tn)));
}

template <class Ix>
__device__ __forceinline__ void start_fill(float *cur, StartPoint sp, int M, float g, float tr, float tn, Ix ix)
{
    for (int i = threadIdx.x; i < M; i += kGridThreads) {
        const float xa = (float)(i - sp.pii) - sp.pf, xb = xa + 1.0f;
        cur[ix(i)] = cell_mass(xa, xb, tail_mass(xa, g, tr, tn), tail_mass(xb, g, tr, tn));
    }
}

// Sources: p_j = (j + 1/2)(1 - lam dt) + kick = j + ki - off_j with ki = rint(kick) and
// off_j = (j + 1/2) lam dt - 1/2 - (kick - ki); an edge e is at e - p_j = (e - j - ki) + off_j.
struct Kick {
    float kick, kf;
    int ki;
};

__device__ __forceinline__ Kick split_kick(float kick)
{
    const float ki_f = rintf(kick);
    return Kick{kick, kick - ki_f, (int)ki_f};
}

// a step's absorptions (bottom, top) from density cur, summed in the fixed order of block_sum2
template <class Ix>
__device__ __forceinline__ float2 absorb_sums(const float *cur, int M, float ldt, Kick kk, float g, float tr, float tn,
                                              float2 *red, Ix ix)
{
    float bot = 0.0f, top = 0.0f;
    for (int j = threadIdx.x; j < M; j += kGridThreads) {
        const float m = cur[ix(j)];
        const float off = fmaf((float)j + 0.5f, ldt, -0.5f - kk.kf);
        const float xb = (float)(-j - kk.ki) + off;              // edge 0
        const float xt = (float)(j + kk.ki - M) - off;           // p_j - B: mass above B
        bot = fmaf(m, lower_mass(xb, tail_mass(xb, g, tr, tn)), bot);
        top = fmaf(m, lower_mass(xt, tail_mass(xt, g, tr, tn)), top);
    }
    return block_sum2(bot, top, red);
}

// a step's propagation cur -> nxt with every weight evaluated on the fly (no __syncthreads)
template <class Ix>
__device__ __forceinline__ void propagate_direct(const float *cur, float *nxt, int M, float ldt, Kick kk, float reach,
                                                 float inv_decay, float g, float tr, float tn, Ix ix)
{
    for (int i0 = threadIdx.x * kRun; i0 < M; i0 += kGridThreads * kRun) {
        float acc[kRun];
#pragma unroll
        for (int q = 0; q < kRun; ++q) acc[q] = 0.0f;
        const int2 range = source_range(i0, reach, kk.kick, inv_decay, M);
        for (int j = range.x; j <= range.y; ++j) {
            const float m = cur[ix(j)];
            const float off = fmaf((float)j + 0.5f, ldt, -0.5f - kk.kf);
            float xe[kRun + 1], te[kRun + 1];
#pragma unroll
            for (int q = 0; q <= kRun; ++q) {
                xe[q] = (float)(i0 + q - j - kk.ki) + off;
                te[q] = tail_mass(xe[q], g, tr, tn);
            }
#pragma unroll
            for (int q = 0; q < kRun; ++q) acc[q] = fmaf(m, cell_mass(xe[q], xe[q + 1], te[q], te[q + 1]), acc[q]);
        }
#pragma unroll
        for (int q = 0; q < kRun; ++q)
            if (i0 + q < M) nxt[ix(i0 + q)] = acc[q];
    }
}

__device__ __forceinline__ float grid_reach(float g) { return (float)kGridSigmas / (g * 1.4142135623730951f) + 2.0f; }

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

    const DenseCells ix;
    for (int k = 0; k < n_steps; ++k) {
        float kick = 0.0f;
        if (k % a.spp == 0) kick = r.gain_cells * pl[k / a.spp];
        kick = clamp_kick(kick, M, g);
        const bool last = k == n_steps - 1;
        const bool want_abs = law_mode || last;
        const bool want_next = law_mode || !last || r.side == 2;

        if (k == 0) {
            const StartPoint sp = start_point(r.p0, kick);
            if (want_abs && tid == 0) {
                const float2 s = start_absorb(sp, M, g, tr, tn);
                if (law_mode) {
                    a.law[row * 2ll * a.n_max + 0] = s.x;
                    a.law[row * 2ll * a.n_max + a.n_max] = s.y;
                } else if (last && r.side < 2) {
                    const float pr = r.side == 0 ? s.x : s.y;
                    a.out[row] = logf(pr) - dt_log;
                }
            }
            if (want_next) start_fill(cur, sp, M, g, tr, tn, ix);
            __syncthreads();
            continue;
        }

        const Kick kk = split_kick(kick);
        if (want_abs) {
            const float2 s = absorb_sums(cur, M, r.ldt, kk, g, tr, tn, red, ix);
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

        propagate_direct(cur, nxt, M, r.ldt, kk, grid_reach(g), 1.0f / (1.0f - r.ldt), g, tr, tn, ix);
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

// out[i] = sum over t = 0..T-1 in that order, in fp64, of ws[t * ld_t + i * ld_i], for i < N
__global__ void grid_chain_sum_kernel(const float *ws, long long T, long long N, long long ld_t, long long ld_i,
                                      float *out)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    double s = 0.0;
    for (long long t = 0; t < T; ++t) s += (double)ws[t * ld_t + i * ld_i];
    out[i] = (float)s;
}

// ---- the batched potential: each theta's kick-free weights tabulated once, applied to a group of its trials ----
//
// On a step without a kick (199 of every 200 at the simulator's schedule) source j's offset is
// off_j = (j + 1/2) lam dt - 1/2: it does not depend on the step, so the step's weights are the same fp32 numbers on
// every such step, and on every trial of the same theta.  The table pass writes them once per theta (band_max x
// runs float4: entry [it][run] holds the weights of source jlo(run) + it to the kRun targets of the run), with the
// helpers and arguments of the row kernel.  The propagation pass runs one CTA per (theta, group of up to
// kPotMaxG of its trials) with the group's densities in shared memory; a tap is one table load shared by the
// group and one fmaf per trial.  Step 0 and kick steps use the row kernel's direct code per trial, absorptions and
// survival sums its block_sum2 order, and every target accumulates its sources in ascending j with fmaf as the
// row kernel does: every (trial, theta) value has the bits of ddm_grid_loglik_f32.
constexpr int kPotMaxG = 8;                          // trials per CTA
constexpr int kPotSlices = 32;                       // CTAs per theta in the table pass
constexpr int kPotTableThreads = 256;
constexpr int kPotRuns = kGridMaxCells / kRun;       // runs of the largest grid
constexpr size_t kPotSmemBytes = 227 * 1024 - 1024;  // dynamic shared memory of a propagation CTA
constexpr size_t kPotTableBudget = (size_t)7 << 28;  // bytes of tables per chunk of theta (1.75 GiB)

__host__ __device__ inline int pot_stride(int M) { return M + ((M + 31) >> 5); }   // floats per padded density
__host__ __device__ inline int pot_group(int M)
{
    const int g = (int)(kPotSmemBytes / (2 * sizeof(float) * (size_t)pot_stride(M)));
    return g < kPotMaxG ? g : kPotMaxG;
}

// An upper bound of jhi - jlo + 1 for any admitted theta: sigma_eff <= s and h > s / (2q) (M >= 2), so the reach is
// below 12 q + 2 cells, and 1 / (1 - lam dt) <= 2 for lam dt < 0.5.  The table pass flags a theta that exceeds it.
static int pot_band_max(double q) { return (int)fmin((double)kGridMaxCells, ceil(48.0 * q) + 24.0); }

struct PotArgs {
    GridArgs a;                 // schedule, theta (D*C rows), x and pulses (D*T rows)
    long long T, C;             // trials and chains per dataset
    long long n0;               // first theta row (d * C + c) of this chunk
    int groups;                 // propagation CTAs per theta
    int band_max;
    const int *order;           // (D, T): each dataset's trials by rt, choice 2 last
    float4 *table;              // per theta of the chunk: band_max * kPotRuns float4
    int *flag;                  // per theta of the chunk: 1 if a band exceeded band_max
    float *rows;                // (chunk, T): row log-likelihoods in the original trial order
};

// theta's scalars without a trial; bad also for lam dt >= 0.5, which the host refuses in loglik_rows
__device__ __forceinline__ RowScal pot_scalars(const GridArgs &a, const float *th)
{
    GridArgs b = a;
    b.mode = kModeLaw;
    RowScal r = row_scalars(b, th, nullptr);
    r.bad = r.bad || !((double)th[1] * (double)a.dt < 0.5);
    return r;
}

// rank of each trial of its dataset under (choice 2 last, rt, index): order[d * T + rank] = t
__global__ void grid_trial_order_kernel(const float *x, long long D, long long T, int *order)
{
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= D * T) return;
    const long long d = e / T, t = e % T;
    const float *xd = x + 2 * d * T;
    auto key = [](const float *xr) {
        const uint32_t b = __float_as_uint(xr[0]);
        const uint32_t mono = (b & 0x80000000u) ? ~b : (b | 0x80000000u);   // float order as unsigned order
        const bool censored = !(xr[1] == 0.0f || xr[1] == 1.0f);
        return ((unsigned long long)censored << 32) | mono;
    };
    const unsigned long long kt = key(xd + 2 * t);
    long long rank = 0;
    for (long long u = 0; u < T; ++u) {
        const unsigned long long ku = key(xd + 2 * u);
        rank += (ku < kt) || (ku == kt && u < t);
    }
    order[d * T + rank] = (int)t;
}

__global__ void __launch_bounds__(kPotTableThreads) grid_table_kernel(PotArgs p)
{
    const long long nl = blockIdx.x / kPotSlices;
    const int slice = blockIdx.x % kPotSlices;
    const RowScal r = pot_scalars(p.a, p.a.theta + (p.n0 + nl) * p.a.ld_theta);
    if (r.bad) return;
    const int M = r.M, R = (M + kRun - 1) / kRun;
    const float g = r.g, tr = p.a.tail_r, tn = p.a.tail_norm;
    const float reach = grid_reach(g), inv_decay = 1.0f / (1.0f - r.ldt);
    float4 *tab = p.table + nl * (long long)p.band_max * kPotRuns;
    const long long total = (long long)R * p.band_max;
    for (long long e = (long long)slice * kPotTableThreads + threadIdx.x; e < total;
         e += (long long)kPotSlices * kPotTableThreads) {
        const int run = (int)(e % R), it = (int)(e / R);
        const int i0 = run * kRun;
        const int2 range = source_range(i0, reach, 0.0f, inv_decay, M);
        if (it == 0 && range.y - range.x + 1 > p.band_max) p.flag[nl] = 1;
        if (it > range.y - range.x) continue;
        const int j = range.x + it;
        const float off = fmaf((float)j + 0.5f, r.ldt, -0.5f);    // the row kernel's offset with kick 0
        float xe[kRun + 1], te[kRun + 1];
#pragma unroll
        for (int q = 0; q <= kRun; ++q) {
            xe[q] = (float)(i0 + q - j) + off;
            te[q] = tail_mass(xe[q], g, tr, tn);
        }
        tab[(long long)it * R + run] = make_float4(cell_mass(xe[0], xe[1], te[0], te[1]), cell_mass(xe[1], xe[2], te[1], te[2]),
                                                   cell_mass(xe[2], xe[3], te[2], te[3]), cell_mass(xe[3], xe[4], te[3], te[4]));
    }
}

// one kick-free step of NG densities (stride S floats apart) from the table
template <int NG>
__device__ __forceinline__ void propagate_table(const float *cur, float *nxt, int S, const float4 *__restrict__ tab,
                                                int M, float reach, float inv_decay)
{
    const PaddedCells ix;
    const int R = (M + kRun - 1) / kRun;
    for (int run = threadIdx.x; run < R; run += kGridThreads) {
        const int i0 = run * kRun;
        const int2 range = source_range(i0, reach, 0.0f, inv_decay, M);
        float acc[NG][kRun];
#pragma unroll
        for (int t = 0; t < NG; ++t)
#pragma unroll
            for (int q = 0; q < kRun; ++q) acc[t][q] = 0.0f;
        const float4 *w = tab + run;
        for (int j = range.x; j <= range.y; ++j, w += R) {
            const float4 c = __ldg(w);
            const int jj = ix(j);
#pragma unroll
            for (int t = 0; t < NG; ++t) {
                const float m = cur[t * S + jj];
                acc[t][0] = fmaf(m, c.x, acc[t][0]);
                acc[t][1] = fmaf(m, c.y, acc[t][1]);
                acc[t][2] = fmaf(m, c.z, acc[t][2]);
                acc[t][3] = fmaf(m, c.w, acc[t][3]);
            }
        }
#pragma unroll
        for (int t = 0; t < NG; ++t)
#pragma unroll
            for (int q = 0; q < kRun; ++q)
                if (i0 + q < M) nxt[t * S + ix(i0 + q)] = acc[t][q];
    }
}

__global__ void __launch_bounds__(kGridThreads, 1) grid_potential_kernel(PotArgs p)
{
    extern __shared__ float smem[];
    __shared__ float2 red[kGridThreads / 32];
    // the group's live trials, by number of propagated steps ascending: trial, side, observed step, steps propagated
    __shared__ int s_t[kPotMaxG], s_side[kPotMaxG], s_n[kPotMaxG], s_prop[kPotMaxG];
    __shared__ int s_live;

    const GridArgs &a = p.a;
    const long long nl = blockIdx.x / p.groups;
    const int grp = blockIdx.x % p.groups;
    const long long n = p.n0 + nl, d = n / p.C;
    const float *th = a.theta + n * a.ld_theta;
    const RowScal r = pot_scalars(a, th);
    const int M = r.M, G = pot_group(M), S = pot_stride(M);
    if ((long long)grp * G >= p.T) return;
    const int ng = (int)min((long long)G, p.T - (long long)grp * G);
    const bool bad = r.bad || p.flag[nl] != 0;
    float *rows = p.rows + nl * p.T;
    const float g = r.g, tr = a.tail_r, tn = a.tail_norm;
    const int tid = threadIdx.x;
    const float dt_log = logf(a.dt);

    if (tid == 0) {
        int live = 0;
        for (int i = 0; i < ng; ++i) {
            const int t = p.order[d * p.T + (long long)grp * G + i];
            const RowScal rt = row_scalars(a, th, a.x + 2 * (d * p.T + t));
            float res = 0.0f;
            bool done = true;
            if (bad) res = NAN;
            else if (rt.side < 2 && (rt.target < 1 || rt.target > rt.W)) res = -INFINITY;
            else if (rt.side == 2 && rt.W == 0) res = 0.0f;
            else done = false;
            if (done) {
                rows[t] = res;
                continue;
            }
            // choice 0 / 1 propagate up to the step before the observed one and absorb there; choice 2 all W steps
            const int prop = rt.side == 2 ? rt.target : rt.target - 1;
            int k = live++;
            for (; k > 0 && s_prop[k - 1] > prop; --k) {
                s_t[k] = s_t[k - 1], s_side[k] = s_side[k - 1], s_n[k] = s_n[k - 1], s_prop[k] = s_prop[k - 1];
            }
            s_t[k] = t, s_side[k] = rt.side, s_n[k] = rt.target, s_prop[k] = prop;
        }
        s_live = live;
    }
    __syncthreads();
    const int live = s_live;
    if (live == 0) return;
    int n_steps = 0;
    for (int i = 0; i < live; ++i) n_steps = max(n_steps, s_n[i]);

    const PaddedCells ix;
    const float4 *tab = p.table + nl * (long long)p.band_max * kPotRuns;
    const float reach = grid_reach(g), inv_decay = 1.0f / (1.0f - r.ldt);
    float *cur = smem, *nxt = smem + (size_t)G * S;
    int first = 0;                                   // live trials first.. propagate at this step
    for (int k = 0; k < n_steps; ++k) {
        while (first < live && s_prop[first] <= k) ++first;
        if (k == 0 || k % a.spp == 0) {              // step 0 and kick steps: the row kernel's direct code
            for (int i = 0; i < live; ++i) {
                const float *pl = a.pulses + (d * p.T + s_t[i]) * a.ld_pulses;
                const float kick = clamp_kick(r.gain_cells * pl[k / a.spp], M, g);
                const bool absorb = s_side[i] < 2 && s_n[i] - 1 == k;
                if (k == 0) {
                    const StartPoint sp = start_point(r.p0, kick);
                    if (absorb && tid == 0) {
                        const float2 s = start_absorb(sp, M, g, tr, tn);
                        rows[s_t[i]] = logf(s_side[i] == 0 ? s.x : s.y) - dt_log;
                    }
                    if (s_prop[i] > 0) start_fill(cur + (size_t)i * S, sp, M, g, tr, tn, ix);
                    continue;
                }
                const Kick kk = split_kick(kick);
                if (absorb) {
                    const float2 s = absorb_sums(cur + (size_t)i * S, M, r.ldt, kk, g, tr, tn, red, ix);
                    if (tid == 0) rows[s_t[i]] = logf(s_side[i] == 0 ? s.x : s.y) - dt_log;
                }
                if (s_prop[i] > k)
                    propagate_direct(cur + (size_t)i * S, nxt + (size_t)i * S, M, r.ldt, kk, reach, inv_decay, g, tr,
                                     tn, ix);
            }
        } else {
            const Kick none = split_kick(0.0f);
            for (int i = 0; i < live; ++i)
                if (s_side[i] < 2 && s_n[i] - 1 == k) {
                    const float2 s = absorb_sums(cur + (size_t)i * S, M, r.ldt, none, g, tr, tn, red, ix);
                    if (tid == 0) rows[s_t[i]] = logf(s_side[i] == 0 ? s.x : s.y) - dt_log;
                }
            const float *c0 = cur + (size_t)first * S;
            float *n0 = nxt + (size_t)first * S;
            switch (live - first) {
            case 1: propagate_table<1>(c0, n0, S, tab, M, reach, inv_decay); break;
            case 2: propagate_table<2>(c0, n0, S, tab, M, reach, inv_decay); break;
            case 3: propagate_table<3>(c0, n0, S, tab, M, reach, inv_decay); break;
            case 4: propagate_table<4>(c0, n0, S, tab, M, reach, inv_decay); break;
            case 5: propagate_table<5>(c0, n0, S, tab, M, reach, inv_decay); break;
            case 6: propagate_table<6>(c0, n0, S, tab, M, reach, inv_decay); break;
            case 7: propagate_table<7>(c0, n0, S, tab, M, reach, inv_decay); break;
            case 8: propagate_table<8>(c0, n0, S, tab, M, reach, inv_decay); break;
            default: break;
            }
        }
        __syncthreads();
        if (k > 0) {
            float *t = cur;
            cur = nxt;
            nxt = t;
        }
        for (int i = 0; i < live; ++i)               // choice 2: the mass still inside after its W steps
            if (s_side[i] == 2 && s_prop[i] == k + 1) {
                float part = 0.0f;
                for (int j = tid; j < M; j += kGridThreads) part += cur[(size_t)i * S + ix(j)];
                const float2 s = block_sum2(part, 0.0f, red);
                if (tid == 0) rows[s_t[i]] = logf(s.x);
            }
    }
}

// The batched potential's workspace, in floats: the trial order (D * T ints, not chunked), then per chunk of theta
// the flags, the rows (chunk * T) and the tables (at most kPotTableBudget bytes).  Every part starts on a 256-byte
// boundary.
struct PotLayout {
    size_t order, flag, rows, table, total;
    long long chunk;
    int band_max;
};

static PotLayout pot_layout(long long D, long long T, long long C, double q)
{
    auto up = [](size_t f) { return (f + 63) & ~(size_t)63; };
    PotLayout l = {};
    l.band_max = pot_band_max(q);
    const size_t per_theta = (size_t)l.band_max * kPotRuns * kRun;
    const long long fit = (long long)(kPotTableBudget / (per_theta * sizeof(float)));
    l.chunk = std::max(1ll, std::min(D * C, fit));
    l.order = 0;
    l.flag = up((size_t)(D * T));
    l.rows = l.flag + up((size_t)l.chunk);
    l.table = l.rows + up((size_t)(l.chunk * T));
    l.total = l.table + (size_t)l.chunk * per_theta;
    return l;
}

static int grid_check_schedule(const GridArgs &a, const char *what)
{
    DDM_REQUIRE(a.n_max >= 0 && a.n_max <= (1 << 24), "%s: n_max out of range", what);
    DDM_REQUIRE(a.spp >= 1, "%s: steps_per_pulse must be >= 1", what);
    DDM_REQUIRE(a.dt > 0.0f && isfinite(a.dt) && a.noise_scale > 0.0f && isfinite(a.noise_scale) && isfinite(a.t_max),
                "%s: bad schedule scalars", what);
    DDM_REQUIRE(a.cells_per_sigma > 0.0 && a.cells_per_sigma <= 64.0, "%s: cells_per_sigma must be in (0, 64]", what);
    return DDM_OK;
}

// pointer and pulse-width checks, and the truncation constants
static int grid_check_inputs(GridArgs &a, int64_t P, const char *what)
{
    DDM_REQUIRE(a.theta && a.pulses, "%s: null input", what);
    DDM_REQUIRE(a.ld_theta >= 5, "%s: ld_theta must be >= 5", what);
    const int64_t need = (a.n_max + a.spp - 1) / a.spp;
    DDM_REQUIRE(P >= need, "%s: pulses have %lld columns, the schedule needs %lld", what, (long long)P,
                (long long)need);
    DDM_REQUIRE(a.ld_pulses >= P, "%s: ld_pulses must be >= P", what);
    const double tr = 0.5 * erfc(kGridSigmas / 1.4142135623730951);
    a.tail_r = (float)tr;
    a.tail_norm = (float)(1.0 / (1.0 - 2.0 * tr));
    return DDM_OK;
}

static int grid_launch(GridArgs a, int64_t P, const char *what, void *stream)
{
    DDM_REQUIRE(a.N >= 0, "%s: N must be >= 0", what);
    int rc = grid_check_schedule(a, what);
    if (rc != DDM_OK) return rc;
    if (a.N == 0) return DDM_OK;
    rc = grid_check_inputs(a, P, what);
    if (rc != DDM_OK) return rc;
    DDM_REQUIRE(a.N <= 0x7FFFFFFFll, "%s: at most 2^31 - 1 rows per call", what);
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
    grid_chain_sum_kernel<<<(unsigned)((C + 255) / 256), 256, 0, st>>>(workspace_dev, T, C, C, 1, out_dev);
    DDM_CUDA_TRY(cudaGetLastError());
    return DDM_OK;
}

DDM_API size_t ddm_grid_loglik_sum_batched_workspace_floats(int64_t D, int64_t T, int64_t C, float cells_per_sigma)
{
    if (D <= 0 || T <= 0 || C <= 0 || !(cells_per_sigma > 0.0f && cells_per_sigma <= 64.0f)) return 0;
    return pot_layout(D, T, C, (double)cells_per_sigma).total;
}

DDM_API int ddm_grid_loglik_sum_batched_f32(const float *theta_dev, int64_t ld_theta, const float *x_dev,
                                            const float *pulses_dev, int64_t ld_pulses, int64_t D, int64_t T,
                                            int64_t C, int64_t P, int64_t n_max, int64_t steps_per_pulse, float dt,
                                            float t_max, float t_nd_hi, float noise_scale, float cells_per_sigma,
                                            float *out_dev, float *workspace_dev, void *stream)
{
    const char *what = "ddm_grid_loglik_sum_batched_f32";
    DDM_REQUIRE(D >= 0 && T >= 0 && C >= 0, "%s: D, T and C must be >= 0", what);
    DDM_REQUIRE(D * C <= 0x7FFFFFFFll && D * T <= 0x7FFFFFFFll, "%s: D * C and D * T must be < 2^31", what);
    GridArgs a = grid_args(theta_dev, ld_theta, pulses_dev, ld_pulses, D * T, n_max, steps_per_pulse, dt, t_max,
                           t_nd_hi, noise_scale, cells_per_sigma);
    a.mode = kModeLoglik;
    a.x = x_dev;
    int rc = grid_check_schedule(a, what);
    if (rc != DDM_OK) return rc;
    if (D * C == 0) return DDM_OK;
    DDM_REQUIRE(out_dev != nullptr, "%s: null output", what);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (T == 0) {
        DDM_CUDA_TRY(cudaMemsetAsync(out_dev, 0, (size_t)(D * C) * sizeof(float), st));
        return DDM_OK;
    }
    rc = grid_check_inputs(a, P, what);
    if (rc != DDM_OK) return rc;
    DDM_REQUIRE(workspace_dev != nullptr && x_dev != nullptr, "%s: null workspace / x", what);
    const PotLayout l = pot_layout(D, T, C, (double)cells_per_sigma);
    PotArgs p = {};
    p.a = a;
    p.T = T;
    p.C = C;
    p.groups = (int)((T + pot_group(kGridMaxCells) - 1) / pot_group(kGridMaxCells));
    DDM_REQUIRE(l.chunk * p.groups <= 0x7FFFFFFFll, "%s: too many trials per dataset", what);
    p.band_max = l.band_max;
    p.order = reinterpret_cast<const int *>(workspace_dev + l.order);
    p.flag = reinterpret_cast<int *>(workspace_dev + l.flag);
    p.rows = workspace_dev + l.rows;
    p.table = reinterpret_cast<float4 *>(workspace_dev + l.table);
    grid_trial_order_kernel<<<(unsigned)((D * T + 255) / 256), 256, 0, st>>>(x_dev, D, T,
                                                                             reinterpret_cast<int *>(workspace_dev + l.order));
    DDM_CUDA_TRY(cudaGetLastError());
    DDM_CUDA_TRY(cudaFuncSetAttribute(grid_potential_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)kPotSmemBytes));
    for (long long n0 = 0; n0 < D * C; n0 += l.chunk) {
        const long long nc = std::min(l.chunk, D * C - n0);
        p.n0 = n0;
        DDM_CUDA_TRY(cudaMemsetAsync(p.flag, 0, (size_t)nc * sizeof(int), st));
        grid_table_kernel<<<(unsigned)(nc * kPotSlices), kPotTableThreads, 0, st>>>(p);
        DDM_CUDA_TRY(cudaGetLastError());
        grid_potential_kernel<<<(unsigned)(nc * p.groups), kGridThreads, kPotSmemBytes, st>>>(p);
        DDM_CUDA_TRY(cudaGetLastError());
        grid_chain_sum_kernel<<<(unsigned)((nc + 255) / 256), 256, 0, st>>>(p.rows, T, nc, 1, T, out_dev + n0);
        DDM_CUDA_TRY(cudaGetLastError());
    }
    return DDM_OK;
}
