/*
 * ddm_b200.h -- C ABI of libddm_b200.so: the B200 (sm_100a) hot path of
 * jfour1e/SBI-for-Diffusion-Models.
 *
 * Conventions
 *   - Every pointer named *_dev is DEVICE memory owned by the caller (torch allocates
 *     it in the Python host layer); the library never allocates or frees user-visible
 *     memory and keeps no global state besides a thread-local error string and opaque
 *     MNLE weight handles the caller creates and destroys.
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).  All
 *     entry points enqueue work and return without synchronising.
 *   - Return value: 0 on success, negative on error (DDM_ERR_*); ddm_last_error()
 *     returns a thread-local description.  No C++ exception crosses this boundary.
 *   - There is no CPU fallback: without a CUDA device every compute entry point returns
 *     DDM_ERR_CUDA.
 *
 * Reference interfaces replaced (paths relative to
 * /root/reference/src/sbi_for_diffusion_models):
 *   ddm_sim_f32              models/rt_choice_model.py:112-221 (_simulate_rt_choice_batch_torch)
 *                            + :332-342 (pack_x_rt_choice) fused as the `log_rt` epilogue;
 *                            reached through rt_choice_model_simulator_torch (:251-283),
 *                            data_simulator.py:14-30 (sim_wrapper), :33-71, :74-99 and
 *                            rt_choice_model.py:286-329 (simulate_session_data_rt_choice).
 *   ddm_philox_normals_f32   models/rt_choice_model.py:186 (the torch.randn draw) -- exposes
 *                            the exact normals the simulator consumed so a run can be
 *                            replayed through the reference bit for bit.
 *   ddm_pulses_pcg64         models/rt_choice_model.py:62-91 (generate_pulse_matrix_numpy)
 *                            + models/choice_model.py:43-60 (generate_pulse_sides), i.e.
 *                            the body of proposals.py:30-40 (PulseSequenceProposal.sample).
 *   mnle_*                   potentials.py:75-117 (ConditionedMNLELogLikelihood.forward) and
 *                            the estimator.log_prob call at potentials.py:113.
 */
#ifndef DDM_B200_H
#define DDM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DDM_OK 0
#define DDM_ERR_INVALID (-1) /* bad argument (shape, range, null pointer) */
#define DDM_ERR_CUDA (-2)    /* CUDA runtime error, or no device */
#define DDM_ERR_STATE (-3)   /* bad or destroyed handle */

#define DDM_ABI_VERSION 1

int ddm_abi_version(void);
const char *ddm_last_error(void);

/* sm_count, SM clock (kHz, cudaDevAttrClockRate) and compute capability of `device`. */
int ddm_device_info(int device, int *sm_count, int *sm_clock_khz, int *cc_major, int *cc_minor);

/* Do kernel launches in this process return before the kernel has finished?  Launches a one-thread kernel that
 * waits (at most timeout_us) for a word the host raises as soon as the launch call is back; *blocking = 1 when
 * the kernel timed out instead (CUDA_LAUNCH_BLOCKING=1, Nsight Compute, compute-sanitizer, a debugger: any tool
 * that serialises launches).  The streaming ingest (ddm_sim_stream_f32 / ddm_sim_packed_f32 with ready_dev)
 * launches its persistent kernel BEFORE the copies it consumes only when this reports 0. */
int ddm_probe_launch_blocking(int64_t timeout_us, int *blocking);

/* Widest SIMD path ddm_pack_z_host uses on this CPU: 512 (AVX-512 F+DQ+VL), 256 (AVX2) or 128 (SSE2). */
int ddm_pack_simd_bits(void);

/* ---------------------------------------------------------------- simulator --- */

/* Device scratch the simulator needs per call (work queue + counters). */
size_t ddm_sim_workspace_bytes(void);

/* Layout of the workspace after the kernel has finished (all uint64):
 *   [0] trial queue cursor (>= N when done)
 *   [1] sum over trials of hit_step  == useful Euler steps executed
 *   [2] number of trials whose pulse row held values other than +-1 (slow kick path)
 *   [3] lane-steps issued (useful + idle lanes), for lane-efficiency accounting */
#define DDM_WS_QUEUE 0
#define DDM_WS_USEFUL_STEPS 1
#define DDM_WS_GENERIC_ROWS 2
#define DDM_WS_LANE_STEPS 3
#define DDM_WS_ERROR 4 /* non-zero: streaming launch timed out waiting for data */
#define DDM_WS_WORDS 8
#define DDM_MAX_PEERS 15 /* other GPUs a fused-gather launch can write to */

/*
 * Simulate N pulse-driven DDM trials.
 *
 *   theta_dev   (N, >=5) fp32, row stride ld_theta floats: [a0, lam, v, B, t_nd];
 *               ld_theta == 0 broadcasts one parameter row to every trial (a session)
 *   pulses_dev  (N, P) fp32 pulse sides, row stride ld_pulses floats; ld_pulses == 0
 *               broadcasts one row to every trial (rt_choice_model.py:166-168).  Only
 *               the first ceil(n_max / steps_per_pulse) columns are read (:178); P smaller
 *               than that is DDM_ERR_INVALID (:173-176).
 *   n_max, steps_per_pulse      time grid (rt_choice_model.py:45-59); 0 <= n_max <= 2^30
 *   dt, t_max, t_nd_hi, noise_scale
 *               the Python floats of the reference ALREADY ROUNDED to fp32 the way a
 *               float32 tensor op sees them: (float)DT_CHOICE, (float)T_MAX,
 *               (float)(T_MAX - 1e-6), (float)(mu_sensory * sqrt(DT_CHOICE)).
 *   seed, trial_offset
 *               native noise: Philox4x32-10 with key = (lo32, hi32) of seed and counter words
 *               (lo32(g), b >> 1, hi32(g), b & 1) for global trial g = trial_offset + i and block
 *               b = step / 6 -- one 128-bit block gives six 21-bit fields =
 *               three Box-Muller pairs = the normals of six consecutive steps: results do
 *               not depend on how trials are split over launches, streams or GPUs.
 *   noise_dev   NULL for native noise; otherwise (n_max, >=N) fp32 standard normals,
 *               step-major with row stride ld_noise floats (the reference draws one (N,)
 *               vector per step), consumed INSTEAD of Philox.  With shared noise the
 *               output equals the reference's bit for bit.
 *   log_rt      0: x[:,0] = rt;  1: x[:,0] = log(max(rt, 1e-6))  (pack_x_rt_choice)
 *   x_out_dev   (N, 2) fp32 contiguous: [rt, choice in {0,1,2}]
 *   steps_out_dev  NULL or (N,) int32 hit_step (first-passage step, or the window length
 *               when censored)
 *   workspace_dev  >= ddm_sim_workspace_bytes(), 8-byte aligned; zeroed by this call.
 */
int ddm_sim_f32(const float *theta_dev, int64_t ld_theta,
                const float *pulses_dev, int64_t ld_pulses,
                int64_t N, int64_t P,
                int64_t n_max, int64_t steps_per_pulse,
                float dt, float t_max, float t_nd_hi, float noise_scale,
                uint64_t seed, uint64_t trial_offset,
                const float *noise_dev, int64_t ld_noise,
                int log_rt,
                float *x_out_dev, int32_t *steps_out_dev,
                void *workspace_dev, void *stream);

/*
 * ddm_sim_f32 with the all-gather of x fused into the kernel (native noise): every finished trial's (rt, choice)
 * is stored to x_out_dev[i] AND to x_peer_blocks[d][i] for d < n_peers -- blocks in OTHER GPUs' memory mapped into
 * this process (CUDA peer access / symmetric memory), normally "rank r's slot" of each peer's gathered (world*N, 2)
 * array.  8 bytes per trial and peer travel over NVLink as posted stores while the kernel keeps simulating, so
 * sharded runs (SURVEY 8e: the path's only exchange is this gather) need no separate collective and no second pass
 * over x.  x_peer_blocks is a HOST array of n_peers device pointers (n_peers <= DDM_MAX_PEERS).  The stores are
 * visible to a peer once this launch has completed and the ranks have synchronised (a barrier on the stream).
 */
int ddm_sim_gather_f32(const float *theta_dev, int64_t ld_theta, const float *pulses_dev,
                       int64_t ld_pulses, int64_t N, int64_t P, int64_t n_max,
                       int64_t steps_per_pulse, float dt, float t_max, float t_nd_hi,
                       float noise_scale, uint64_t seed, uint64_t trial_offset, int log_rt,
                       float *x_out_dev, float *const *x_peer_blocks, int n_peers, void *workspace_dev,
                       void *stream);

/* ddm_sim_f32 launches of at most this many trials (native noise) run the small-batch kernel: CTAs of 32
 * trials in lock-step, one warp integrating while seven generate the noise of the next 42 steps into shared memory
 * -- same results bit for bit, ~15 % lower latency when the trials cannot fill the GPU (0.38 vs 0.44 ms) (process-wide, default
 * 8192; 0 switches it off). */
int ddm_sim_set_small_batch_max(int64_t max_trials);

/* How long a streaming launch (ready_dev != NULL) waits for rows that have not arrived before it sets
 * workspace[DDM_WS_ERROR] and gives the remaining trials up (process-wide, default 20 s; [1 ms, 600 s]). */
int ddm_sim_set_stream_timeout_us(int64_t timeout_us);

/*
 * Streaming variant for HOST-resident inputs: the caller enqueues the host->device copies of z
 * in chunks on a copy stream, each followed by an 8-byte copy that raises *ready_dev to the
 * number of trials delivered so far, and launches this ONE persistent kernel on another stream
 * without waiting for them.  A warp that claims trials beyond *ready_dev sleeps until the copy
 * engine has caught up, so ingest over PCIe and simulation overlap inside a single launch and
 * there is only one drain phase per batch.  All copies must be enqueued BEFORE this call (the
 * kernel never blocks them); if *ready_dev makes no progress for 20 s the kernel gives up and
 * sets workspace[DDM_WS_ERROR].  Native Philox noise only; same results as ddm_sim_f32.
 */
int ddm_sim_stream_f32(const float *theta_dev, int64_t ld_theta,
                       const float *pulses_dev, int64_t ld_pulses,
                       int64_t N, int64_t P,
                       int64_t n_max, int64_t steps_per_pulse,
                       float dt, float t_max, float t_nd_hi, float noise_scale,
                       uint64_t seed, uint64_t trial_offset, int log_rt,
                       float *x_out_dev, void *workspace_dev,
                       const uint64_t *ready_dev, void *stream);

/*
 * PCIe ingest path for HOST-resident z.  Pulse sides are +-1, so a 340-byte fp32 row carries 32 bytes
 * of information; over a ~55 GB/s PCIe 5 x16 link the fp32 rows take longer to copy than the kernel
 * needs to simulate them.  ddm_pack_z_host (host code, n_threads CPU threads, no CUDA) turns rows
 * [theta (5), pulses (n_pulses <= 96)] of z_host (row stride ld floats) into 32-byte records
 * [theta bits x 5, sign masks x 3] (bit j of mask w = pulses[32 w + j] > 0; bits past n_pulses = 1) in
 * packed_host (N x 8 uint32) and returns the number of rows holding a pulse value other than +-1
 * (such batches must take the fp32 entry points), or a negative DDM_ERR_*.
 * ddm_sim_packed_f32 simulates from the records (device copy, 16-byte aligned): same arguments and
 * bit-identical results as ddm_sim_f32 / ddm_sim_stream_f32 (ready_dev != NULL: streaming ingest).
 */
int64_t ddm_pack_z_host(const float *z_host, int64_t ld, int64_t N, int64_t n_pulses, uint32_t *packed_host,
                        int n_threads);
/* The device->host mirror: ddm_pack_z_dev turns rows of a DEVICE z (row stride ld floats) into the same 32-byte
 * records (one warp per row; *generic_rows_dev = rows holding a pulse value other than +-1, whose records must not
 * be used), and ddm_unpack_z_host (host code, n_threads CPU threads) rebuilds z_host rows [theta (5), pulses (+-1)]
 * from records: a caller that wants z in host memory moves 32 instead of 340 bytes per trial over the link.  With
 * AVX-512, ld == 5 + n_pulses and a 64-byte aligned z_host the rows leave with non-temporal stores. */
int ddm_pack_z_dev(const float *z_dev, int64_t ld, int64_t N, int64_t n_pulses, uint32_t *packed_dev,
                   uint64_t *generic_rows_dev, void *stream);
int ddm_unpack_z_host(const uint32_t *packed_host, int64_t N, int64_t n_pulses, float *z_host, int64_t ld, int n_threads);

/* The ingest loop of one batch in one call (host code + copies on copy_stream): for every chunk of
 * chunk_rows rows, pack it into staging_host (pinned, N x 8 uint32), enqueue its copy to packed_dev and
 * an 8-byte copy of marks_host[k] (pinned; rows delivered once chunk k has landed, the last entry >= N)
 * to *ready_dev -- what a ddm_sim_packed_f32 launched with ready_dev waits on.  *generic_rows = rows
 * holding a pulse value other than +-1. */
int ddm_ingest_packed(const float *z_host, int64_t ld, int64_t N, int64_t n_pulses, int64_t chunk_rows,
                      uint32_t *staging_host, uint32_t *packed_dev, uint64_t *ready_dev,
                      const uint64_t *marks_host, int n_threads, void *copy_stream, int64_t *generic_rows);
int ddm_sim_packed_f32(const uint32_t *packed_dev, int64_t N, int64_t n_max, int64_t steps_per_pulse, float dt,
                       float t_max, float t_nd_hi, float noise_scale, uint64_t seed, uint64_t trial_offset,
                       int log_rt, float *x_out_dev, int32_t *steps_out_dev, void *workspace_dev,
                       const uint64_t *ready_dev, void *stream);

/* The standard normals ddm_sim_f32 consumes under native noise for trials
 * [trial_offset, trial_offset + N) and steps [0, n_steps): out (n_steps, N) step-major,
 * row stride ld_out floats. */
int ddm_philox_normals_f32(uint64_t seed, uint64_t trial_offset, int64_t N, int64_t n_steps,
                           float *out_dev, int64_t ld_out, void *stream);

/* Same indexing, raw Philox4x32-10 words (integer; checked bit-exactly on the host). */
int ddm_philox_words_u32(uint64_t seed, uint64_t trial_offset, int64_t N, int64_t n_steps,
                         uint32_t *out_dev, int64_t ld_out, void *stream);

/* ------------------------------------------------------------ pulse generator --- */

/*
 * Rows [first_trial, first_trial + n) of generate_pulse_matrix_numpy(rng, ., P, p) for a
 * NumPy PCG64 generator whose bit_generator.state is (state, inc) before the call.
 * threshold = ceil(clip(p_success, 0, 1) * 2^53).  out (n, P) fp32 +-1, row stride ld.
 * Bit-identical to NumPy (integer arithmetic only).
 */
int ddm_pulses_pcg64(uint64_t state_hi, uint64_t state_lo, uint64_t inc_hi, uint64_t inc_lo,
                     uint64_t first_trial, int64_t n, int64_t P, uint64_t threshold,
                     float *out_dev, int64_t ld, void *stream);

/* Host-side helper: PCG64 state after `draws` more doubles (no device work). */
int ddm_pcg64_advance(uint64_t *state_hi, uint64_t *state_lo, uint64_t inc_hi, uint64_t inc_lo,
                      uint64_t draws);

/* ------------------------------------------------------- MNLE log-likelihood --- */

/*
 * Packed fp32 parameters of the MNLE density estimator the reference builds with
 * likelihood_nn(model="mnle", hidden_features=128, num_transforms=10, num_bins=24,
 * log_transform_x=True, z_score_theta="independent", z_score_x="independent")
 * (mnle.py:31-39), in this order, z-scoring of the condition folded into the first layers
 * by the host packer (sbi_for_diffusion_models_b200/mnle_net.py):
 *   categorical net: W0[128][85] b0[128] W1[128][128] b1[128] W2[128][128] b2[128]
 *                    Wo[K][128] bo[K]                      (K = n_choices, sigmoid)
 *   flow k = 0..9:   W1[128][86] b1[128] W2[128][128] b2[128] W3[71][128] b3[71]   (ReLU)
 *   mu_y, sigma_y    standardisation of log rt
 * mnle_packed_floats(K) is the required length (0 if K is unsupported).
 */
size_t mnle_packed_floats(int n_choices);

/* Copies the packed parameters to the current device and builds the tensor-core operand pack
 * from them there: one kernel on the legacy default stream, waited for before the call returns.
 * *handle_out is an opaque read-only handle owned by the caller (mnle_destroy).  One handle per
 * (process, device). */
int mnle_create(const float *packed_host, size_t n_floats, int n_choices, void **handle_out);
int mnle_destroy(void *handle);

/* estimator.log_prob(x (1,R,2), condition=(R,85)) -> (1,R)   (potentials.py:113):
 * x_dev (R,2) = [rt seconds, choice], cond_dev (R,85) row stride ld_cond, out_dev (R,). */
int mnle_log_prob_rows_f32(void *handle, const float *x_dev, const float *cond_dev, int64_t ld_cond,
                           int64_t R, float *out_dev, void *stream);

/* Same call with the per-row chain (log rt, ten splines, categorical head, final sum) in fp64 on the fp32
 * conditioner outputs -- the accuracy anchor for TRAINED estimators: a trained flow's narrow, steep bins
 * amplify fp32 rounding of the knot positions to ~3e-4 per row in ANY fp32 evaluation (the reference's torch
 * CPU call included); this path sits ~1e-6 from exact arithmetic.  Same arguments and output type. */
int mnle_log_prob_rows_precise_f32(void *handle, const float *x_dev, const float *cond_dev, int64_t ld_cond,
                                   int64_t R, float *out_dev, void *stream);

/* Same call on the 5th-generation tensor cores: the 86-wide context of each row is split into bf16
 * hi + lo operand images in shared memory and every layer (first layers included, K padded to 96) runs
 * as three tcgen05.mma per product; two 128-row tiles per CTA in ping-pong.  Per-row results within ~1e-4 of the fp32 kernel on
 * the default-init net (see mnle_loglik_sum_tc_f32 for the accuracy model). */
int mnle_log_prob_rows_tc_f32(void *handle, const float *x_dev, const float *cond_dev, int64_t ld_cond,
                              int64_t R, float *out_dev, void *stream);

/* Scratch floats mnle_loglik_sum_* needs for T trials x C chains. */
size_t mnle_loglik_workspace_floats(int64_t T, int64_t C);

/*
 * ConditionedMNLELogLikelihood.forward (potentials.py:75-117) without materialising the
 * (T*C, 85) condition matrix:  out[c] = sum_t log p(x[t] | [theta[c], pulses[t]]).
 *   theta_dev (C,5) row stride ld_theta; x_dev (T,2) contiguous; pulses_dev (T,>=80) row
 *   stride ld_pulses; out_dev (C,); workspace_dev >= mnle_loglik_workspace_floats(T,C) floats.
 * The reduction order is fixed, so results are reproducible run to run.
 * _simt: fp32 CUDA-core kernel (accuracy anchor).
 */
int mnle_loglik_sum_simt_f32(void *handle, const float *theta_dev, int64_t ld_theta, const float *x_dev,
                             const float *pulses_dev, int64_t ld_pulses, int64_t T, int64_t C,
                             float *out_dev, float *workspace_dev, void *stream);
/* _precise: fp32 networks, fp64 spline chain (see mnle_log_prob_rows_precise_f32); same workspace. */
int mnle_loglik_sum_precise_f32(void *handle, const float *theta_dev, int64_t ld_theta, const float *x_dev,
                                const float *pulses_dev, int64_t ld_pulses, int64_t T, int64_t C,
                                float *out_dev, float *workspace_dev, void *stream);
/* _tc64: the networks on the tensor cores (rows-mode tcgen05 forward over the T*C expanded rows, writing the raw
 * spline parameters and choice logits), then the spline chain, categorical head and the sum over trials in fp64:
 * the accuracy of _precise at a fraction of its time.  T*C <= 8e6; workspace_dev 256-byte aligned with at least
 * mnle_loglik_tc64_workspace_floats(n_choices, T, C) floats (~3 KB per row). */
size_t mnle_loglik_tc64_workspace_floats(int n_choices, int64_t T, int64_t C);
int mnle_loglik_sum_tc64_f32(void *handle, const float *theta_dev, int64_t ld_theta, const float *x_dev,
                             const float *pulses_dev, int64_t ld_pulses, int64_t T, int64_t C, float *out_dev,
                             float *workspace_dev, void *stream);

/*
 * Value and gradient with respect to theta of the same sum (what autograd gives the reference's
 * NUTS sampler through potentials.py:112 with track_gradients=True): out_dev (C,),
 * grad_dev (C,5) row-major, grad[c][i] = d out[c] / d theta[c][i].  Forward-mode (five tangents
 * per row) on the fp32 CUDA-core path; C <= 65535.  workspace_dev >=
 * mnle_loglik_grad_workspace_floats(T,C) floats.
 */
size_t mnle_loglik_grad_workspace_floats(int64_t T, int64_t C);
int mnle_loglik_sum_grad_f32(void *handle, const float *theta_dev, int64_t ld_theta, const float *x_dev,
                             const float *pulses_dev, int64_t ld_pulses, int64_t T, int64_t C,
                             float *out_dev, float *grad_dev, float *workspace_dev, void *stream);

/*
 * The same value and gradient in REVERSE mode on the tensor cores (what autograd does for the reference, with
 * the MNLE training step's kernels): the (T*C, 85) rows of the reference's expansion go through the tcgen05
 * forward with activations kept, the per-row spline sweep, the tcgen05 backward-data pass, and the five theta
 * columns of every first layer are contracted and summed over the trials in a fixed order.  Same arguments as
 * mnle_loglik_sum_grad_f32; T*C <= 8e6 rows; workspace_dev 256-byte aligned with at least
 * mnle_loglik_grad_tc_workspace_floats(n_choices, T, C) floats (~6.2 KB per row: ~46 GiB at 8e6 rows).
 */
size_t mnle_loglik_grad_tc_workspace_floats(int n_choices, int64_t T, int64_t C);
int mnle_loglik_sum_grad_tc_f32(void *handle, const float *theta_dev, int64_t ld_theta, const float *x_dev,
                                const float *pulses_dev, int64_t ld_pulses, int64_t T, int64_t C, float *out_dev,
                                float *grad_dev, float *workspace_dev, void *stream);

/*
 * Same contract on the 5th-generation tensor cores (tcgen05.mma, accumulators in TMEM): the
 * 128x128 / 128x71 layers run as bf16 hi/lo split GEMMs (three MMAs per product, fp32
 * accumulate), the five global parameters enter through a K = 32 six-term stage, and the
 * pulse / choice part of every first layer is computed once per trial.  Sums agree with the
 * _simt kernel to ~1e-6 relative.  workspace_dev >= mnle_loglik_tc_workspace_floats(T,C) floats,
 * 16-byte aligned.
 */
size_t mnle_loglik_tc_workspace_floats(int64_t T, int64_t C);
int mnle_loglik_sum_tc_f32(void *handle, const float *theta_dev, int64_t ld_theta, const float *x_dev,
                           const float *pulses_dev, int64_t ld_pulses, int64_t T, int64_t C,
                           float *out_dev, float *workspace_dev, void *stream);

/*
 * D independent datasets in one launch (the SBC loop, mnle.py:183-218, evaluates one potential per
 * dataset): theta_dev (D*C,5), x_dev (D*T,2), pulses_dev (D*T,>=80), out_dev (D*C,);
 * out[d*C + c] = sum_t log p(x[d*T + t] | [theta[d*C + c], pulses[d*T + t]]).
 * D*T <= 524280 per call.
 */
size_t mnle_loglik_batched_tc_workspace_floats(int64_t D, int64_t T, int64_t C);
int mnle_loglik_sum_batched_tc_f32(void *handle, const float *theta_dev, int64_t ld_theta, const float *x_dev,
                                   const float *pulses_dev, int64_t ld_pulses, int64_t D, int64_t T, int64_t C,
                                   float *out_dev, float *workspace_dev, void *stream);

/*
 * D observed sessions of different lengths in one launch: session d owns the flat trials
 * [trial_offsets[d], trial_offsets[d+1]) of x_dev (N,2) and pulses_dev (N,>=80, row stride ld_pulses);
 * theta_dev (D*C,5) row stride ld_theta, out_dev (D*C,);
 * out[d*C + c] = sum over the trials t of session d of log p(x[t] | [theta[d*C + c], pulses[t]]),
 * 0 for an empty session.  Every output is the bits mnle_loglik_sum_tc_f32 gives for that session alone.
 * trial_offsets_dev: DEVICE int64 (D+1,) with offsets[0] = 0, offsets[D] = N and offsets[d] <= offsets[d+1];
 * the kernels do not check them (they would have to copy them to the host), the caller must.
 * N <= 524280 per call; workspace_dev >= mnle_loglik_sessions_tc_workspace_floats(D,N,C) floats, 16-byte aligned.
 */
size_t mnle_loglik_sessions_tc_workspace_floats(int64_t D, int64_t N, int64_t C);
int mnle_loglik_sum_sessions_tc_f32(void *handle, const float *theta_dev, int64_t ld_theta, const float *x_dev,
                                    const float *pulses_dev, int64_t ld_pulses, const int64_t *trial_offsets_dev,
                                    int64_t D, int64_t N, int64_t C, float *out_dev, float *workspace_dev, void *stream);
/* The same ragged sessions on the _tc64 path (tensor-core networks, fp64 spline chain and fp64 sums over each
 * session's trials in trial order); every output is the bits mnle_loglik_sum_tc64_f32 gives for that session
 * alone.  N*C <= 8e6 and D <= 65535 per call; workspace_dev 256-byte aligned with at least
 * mnle_loglik_sessions_tc64_workspace_floats(n_choices, D, N, C) floats. */
size_t mnle_loglik_sessions_tc64_workspace_floats(int n_choices, int64_t D, int64_t N, int64_t C);
int mnle_loglik_sum_sessions_tc64_f32(void *handle, const float *theta_dev, int64_t ld_theta, const float *x_dev,
                                      const float *pulses_dev, int64_t ld_pulses, const int64_t *trial_offsets_dev,
                                      int64_t D, int64_t N, int64_t C, float *out_dev, float *workspace_dev, void *stream);

/*
 * estimator.sample(sample_shape, condition) (sbi MixedDensityEstimator.sample): for each of B condition rows
 * (cond_dev (B,85), row stride ld_cond) S draws of [rt seconds, choice].  x_out_dev (S,B,2) contiguous: sample s of
 * condition b is row r = s*B + b.  The choice c is the smallest j with u_c < sum_{i<=j} softmax(logits)_i in fp64
 * (K - 1 when rounding leaves u_c at or above the total); then u = n ~ N(0,1) goes through the ten spline transforms
 * INVERTED, transform 9 first, each the identity outside [-10, 10] and located on the height knots inside, and
 * rt = exp(mu_y + sigma_y * u).  The networks run on the tensor cores (the rows-mode tcgen05 forward, once for the
 * categorical net and once for the ten conditioners on the sampled choice), the choice draw and the inverse chain
 * in fp64.  rt is NOT clamped to the simulator's window: the estimator is a continuous density.
 *   seed, sample_offset
 *               native draws (draws_dev == NULL): one Philox4x32-10 block per row, key = (lo32(seed), hi32(seed)),
 *               counter = (lo32(g), hi32(g), b, 0x4D4E4C45) for the global sample index g = sample_offset + s, so
 *               splitting S over calls with matching offsets gives the bits of one call.  From its words w0..w3:
 *                 u_c = (w0 + 0.5) * 2^-32
 *                 u_1 = (((w1 >> 5) << 26 | (w2 >> 6)) + 0.5) * 2^-53
 *                 n   = sqrt(-2 log u_1) * cos(pi * (w3 + 0.5) * 2^-31)            (fp64)
 *   draws_dev   NULL, or (S*B, 2) fp32 [u_c in (0,1), n] per row, used INSTEAD of Philox.
 * B*S <= 8e6 per call; workspace_dev 256-byte aligned with at least mnle_sample_tc_workspace_floats(K, B, S)
 * floats (~3.7 KB per row; 0 when the shape is out of range).
 */
size_t mnle_sample_tc_workspace_floats(int n_choices, int64_t B, int64_t S);
int mnle_sample_tc_f32(void *handle, const float *cond_dev, int64_t ld_cond, int64_t B, int64_t S,
                       uint64_t seed, uint64_t sample_offset, const float *draws_dev,
                       float *x_out_dev, float *workspace_dev, void *stream);

/* ------------------------------------------------------------ MNLE training --- */

/*
 * One optimisation step of what sbi's MNLE.train does for the reference (mnle.py:41-48; Adam on
 * -mean log p over minibatches of TRAIN_BATCH_SIZE rows, run_config.py:12), on device buffers the
 * caller owns.  params_dev / grad_dev / m_dev / v_dev hold mnle_packed_floats(K) floats in the
 * packed layout above (during training the condition is standardised by the caller, so the first
 * layers are the raw ones; mu_y / sigma_y at the tail are read, never updated).
 *
 * mnle_train_nll_grad_f32: minibatch row r is dataset row row_index_dev[r] (int64; NULL = rows
 * 0..R-1) of x_dev (N,2) = [rt seconds, choice] and cond_dev (N,85) with row stride ld_cond.
 *   stats_dev[0] = -mean_r log p(x_r | cond_r),  stats_dev[1] = |grad|^2
 *   grad_dev[i]  = d stats[0] / d params[i]   (NULL: loss only, e.g. the validation pass)
 * All reductions run in a fixed order: results are bit-reproducible.  workspace_dev >=
 * mnle_train_workspace_floats(K, R) floats, 16-byte aligned.  The forward pass runs on the tensor cores
 * (tcgen05, bf16 hi/lo operands ~ 17 bits: activations within ~1e-5 of fp32, so a ReLU unit that close to
 * its kink may be masked differently) and so do the backward-data and weight-gradient GEMMs; flags =
 * DDM_TRAIN_FP32_FORWARD runs forward and backward-data on the fp32 CUDA cores (accuracy anchor, ~0.15 ms
 * slower per 4096 rows; the weight gradients stay on the tensor cores).
 *
 * mnle_train_adam_f32: torch.optim.Adam update (no weight decay) for step = 1, 2, ... after
 * scaling the gradient like torch.nn.utils.clip_grad_norm_(max_grad_norm) using stats_dev[1]
 * (max_grad_norm <= 0: no clipping).
 */
size_t mnle_train_workspace_floats(int n_choices, int64_t R);
#define DDM_TRAIN_FP32_FORWARD 1 /* flags: forward pass on the fp32 CUDA cores instead of the tensor cores */
int mnle_train_nll_grad_f32(const float *params_dev, int n_choices, const float *x_dev, const float *cond_dev,
                            int64_t ld_cond, const int64_t *row_index_dev, int64_t R, float *stats_dev,
                            float *grad_dev, float *workspace_dev, int flags, void *stream);
int mnle_train_adam_f32(float *params_dev, const float *grad_dev, float *m_dev, float *v_dev, int n_choices,
                        const float *stats_dev, float lr, float beta1, float beta2, float eps, int64_t step,
                        float max_grad_norm, void *stream);

/* Debug aid: when trace_dev != NULL, CTA 0 of every following mnle_loglik_sum_tc_f32 launch writes
 * 34 stages x 2 tiles x 8 clock64() stamps there (issuer saw A operand / had the weights, epilogue
 * saw the accumulators / finished).  NULL switches it off (the default). */
int mnle_tc_set_trace(long long *trace_dev);

/* Tensor-core building-block check: D (128,N) = A (128,128) * B (N,128)^T through the smem
 * operand layout, UMMA descriptors, tcgen05.mma and TMEM loads of the fused kernel.
 * passes = 1: bf16(A) bf16(B); passes = 3: bf16 hi/lo split (near-fp32).  lbo_a / lbo_b / sbo = 0
 * use the layout's own descriptor strides (non-zero values are for hardware probing only). */
int mnle_tc_selftest(const float *a_dev, const float *b_dev, int N, int passes, uint32_t lbo_a,
                     uint32_t lbo_b, uint32_t sbo, float *d_dev, void *stream);

/* ------------------------------------------------------------ slice sampler --- */

/*
 * Bookkeeping of the many-chain slice sampler that drives the potential (host side: samplers.py; the reference hands
 * this job to sbi's MCMCPosterior, mnle.py:77-93).  Every chain runs its own state machine (Neal 2003: stepping out
 * with a limit, then shrinkage).  Per iteration: ddm_slice_propose_f32 writes the point each chain needs evaluated next
 * into row c of query_dev (N, D); the caller evaluates the potential there; ddm_slice_update_f32 applies f_dev (N,) --
 * bracket moves, acceptance, width tuning, coordinate / sweep accounting, recording of draws, start of the next update.
 * state_ptrs: HOST array of 16 device pointers [x (N,D), lp, width (N,D), tuned (N,D), lo, hi, x0, log_y, J, K (float),
 * d, sweeps, taken, phase, nshr (int64), out (S,N,D)]; state_ints: HOST array [N, D, S, thin, warmup, total sweeps,
 * max_step_out, max_shrink]; u_dev (4, N) uniforms in (0, 1) of this iteration.
 */
int ddm_slice_propose_f32(const void *const *state_ptrs, const int64_t *state_ints, const float *u_dev, float *query_dev,
                          void *stream);
int ddm_slice_update_f32(const void *const *state_ptrs, const int64_t *state_ints, const float *u_dev, const float *f_dev,
                         void *stream);

#ifdef __cplusplus
}
#endif
#endif /* DDM_B200_H */
