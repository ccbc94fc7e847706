/*
 * lgae_b200.h -- C ABI of the B200-native LGAE hot path (fp64, sm_100a).
 *
 * Drop-in boundary: the reference (zichunhao/lgn-autoencoder) is pure Python; its "operator API" for this
 * path is the lgn/ module surface.  The Python package lgn_autoencoder_b200 mirrors that surface and calls
 * the entry points below through ctypes.  Every pointer is a DEVICE pointer to float64 unless stated; every
 * function returns 0 on success or a negative LGAE_E_* code (never throws), and enqueues its work on the
 * CUDA stream passed as `stream` (a cudaStream_t cast to void*).
 *
 * Reference interfaces replaced (paths relative to the reference repository):
 *   lgae_encoder_forward / _backward   lgn/models/lgn_encoder.py:255-336  (LGNEncoder.forward) + autograd
 *   lgae_decoder_forward / _backward   lgn/models/lgn_decoder.py:218-303  (LGNDecoder.forward) + autograd
 *   lgae_level_forward  / _backward    lgn/models/lgn_levels.py:96-121    (LGNNodeLevel.forward), which wraps
 *                                      lgn/cg_lib/cg_ops.py:135-298 (cg_product, aggregate and power),
 *                                      lgn/nn/g_nn.py:260-278 (CatMixReps), lgn/models/lgn_cg.py:167 (edge features),
 *                                      lgn/nn/position_levels.py:118-209 (RadPolyTrig.forward),
 *                                      lgn/cg_lib/zonal_functions.py:123-248 (pairwise zonal functions / norms)
 *   lgae_mlp_forward    / _backward    lgn/models/lgn_levels.py:191-227   (CGMLP.forward)
 *   lgae_chamfer                       utils/losses/chamfer_loss/chamfer_loss.py:16-31 + distance_sq.py:263-304
 *   lgae_cg_product_*, lgae_mix_*      lgn/cg_lib/cg_ops.py:135-218, lgn/nn/g_nn.py:95-117 (generic layer API)
 *
 * Internal activation layout ("node layout"): complex numbers are interleaved (re, im) pairs.
 *   scalars S : (B, N, C, 2)         vectors V : (B, N, C, 4, 2)   (canonical basis of the (1,1) irrep)
 * The reference's planar layout (2, B, N, C, d) only appears at the module boundary (latent, output).
 */
#ifndef LGAE_B200_H
#define LGAE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LGAE_MAX_LEVELS 8
#define LGAE_MAX_LINEAR 12
#define LGAE_MAX_CHANNELS 8

#define LGAE_OK 0
#define LGAE_E_BADARG (-1)      /* null pointer / negative size / inconsistent descriptor              */
#define LGAE_E_UNSUPPORTED (-2) /* configuration outside what the fused path implements                  */
#define LGAE_E_CUDA (-3)        /* a CUDA runtime call or kernel launch failed (see lgae_last_cuda_error) */
#define LGAE_E_NODEVICE (-4)

/* latent aggregation modes (lgn/models/lgn_encoder.py:419-496) */
#define LGAE_LATENT_MEAN 0
#define LGAE_LATENT_MINMAX 1 /* "min&max": tau doubles                                                    */
#define LGAE_LATENT_MIN 2
#define LGAE_LATENT_MAX 3
#define LGAE_LATENT_SUM 4
#define LGAE_LATENT_MIX 5    /* nodes x channels mixed by the latent MixReps; no pooling                  */

/* CGMLP activations (LgaeModelDesc::mlp_activation), the reference's get_activation_fn table.  Any other code is
 * refused with LGAE_E_UNSUPPORTED when has_mlp is set. */
#define LGAE_ACT_LEAKYRELU 0 /* LeakyReLU(0.01)                                                           */
#define LGAE_ACT_RELU 1
#define LGAE_ACT_ELU 2       /* alpha = 1                                                                  */
#define LGAE_ACT_SIGMOID 3
#define LGAE_ACT_LOGSIGMOID 4
#define LGAE_ACT_TANH 5
#define LGAE_ACT_ATAN 6
#define LGAE_ACT_COUNT 7

/* get_real modes (utils/utils.py:194-207): how the complex reconstruction becomes the real 4-momenta the loss sees.
 * The reference's default is 'real' (main.py:295-300); examples/main.sh and the benchmarked configuration use 'sum'. */
#define LGAE_GET_REAL_REAL 0
#define LGAE_GET_REAL_IMAG 1
#define LGAE_GET_REAL_SUM 2
#define LGAE_GET_REAL_MEAN 3
#define LGAE_GET_REAL_NORM 4 /* sqrt(re^2 + im^2 + 1e-16) */

/* Model descriptor: geometry + offsets (in doubles) of every parameter inside one flat fp64 buffer `theta`.
 * Gradients are written to a buffer `gtheta` with the same offsets.  Parameter shapes are the reference's
 * state-dict shapes (SURVEY.md appendix A.9); complex weights are planar (2, C_out, C_in). */
typedef struct LgaeModelDesc {
    int32_t is_decoder;
    int32_t n_levels;                       /* number of LGN message-passing levels                         */
    int32_t n_particles;                    /* N                                                            */
    int32_t n_basis;                        /* K = 2*num_basis_fn radial basis functions (encoder only)     */
    int32_t channels[LGAE_MAX_LEVELS + 1];  /* C_0 .. C_L                                                   */
    int32_t has_mlp;                        /* CGMLP after each level                                       */
    int32_t mlp_hidden;                     /* number of hidden layers (mlp_depth); linears = hidden + 1    */
    int32_t mlp_width[LGAE_MAX_LEVELS];     /* hidden width of level l = mlp_width_mul * 2 * C_{l+1}        */
    int32_t latent_mode;                    /* encoder: LGAE_LATENT_*                                       */
    int32_t tau_s, tau_v;                   /* encoder: latent MixReps outputs; decoder: latent inputs      */
    int32_t mlp_activation;                 /* CGMLP hidden-layer activation: LGAE_ACT_* (0: LeakyReLU(0.01))  */
    int64_t n_params;                       /* length of theta                                              */
    int64_t off_in00, off_in11;             /* input_func_node.weights.(0, 0) / (1, 1): (2, C_0, 1)         */
    int64_t off_rad_a[LGAE_MAX_LEVELS], off_rad_b[LGAE_MAX_LEVELS], off_rad_c[LGAE_MAX_LEVELS];
    int64_t off_rad_w0[LGAE_MAX_LEVELS], off_rad_b0[LGAE_MAX_LEVELS];   /* linear.0: (2C|C, K), (2C|C)      */
    int64_t off_rad_w1[LGAE_MAX_LEVELS], off_rad_b1[LGAE_MAX_LEVELS];   /* linear.1                          */
    int64_t off_mix00[LGAE_MAX_LEVELS], off_mix11[LGAE_MAX_LEVELS];     /* cat_mix weights (2, C', 5C)       */
    int64_t off_mlp_w[LGAE_MAX_LEVELS][LGAE_MAX_LINEAR];
    int64_t off_mlp_b[LGAE_MAX_LEVELS][LGAE_MAX_LINEAR];
    int64_t off_lat00, off_lat11;           /* encoder mix_reps: (2, tau_s, C_L) / (2, tau_v, C_L) [x N: mix] */
    int64_t off_graph00, off_graph11;       /* decoder latent_to_graph: (2, N, tau_s) / (2, N, tau_v)        */
    int64_t off_out00, off_out11;           /* decoder mix_to_output: (2, 1, C_L)                            */
    double input_scale;                     /* encoder: p4 is multiplied by this first (lgn_encoder.py:371); 0 means 1 */
    /* Maximal irrep dimension of every level: 0 or 2 = maxdim 2 (nodes (0,0), (1,1)); 3 = maxdim 3 (nodes (0,0), (1,1), (2,0),
     * (0,2), (2,2)), which the forward entry points run and everything else refuses with LGAE_E_UNSUPPORTED.  Others: refused. */
    int32_t maxdim;
    int64_t off_mix20[LGAE_MAX_LEVELS], off_mix02[LGAE_MAX_LEVELS], off_mix22[LGAE_MAX_LEVELS];   /* maxdim 3: cat_mix weights */
} LgaeModelDesc;

/* ---- library / device ---------------------------------------------------------------------------- */
int lgae_version(void);
const char* lgae_error_string(int code);
const char* lgae_last_cuda_error(void);
int lgae_device_sm_count(void);
/* Number of kernels launched by this library since load (all entry points); bench.py reports the delta. */
int64_t lgae_launch_count(void);
/* Per-kernel timing for bench.py: while enabled every kernel launch of the library is bracketed by CUDA events on its
 * stream (do not enable during CUDA-graph capture).  lgae_timing_report synchronises the device and writes one line
 * "name launches total_ms" per kernel into buf; returns the number of lines or a negative error code. */
void lgae_timing_enable(int32_t on);
int lgae_timing_report(char* buf, int32_t cap);

/* ---- workspace geometry -------------------------------------------------------------------------- */
/* Doubles of per-batch workspace holding what the backward pass keeps (level inputs, neighbour sums,
 * pre-MLP scalars, MLP activations).  Allocated by the caller (torch.empty), never by the library. */
int64_t lgae_workspace_doubles(const LgaeModelDesc* d, int32_t batch);
/* Offset (doubles) of one saved tensor inside the workspace, or -1.  kind: 0 = S_in[level] (B,N,C,2),
 * 1 = V_in[level] (B,N,C,4,2) (level == n_levels gives the final features), 2 = pre-MLP scalars of level,
 * 3 = canonical momenta y (B,N,4,2), 4 = neighbour sums of level (B,N,C,10,2), 5 = masses (B,N) (encoder),
 * 6 = MLP activations of level (hidden, B*N, padded width), 7 = radial weights of level (B,N,C,32,4) (encoder, N <= 32),
 * 8 = dL/dR of level (B,N,C,32,4) (encoder, N <= 32; one buffer per level). */
int64_t lgae_workspace_offset(const LgaeModelDesc* d, int32_t batch, int32_t kind, int32_t level);
/* maxdim 3 (forward only): the workspace holds kinds 0, 1 (S, V: the (0,0) and (1,1) parts), 2 (pre-MLP scalars), 3 (y,
 * decoder), 5 (masses), 6 (MLP activations) as above and kind 9 = H_in[level] (B,N,C,15,2), the (2,0) | (0,2) | (2,2) parts
 * (level >= 1), plus the neighbour sums of the level being evaluated; no saved state for an adjoint (kinds 4, 7, 8 return -1). */
/* Doubles of scratch for the per-CTA rows of parameter-gradient partials the backward entry points write (every
 * backward kernel owns a block of compact rows; one reduce launch sums them into gtheta, in a fixed order). */
int64_t lgae_partials_doubles(const LgaeModelDesc* d, int32_t batch);
/* Doubles of the one caller-allocated scratch buffer of lgae_encoder_backward_tiled / lgae_decoder_backward_tiled: the
 * adjoints of the neighbour sums (B*N*C*10 complex), the encoder's dL/dR of one level (B * ceil(N/32) * N * C * 128 doubles:
 * 1.57 GB at B = 512, N = 150, C = 4) and the rows of parameter-gradient partials.  -1 for bad arguments, -2
 * (LGAE_E_UNSUPPORTED) for a configuration the tiled adjoint cannot run (e.g. a latent or input-map adjoint whose shared
 * memory does not fit at this particle count).  Needs no GPU. */
int64_t lgae_backward_tiled_scratch_doubles(const LgaeModelDesc* d, int32_t batch);

/* ---- whole-model entry points -------------------------------------------------------------------- */
/* LGNEncoder.forward.  p4 (B,N,4) Cartesian (E,px,py,pz); node_mask (B,N) uint8 or NULL (=> p4[...,0] != 0).
 * Outputs, planar like the reference: lat00 (2,B,1,T_s,1), lat11 (2,B,1,T_v,4) with T = tau (x2 for min&max);
 * sel (int32, device) receives the selected particle indices for min/max modes: (4, 2, B, tau_max) laid out as
 * [kind: smin, smax, vmin, vmax][re/im][b][t]; may be NULL for mean/sum/mix. */
int lgae_encoder_forward(const LgaeModelDesc* d, const double* theta, const double* p4, const uint8_t* node_mask,
                         int32_t batch, double* workspace, double* lat00, double* lat11, int32_t* sel, void* stream);
/* Adjoint.  g_lat00 / g_lat11 may be NULL (treated as zero).  gtheta (n_params) is OVERWRITTEN with the
 * parameter gradient.  partials: scratch of lgae_partials_doubles(d, batch).  Needs N <= 32 (any N: the tiled entry point).
 * l1_lambda != 0 folds the L1 regulariser (lgn_encoder.py:249-250, utils/train.py:483-492) into the same launches:
 * gtheta += l1_lambda sign(theta) and, when loss_accumulate != NULL, loss_accumulate[0] += l1_lambda |theta|_1. */
int lgae_encoder_backward(const LgaeModelDesc* d, const double* theta, const double* p4, const uint8_t* node_mask,
                          int32_t batch, double* workspace, const int32_t* sel, const double* g_lat00,
                          const double* g_lat11, double* gtheta, double* partials, double l1_lambda,
                          double* loss_accumulate, void* stream);
/* The same adjoint for any N >= 1 (the forward is lgae_encoder_forward unchanged).  It works on blocks of 32 particles and
 * re-evaluates the radial weights tile by tile instead of reading saved ones; at N <= 32 it runs one block per jet.
 * scratch: lgae_backward_tiled_scratch_doubles(d, batch) doubles, in place of `partials`; everything else as
 * lgae_encoder_backward (gtheta overwritten, L1 folded in).  LGAE_E_UNSUPPORTED, before any launch, where the size query
 * returns -2. */
int lgae_encoder_backward_tiled(const LgaeModelDesc* d, const double* theta, const double* p4, const uint8_t* node_mask,
                                int32_t batch, double* workspace, const int32_t* sel, const double* g_lat00,
                                const double* g_lat11, double* gtheta, double* scratch, double l1_lambda,
                                double* loss_accumulate, void* stream);
/* The encoder adjoints with the gradient with respect to the jets.  Arguments as lgae_encoder_backward /
 * lgae_encoder_backward_tiled, plus g_p4 (B,N,4), overwritten with dL/dp4 of the caller's unscaled p4, and gp_scratch
 * (lgae_encoder_input_grad_scratch_doubles(d, batch) doubles).  g_p4 == NULL: exactly the entry point without _p4 (gp_scratch
 * unused).  The parameter gradient is bit-identical either way.  dL/dp4 gathers the input map (mass scalar and canonical vector),
 * the edge features R_ij canon(p_i - p_j) and the pair norms of the radial functions of every level; min / max selections are
 * constants.  Where p^2 == 0 exactly (zero-momentum padding) the mass scalar's term, 0 * inf in the reference, is dropped, so
 * every particle gets a finite gradient (DESIGN.md section 4e).  Deterministic, no atomics. */
int lgae_encoder_backward_p4(const LgaeModelDesc* d, const double* theta, const double* p4, const uint8_t* node_mask,
                             int32_t batch, double* workspace, const int32_t* sel, const double* g_lat00,
                             const double* g_lat11, double* gtheta, double* partials, double l1_lambda,
                             double* loss_accumulate, double* g_p4, double* gp_scratch, void* stream);
int lgae_encoder_backward_tiled_p4(const LgaeModelDesc* d, const double* theta, const double* p4, const uint8_t* node_mask,
                                   int32_t batch, double* workspace, const int32_t* sel, const double* g_lat00,
                                   const double* g_lat11, double* gtheta, double* scratch, double l1_lambda,
                                   double* loss_accumulate, double* g_p4, double* gp_scratch, void* stream);
/* Doubles of gp_scratch: B*N*4, plus B*N*Cmax*20 at N <= 32.  -1 for bad arguments (including a decoder descriptor), -2
 * (LGAE_E_UNSUPPORTED) where the adjoint matching N (per-lane at N <= 32, tiled above) or the input-gradient kernels refuse the
 * configuration.  Needs no GPU. */
int64_t lgae_encoder_input_grad_scratch_doubles(const LgaeModelDesc* d, int32_t batch);
/* LGNDecoder.forward.  lat11 (2,B,1,tau_v,4) planar complex Cartesian.  recon (2,B,N,4); gen00 (2,B,N,1,1) or NULL
 * (NULL: the output scalars are not wanted, the last level's scalar MLP -- which feeds only them -- is then not run;
 * pass g_gen00 = NULL to the backward accordingly). */
int lgae_decoder_forward(const LgaeModelDesc* d, const double* theta, const double* lat11, int32_t batch,
                         double* workspace, double* recon, double* gen00, void* stream);
/* g_recon (2,B,N,4); g_gen00 (2,B,N,1,1) or NULL.  g_lat11 (2,B,1,tau_v,4) receives the latent gradient.  Needs N <= 32 (any N:
 * the tiled entry point); LGAE_E_UNSUPPORTED before any launch otherwise. */
int lgae_decoder_backward(const LgaeModelDesc* d, const double* theta, const double* lat11, int32_t batch,
                          double* workspace, const double* g_recon, const double* g_gen00, double* g_lat11,
                          double* gtheta, double* partials, double l1_lambda, double* loss_accumulate, void* stream);
/* The same adjoint for any N >= 1, with `scratch` (lgae_backward_tiled_scratch_doubles) in place of `partials`; g_lat11
 * receives the latent gradient.  The closed-form level adjoint runs one CTA per jet over its blocks of 32 particles. */
int lgae_decoder_backward_tiled(const LgaeModelDesc* d, const double* theta, const double* lat11, int32_t batch,
                                double* workspace, const double* g_recon, const double* g_gen00, double* g_lat11,
                                double* gtheta, double* scratch, double l1_lambda, double* loss_accumulate, void* stream);

/* ---- the whole training step ---------------------------------------------------------------------- */
/* utils/train.py:283-327 in one call: [normalize_p4] -> encoder -> decoder -> chamfer (sum over the batch) of get_real(recon) +
 * l1_lambda (|theta_enc|_1 + |theta_dec|_1) -> decoder adjoint -> encoder adjoint.  The parameter gradients of both models
 * land in ONE bucket `gtheta`: encoder at [0, enc->n_params), decoder at [gtheta_dec_offset, + dec->n_params) (so a single
 * all-reduce exchanges them), produced by one gradient-init and one reduce launch for both models.  p4_in (B,N,4); when
 * normalize != 0 the normalised jets go to p4 and the per-jet factors to norm_factor (B), otherwise p4 / norm_factor are
 * unused.  loss (1) is overwritten; jet_loss (B) gets the per-jet chamfer distances; recon / g_recon (2,B,N,4), lat00, lat11,
 * sel, g_lat11 as in the model entry points.  partials: lgae_train_step_partials_doubles(enc, dec, batch) doubles.  Needs
 * N <= 32 (LGAE_E_UNSUPPORTED before any launch otherwise; any N: lgae_train_step_tiled below). */
int64_t lgae_train_step_partials_doubles(const LgaeModelDesc* enc, const LgaeModelDesc* dec, int32_t batch);
int lgae_train_step(const LgaeModelDesc* enc, const LgaeModelDesc* dec, const double* theta_enc, const double* theta_dec,
                    const double* p4_in, const uint8_t* node_mask, int32_t batch, int32_t normalize, double* p4,
                    double* norm_factor, double* ws_enc, double* ws_dec, double* lat00, double* lat11, int32_t* sel,
                    double* recon, double* g_recon, double* g_lat11, double* jet_loss, double* loss, double* gtheta,
                    int64_t gtheta_dec_offset, double* partials, double l1_lambda, int32_t get_real, int32_t phase, void* stream);
/* The same step from HOST memory: host_p4 (B,N,4) [and host_mask (B,N), may be NULL] in pinned memory are copied to the
 * device buffers p4_in / node_mask at the start of the step and the loss (1 double) back to host_loss at its end, all on
 * `stream` and capturable in one CUDA graph; the copies are ordered so that the step's parameter-only kernels (weight
 * packing, gradient init) overlap the host-to-device transfer.  The caller synchronises the stream before reading
 * host_loss.  (The end-to-end form of the reference's loop body, utils/train.py:283-327, including its .to(device) and
 * .item().) */
int lgae_train_step_host(const LgaeModelDesc* enc, const LgaeModelDesc* dec, const double* theta_enc,
                         const double* theta_dec, const double* host_p4, const uint8_t* host_mask, double* host_loss,
                         double* p4_in, uint8_t* node_mask, int32_t batch, int32_t normalize, double* p4,
                         double* norm_factor, double* ws_enc, double* ws_dec, double* lat00, double* lat11, int32_t* sel,
                         double* recon, double* g_recon, double* g_lat11, double* jet_loss, double* loss, double* gtheta,
                         int64_t gtheta_dec_offset, double* partials, double l1_lambda, int32_t get_real, int32_t phase, void* stream);
/* The training step with the tiled adjoints (lgae_encoder_backward_tiled / lgae_decoder_backward_tiled) for any N >= 1, e.g. padded
 * 150-particle jets.  Arguments, phases, streams and results as lgae_train_step / lgae_train_step_host, with `scratch` in place of
 * `partials`: lgae_train_step_tiled_scratch_doubles(enc, dec, batch) doubles holding the adjoints of the neighbour sums (one
 * region for both models, B*N*Cmax*10 complex), the encoder's dL/dR of one level (B * ceil(N/32) * N * C * 128 doubles: 1.57 GB at
 * B = 512, N = 150, C = 4) and the rows of parameter-gradient partials.  The size query returns -1 for bad arguments and -2
 * (LGAE_E_UNSUPPORTED) where either model's tiled adjoint or one of the step's fused glue kernels does not fit its shared memory;
 * it needs no GPU, and the step then fails with LGAE_E_UNSUPPORTED before launching anything.  At N <= 32 the tiled step also
 * runs: the forward then still writes the saved radial weights, which the tiled adjoint does not read, and the forward results
 * are bit-identical to lgae_train_step's. */
int64_t lgae_train_step_tiled_scratch_doubles(const LgaeModelDesc* enc, const LgaeModelDesc* dec, int32_t batch);
int lgae_train_step_tiled(const LgaeModelDesc* enc, const LgaeModelDesc* dec, const double* theta_enc, const double* theta_dec,
                          const double* p4_in, const uint8_t* node_mask, int32_t batch, int32_t normalize, double* p4,
                          double* norm_factor, double* ws_enc, double* ws_dec, double* lat00, double* lat11, int32_t* sel,
                          double* recon, double* g_recon, double* g_lat11, double* jet_loss, double* loss, double* gtheta,
                          int64_t gtheta_dec_offset, double* scratch, double l1_lambda, int32_t get_real, int32_t phase, void* stream);
int lgae_train_step_tiled_host(const LgaeModelDesc* enc, const LgaeModelDesc* dec, const double* theta_enc,
                               const double* theta_dec, const double* host_p4, const uint8_t* host_mask, double* host_loss,
                               double* p4_in, uint8_t* node_mask, int32_t batch, int32_t normalize, double* p4,
                               double* norm_factor, double* ws_enc, double* ws_dec, double* lat00, double* lat11, int32_t* sel,
                               double* recon, double* g_recon, double* g_lat11, double* jet_loss, double* loss, double* gtheta,
                               int64_t gtheta_dec_offset, double* scratch, double l1_lambda, int32_t get_real, int32_t phase,
                               void* stream);
/* Split step for data-parallel training (`phase` above): phase 0 runs the whole step.  phase 1 runs it up to the point where the
 * DECODER's gradient bucket gtheta[gtheta_dec_offset, ...) is final -- its reduce is the last thing enqueued on the library's
 * auxiliary stream of the current device, which this function returns -- and phase 2 (same thread, same arguments, directly
 * afterwards) runs the encoder adjoint and the encoder bucket's reduce on `stream` and joins the auxiliary stream back.  A caller
 * enqueues the all-reduce of the decoder bucket on the auxiliary stream between the two calls: it then overlaps the encoder
 * adjoint (SURVEY.md section 8(e) describes the exchange; the reference itself is single-process).  Every training step uses
 * the auxiliary stream: if it cannot be created, this function returns NULL, the step fails with LGAE_E_CUDA, and
 * lgae_last_cuda_error says why. */
void* lgae_aux_stream(void);


/* ---- caller-side ops on the hot path ------------------------------------------------------------- */
/* ChamferLoss (sum over the batch) of x = get_real(recon) (LGAE_GET_REAL_*) against target (B,M,4).
 * loss (1 double) is overwritten.  If g_recon != NULL it receives d loss / d recon (2,B,N,4), scaled by
 * *g_loss (device scalar) when g_loss != NULL.  jet_loss (B) optional per-jet loss (anomaly score). */
int lgae_chamfer(const double* recon, const double* target, int32_t batch, int32_t n, int32_t m, int32_t get_real,
                 double* loss, double* jet_loss, const double* g_loss, double* g_recon, void* stream);
/* Per-jet anomaly scores of the Cartesian family (utils/jet_analysis/anomaly_detection.py:251-419) of x = f * get_real(recon)
 * against f * target, both (B,N,4) (recon complex (2,B,N,4)); f = factor[b], or 1 when factor == NULL (the reference scores the
 * un-normalised and the normalised jets).  scores (B,6): [0] chamfer with the Euclidean norm (:498-503), [1] MSE (:473),
 * [2] chamfer with the Minkowski square (:523-527), [3] MSE with the Minkowski metric (:428-437), each averaged over the
 * particles; [4] MSE of the jet momenta (sum over particles, :405), [5] its Minkowski version (:419).  The Hungarian and
 * EMD scores (scipy / energyflow, per jet on the host) are outside the path. */
int lgae_anomaly_scores(const double* recon, const double* target, const double* factor, int32_t batch, int32_t n, int32_t get_real,
                        double* scores, void* stream);
/* normalize_p4(..., 'overall_max') (utils/normalize_p4.py:39-52): out = p4 / (max|p4| + 1e-16) per jet. */
int lgae_normalize_p4(const double* p4, int32_t batch, int32_t n, double* out, double* factor, void* stream);
/* Adjoint of lgae_normalize_p4: g_p4 (B,N,4) overwritten from g_out (B,N,4) and g_factor (B), either may be NULL (zero).  The
 * factor's gradient reaches the maxima as torch's amax adjoint routes it: split evenly between tied particles and, inside a
 * particle, between tied components. */
int lgae_normalize_p4_backward(const double* p4, int32_t batch, int32_t n, const double* g_out, const double* g_factor,
                               double* g_p4, void* stream);
/* d loss / d target (B,M,4) of lgae_chamfer, overwritten, scaled by *g_loss (device scalar) when g_loss != NULL.  Nearest
 * neighbours are chosen as lgae_chamfer chooses them (first index of the minimum). */
int lgae_chamfer_target_grad(const double* recon, const double* target, int32_t batch, int32_t n, int32_t m, int32_t get_real,
                             const double* g_loss, double* g_target, void* stream);
/* L1 regulariser: out[0] (+)= lambda * sum |theta| ; gtheta += lambda * sign(theta)  (lgn_encoder.py:249-250). */
int lgae_l1(const double* theta, int64_t n, double lambda, double* out_accumulate, double* gtheta_accumulate,
            void* stream);

/* ---- stage-level entry points (LGNNodeLevel / CGMLP), node layout --------------------------------- */
/* One LGN level at maxdim 2: radial functions -> edge features -> CG aggregation -> CG self product ->
 * concat -> complex channel mix.  Encoder flavour: p (B,N,4) real Cartesian + node_mask, radial parameters
 * from theta at level `level`.  Decoder flavour: y (B,N,4,2) complex canonical, constant radial weights.
 * s_in (B,N,C,2), v_in (B,N,C,4,2) -> s_pre (B,N,C',2), v_out (B,N,C',4,2), sums (B,N,C,10,2).
 * r_save (encoder, N <= 32, may be NULL): (B,N,C,32,4) copy of the radial weights, required by the adjoint; with more than 32
 * particles pass NULL (the level kernel then evaluates the radial weights tile by tile), a non-NULL r_save returns
 * LGAE_E_UNSUPPORTED. */
int lgae_level_forward(const LgaeModelDesc* d, int32_t level, const double* theta, const double* p_or_y,
                       const uint8_t* node_mask, int32_t batch, const double* s_in, const double* v_in,
                       double* sums, double* r_save, double* s_pre, double* v_out, void* stream);
/* gtheta (n_params) is overwritten: zero except for the parameters of this level.  g_r_scratch (encoder): scratch of
 * B*N*C*128 + B*16*ceil(N(N+1)/32) doubles: dL/dR of the ordered pairs, then the norms of the unordered pairs. */
int lgae_level_backward(const LgaeModelDesc* d, int32_t level, const double* theta, const double* p_or_y,
                        const uint8_t* node_mask, int32_t batch, const double* s_in, const double* v_in,
                        const double* sums, const double* r_save, double* g_r_scratch, const double* g_s_pre,
                        const double* g_v_out, double* g_s_in, double* g_v_in, double* g_y_accumulate, double* gtheta,
                        double* partials, void* stream);
/* CGMLP on rows = batch*N interleaved scalars x (rows, 2C').  acts: (n_hidden, rows, width_padded) saved
 * activations.  y (rows, 2C').  wpack: lgae_mlp_pack_doubles(d, level) doubles (32-byte aligned) that the forward
 * fills with the level's weights in MMA-fragment order and the backward reads. */
int64_t lgae_mlp_pack_doubles(const LgaeModelDesc* d, int32_t level);
int lgae_mlp_forward(const LgaeModelDesc* d, int32_t level, const double* theta, const double* x, int64_t rows,
                     double* wpack, double* acts, double* y, void* stream);
int lgae_mlp_backward(const LgaeModelDesc* d, int32_t level, const double* theta, const double* x, int64_t rows,
                      const double* wpack, const double* acts, const double* g_y, double* g_x, double* gtheta,
                      double* partials, void* stream);

/* ---- layer-level API of the reference, any maxdim --------------------------------------------------------------
 * Clebsch-Gordan product of ONE pair of irreps (k1,n1) x (k2,n2), channel-wise (replaces cg_product /
 * complex_kron_product, lgn/cg_lib/cg_ops.py:135-298, called by CGProduct.forward, cg_ops.py:113-132).
 * z1 (2, rows1, C, d1), z2: planar complex like every GVec part.
 *   n_nbr == 0: point-wise, z2 (2, rows, C, d2), out_o (2, rows, c_total_o, d_o);
 *   n_nbr == N: aggregated, rows = B*N, z1 (2,B,N,C,d1) indexed by the neighbour j, z2 (2,B,N,N,C,d2) indexed (i,j),
 *               out_o[i] = sum_j H_o (z1_j (x) z2_ij)  (cg_ops.py:265-291).
 * The pair writes channels [c_offset, c_offset + C) of every output irrep o (the reference concatenates the pairs'
 * results on the channel axis, cg_ops.py:210-215), so the caller passes the final concatenated tensors.
 * The non-zero CG coefficients H_o[m, a*d2+d] are a term list on the device, given in three orders:
 *   tab  int32: [order 0: by output component | order 1: by a | order 2: by d][n_terms][3] = (component, a, d),
 *               then comp_start[n_comp+1], a_start[d1+1], d_start[d2+1] (first term of every group, per order);
 *   coef fp64:  [3][n_terms] in the same orders.
 * `component` counts over the output irreps of the pair (out_comp0[o] + m). */
#define LGAE_CG_MAX_OUT 16
typedef struct LgaeCgPairDesc {
    int32_t d1, d2;      /* (k1+1)(n1+1), (k2+1)(n2+1) */
    int32_t channels;    /* C, equal in both operands */
    int32_t n_out;       /* output irreps of this pair */
    int32_t n_comp;      /* sum of their dimensions */
    int32_t n_terms;     /* non-zero CG coefficients */
    int32_t out_d[LGAE_CG_MAX_OUT];
    int32_t out_comp0[LGAE_CG_MAX_OUT];
    int32_t out_ctotal[LGAE_CG_MAX_OUT];
    int32_t out_coffset[LGAE_CG_MAX_OUT];
} LgaeCgPairDesc;
int lgae_cg_product_forward(const LgaeCgPairDesc* d, const int32_t* tab, const double* coef, const double* z1,
                            const double* z2, int64_t rows, int32_t n_nbr, double* const* outs, void* stream);
/* Adjoint (autograd of the above).  g_outs: gradients of the concatenated outputs; g_z1 / g_z2 may be NULL;
 * accumulate_*: add to the buffer instead of overwriting it (several pairs share an operand). */
int lgae_cg_product_backward(const LgaeCgPairDesc* d, const int32_t* tab, const double* coef, const double* z1,
                             const double* z2, int64_t rows, int32_t n_nbr, const double* const* g_outs, double* g_z1,
                             double* g_z2, int32_t accumulate_z1, int32_t accumulate_z2, void* stream);
/* All (node irrep, edge irrep) pairs of ONE aggregated cg_product call in one launch: every edge part is read once instead of
 * once per node irrep.  node_parts[p] (2,B,N,C,node_d[p]), edge_parts[q] (2,B,N,N,C,edge_d[q]); the term list addresses the
 * concatenated component axes a_all (over node parts) and d_all (over edge parts):
 *   tab int32: [n_terms][3] = (component, a_all, d_all) sorted by component, then comp_start[n_comp+1], then for every
 *              component (output tensor index, component m inside that irrep, first channel it writes);  coef fp64 [n_terms].
 * Supported when the edge dimensions add up to 1, 4 or 5 (max_zf <= 1); otherwise LGAE_E_UNSUPPORTED (use the per-pair call). */
#define LGAE_CG_MAX_PARTS 8
typedef struct LgaeCgMultiDesc {
    int32_t channels, n_node, n_edge, n_out, n_comp, n_terms;
    int32_t node_d[LGAE_CG_MAX_PARTS], edge_d[LGAE_CG_MAX_PARTS];
    int32_t out_d[LGAE_CG_MAX_OUT], out_ctotal[LGAE_CG_MAX_OUT];
} LgaeCgMultiDesc;
int lgae_cg_aggregate_multi_forward(const LgaeCgMultiDesc* d, const int32_t* tab, const double* coef,
                                    const double* const* node_parts, const double* const* edge_parts, int64_t rows,
                                    int32_t n_nbr, double* const* outs, void* stream);
/* Adjoint of the one-launch aggregate.  tab_b int32: the component of every term with the terms sorted by cell
 * a_all * D2T + d_all (D2T = sum of edge_d), then cell_start[D1T * D2T + 1], then the same [n_comp][3] output map; coef_b in the
 * same order.  g_outs: gradients of the concatenated outputs; g_node[p] / g_edge[q]: gradient buffers (overwritten) or NULL.
 * Node gradients need D1T in {5, 20} with D2T = 5 and N * C <= 256, otherwise LGAE_E_UNSUPPORTED (use the per-pair adjoint). */
int lgae_cg_aggregate_multi_backward(const LgaeCgMultiDesc* d, const int32_t* tab_b, const double* coef_b,
                                     const double* const* node_parts, const double* const* edge_parts, int64_t rows,
                                     int32_t n_nbr, const double* const* g_outs, double* const* g_node,
                                     double* const* g_edge, void* stream);
/* Per-irrep complex channel mixing out[r, co, m] = sum_ci W[co, ci] x[r, ci, m] (replaces mix_zweight_zvec /
 * mix_zweight_zscalar, lgn/g_lib/cplx_lib.py:7-25, called by MixReps.forward, lgn/nn/g_nn.py:95-121).
 * w (2, c_out, c_in), x (2, rows, c_in, d), out (2, rows, c_out, d).  The adjoint needs
 * lgae_mix_partials_doubles(rows, c_in, c_out) doubles of scratch when g_w is requested. */
int64_t lgae_mix_partials_doubles(int64_t rows, int32_t c_in, int32_t c_out);
int lgae_mix_forward(const double* w, const double* x, int64_t rows, int32_t c_in, int32_t c_out, int32_t d, double* out,
                     void* stream);
int lgae_mix_backward(const double* w, const double* x, const double* g_out, int64_t rows, int32_t c_in, int32_t c_out,
                      int32_t d, double* g_x, double* g_w, double* partials, void* stream);

/* Complex scalar x irrep product with channel broadcast, out[e, c, m] = s[e, c] * v[e, c, m] (edge features
 * rad (x) zonal: lgn/models/lgn_cg.py:167 -> g_torch.mul -> mul_zscalar_zirrep, lgn/g_lib/cplx_lib.py:54-72).
 * s (2, edges, cs), v (2, edges, cv, d), out (2, edges, max(cs, cv), d); cs, cv equal or one of them 1. */
int lgae_scalar_irrep_forward(const double* s, const double* v, int64_t edges, int32_t cs, int32_t cv, int32_t d,
                              double* out, void* stream);
int lgae_scalar_irrep_backward(const double* s, const double* v, const double* g_out, int64_t edges, int32_t cs,
                               int32_t cv, int32_t d, double* g_s, double* g_v, void* stream);
/* RadPolyTrig.forward (lgn/nn/position_levels.py:118-209), mix = 'cplx': k2 = 2*num_basis_fn Lorentzian bells
 * b_k / (1 + (c_k x)^2 + 1e-16) + a_k of `edges` scalars x, zeroed where mask[e % n_mask] == 0, then for each of
 * the n_l zonal degrees y_l = W_l bell + bias_l, W_l (n_out, k2).
 *   planar != 0 (Cartesian basis, n_out = 2C): outs[l] is (2, edges, C), entry (o & 1, e, o >> 1);
 *   planar == 0 (canonical basis: x holds the re and im slices, edges = 2*B*N*N): outs[l] is (edges, n_out).
 * w, bias, outs: host arrays of n_l device pointers. */
int lgae_radial_functions_forward(const double* x, const uint8_t* mask, int64_t edges, int64_t n_mask, const double* a,
                                  const double* b, const double* c, int32_t k2, int32_t n_out, int32_t n_l,
                                  const double* const* w, const double* const* bias, double* const* outs, int32_t planar,
                                  void* stream);
int64_t lgae_radial_functions_partials_doubles(int64_t edges, int32_t k2, int32_t n_out, int32_t n_l);
/* Adjoint.  g_params receives, contiguously: dW [n_l][n_out][k2], dbias [n_l][n_out], da[k2], db[k2], dc[k2];
 * g_x (edges) may be NULL. */
int lgae_radial_functions_backward(const double* x, const uint8_t* mask, int64_t edges, int64_t n_mask, const double* a,
                                   const double* b, const double* c, int32_t k2, int32_t n_out, int32_t n_l,
                                   const double* const* w, const double* const* g_outs, int32_t planar, double* g_x,
                                   double* g_params, double* partials, void* stream);
/* One Linear layer on rows, y = act(x W^T + b), act = LeakyReLU(slope) when leaky_relu != 0 (the CGMLP layers,
 * lgn/models/lgn_levels.py:191-227, for widths outside lgae_mlp_forward).  x (rows, n_in), w (n_out, n_in), b (n_out)
 * or NULL, y (rows, n_out).  The adjoint takes the forward output y for the activation's derivative. */
int lgae_linear_forward(const double* x, const double* w, const double* b, int64_t rows, int32_t n_in, int32_t n_out,
                        int32_t leaky_relu, double slope, double* y, void* stream);
int64_t lgae_linear_partials_doubles(int64_t rows, int32_t n_in, int32_t n_out);
int lgae_linear_backward(const double* x, const double* w, const double* y, const double* g_y, int64_t rows, int32_t n_in,
                         int32_t n_out, int32_t leaky_relu, double slope, double* g_x, double* g_w, double* g_b,
                         double* partials, void* stream);

/* ---- data-parallel gradient exchange over NVLink / NVSwitch peer memory (SURVEY.md section 8(e)) ------------------------------
 * One-shot all-reduce(SUM) of the flat fp64 gradient bucket of a training step across the `world` GPUs of one node, in one
 * kernel: bufs[r] = rank r's bucket (n doubles, 16-byte aligned) and signals[r] = rank r's signal pad (zero-initialised,
 * >= lgae_peer_signal_bytes() bytes), both mapped into this process (symmetric memory; HOST arrays of `world` device pointers).
 * out (n, local) receives sum_r bufs[r] added in rank order, i.e. bit-identical on every rank.  Every rank must make the same
 * call in the same order on its stream; the kernel hand-shakes with the peers before reading and after, so the buckets may be
 * overwritten as soon as it has completed.  multicast != NULL: the address of the buckets' NVSwitch multicast mapping (NVLS);
 * the exchange then runs in place through the switch (multimem.ld_reduce / multimem.st, every rank reduces and broadcasts its
 * 1/world slice) and `out` must be this rank's own bucket bufs[rank].  err_flag (device int32, zero-initialised) is set if a
 * hand-shake timed out.
 * Replaces the ncclAllReduce of the bucket (the reference is single-process: utils/train.py has no exchange at all). */
int64_t lgae_peer_signal_bytes(void);
int lgae_peer_allreduce(const double* const* bufs, uint32_t* const* signals, int32_t rank, int32_t world, int64_t n, double* out,
                        double* multicast, int32_t* err_flag, void* stream);

/* ---- the caller of the hot path: optimizer step ------------------------------------------------------------------
 * torch.optim.Adam (amsgrad = False) on the flat parameter / gradient buffers of up to two models in one launch
 * (replaces optimizer_encoder.step(); optimizer_decoder.step(), utils/train.py:342-343; optimizers built in
 * utils/initialize.py:152-158).  exp_avg / exp_avg_sq: the caller's state buffers (zero-initialised), same sizes as
 * theta.  step_state: TWO int64 on the device, zero-initialised by the caller: [0] = number of updates done (advanced by
 * the kernel, so the call can be replayed inside a CUDA graph), [1] = scratch. */
int lgae_adam_step(double* theta_a, const double* grad_a, double* exp_avg_a, double* exp_avg_sq_a, int64_t n_a,
                   double* theta_b, const double* grad_b, double* exp_avg_b, double* exp_avg_sq_b, int64_t n_b, double lr,
                   double beta1, double beta2, double eps, double weight_decay, int64_t* step_state, void* stream);
/* torch.optim.RMSprop (centered = False), the reference's other optimizer choice (utils/initialize.py:159-165: momentum 0.9):
 * same flat layout; momentum_buf_* may be NULL when momentum == 0. */
int lgae_rmsprop_step(double* theta_a, const double* grad_a, double* square_avg_a, double* momentum_buf_a, int64_t n_a,
                      double* theta_b, const double* grad_b, double* square_avg_b, double* momentum_buf_b, int64_t n_b,
                      double lr, double alpha, double eps, double momentum, double weight_decay, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* LGAE_B200_H */
