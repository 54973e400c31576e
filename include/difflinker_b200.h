/*
 * difflinker_b200 -- C-ABI of the B200-native DiffLinker denoising hot path.
 *
 * The reference (igashov/DiffLinker) is pure Python/PyTorch and has no FFI; the boundary this library
 * replaces is the set of Python call sites listed below (SURVEY.md section 8(b)).  Every entry point is
 * extern "C", takes plain pointers/sizes (no torch types), is stream-ordered and non-blocking unless
 * stated, and returns a dl_status.  One engine per GPU, used from one host thread at a time.
 *
 *   reference interface (file:line)                      entry point here
 *   ---------------------------------------------------  ------------------------------------------
 *   Dynamics.__init__            src/egnn.py:324-372     dl_create / dl_destroy
 *   Dynamics.load_state_dict     (ckpt keys, SURVEY 8b)  dl_set_weight / dl_finalize_weights
 *   Dynamics.forward             src/egnn.py:374-447     dl_dynamics_forward (+ _host)
 *   DynamicsWithPockets.forward  src/egnn.py:471-552     dl_dynamics_forward with graph_type != DL_GRAPH_FC
 *   EDM.sample_chain             src/edm.py:126-176      dl_sample_chain (+ _host)
 *     sample_p_zs_given_zt_only_linker  edm.py:178-208
 *     sample_p_xh_given_z0_only_linker  edm.py:210-235
 *   InpaintingEDM.sample_chain   src/edm.py:549-612      dl_sample_chain with DL_SAMPLER_INPAINT
 *   EDM.forward (evaluation)     src/edm.py:41-124       dl_diffusion_loss
 *   SizeClassifier.forward       src/linker_size_lightning.py:83-110  dl_sizegnn_create/.../dl_sizegnn_forward
 *   build_xae_molecule           src/molecule_builder.py:44-102       dl_bond_orders
 *   frame restore + .xyz text    generate.py:163-171, src/visualizer.py:14-31   dl_restore_frame, dl_format_xyz
 *   utils.FoundNaNException      src/utils.py:274-289    DL_NAN_DETECTED + per-molecule nan_flags
 *
 * Memory: all `const` device pointers are caller-owned and only read; outputs are caller-owned.
 * Floats are fp32, masks int8 exactly as datasets.collate produces them (src/const.py:6-7,
 * src/datasets.py:353-369: edge_mask values are {0,-1,-2}, self-loops live).
 */
#ifndef DIFFLINKER_B200_H_
#define DIFFLINKER_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct dl_engine dl_engine; /* opaque */

typedef enum dl_status {
  DL_OK = 0,
  DL_NAN_DETECTED = 1,        /* dynamics produced NaN: see nan_flags (bit0 = coordinates, bit1 = features) */
  DL_ERR_INVALID = -1,        /* bad argument / unsupported configuration */
  DL_ERR_CUDA = -2,           /* CUDA runtime error; dl_last_error() has the text */
  DL_ERR_WEIGHTS = -3,        /* unknown / missing / wrongly sized weight */
  DL_ERR_UNSUPPORTED = -4
} dl_status;

enum { DL_GRAPH_FC = 0, DL_GRAPH_4A = 1, DL_GRAPH_FC_4A = 2, DL_GRAPH_FC_10A_4A = 3 };
enum { DL_EDGE_AUTO = 0, DL_EDGE_SIMT = 1, DL_EDGE_TCGEN05 = 2 };
enum { DL_SAMPLER_LINKER = 0, DL_SAMPLER_INPAINT = 1 };

/* Mirrors the kwargs of Dynamics.__init__ (src/egnn.py:324-329) that reach the hot path. */
typedef struct dl_config {
  int32_t n_dims;               /* 3 */
  int32_t in_node_nf;           /* F: width of the atom-feature block of xh (one-hot [+ charge]) */
  int32_t context_node_nf;      /* C */
  int32_t hidden_nf;            /* H: must be 128 (every published config, configs/[all].yml `nf: 128`) */
  int32_t n_layers;             /* L equivariant blocks */
  int32_t inv_sublayers;        /* S GCLs per block */
  int32_t condition_time;       /* 0/1 */
  int32_t centering;            /* 0/1 (True only for inpainting models, lightning.py:99) */
  int32_t graph_type;           /* DL_GRAPH_* */
  int32_t device;               /* CUDA ordinal */
  int32_t edge_impl;            /* DL_EDGE_*: AUTO = tcgen05 tensor-core path */
  float norm_constant;          /* EquivariantBlock norm_constant (configs: 1e-6) */
  float normalization_factor;   /* 100 */
} dl_config;

/* Per-reverse-step scalars, computed by the caller with the reference's own formulae
 * (edm.py:369-403) so the device loop reproduces them bit-for-bit. Row r = 0..T-1 is reverse step
 * s = T-1-r; row T is the final p(x,h|z0) step. */
typedef struct dl_step_coef {
  float t;          /* value of the time feature fed to the dynamics ((s+1)/T, or 0 for the last row) */
  float a;          /* rows < T: alpha_{t|s}        ; row T: 1/alpha_0                         */
  float b;          /* rows < T: sigma2_{t|s}/alpha_{t|s}/sigma_t ; row T: sigma_0             */
  float c;          /* rows < T: sigma_{t|s}*sigma_s/sigma_t      ; row T: sigma_x = exp(gamma_0/2) */
  int32_t frame;    /* chain frame this step is the LAST writer of ((s*keep)//T, edm.py:162), or -1 */
  /* inpainting only (edm.py:650-670): q(z_s|z_t,x) on fragment atoms */
  float qa;         /* alpha_{t|s}*sigma_s^2/sigma_t^2 */
  float qb;         /* alpha_s*sigma2_{t|s}/sigma_t^2   */
  float pad;
} dl_step_coef;

const char* dl_version(void);
const char* dl_last_error(void);

dl_status dl_create(const dl_config* cfg, dl_engine** out);
dl_status dl_destroy(dl_engine* e);

/* `name` is the reference state_dict key relative to the Dynamics module, e.g.
 * "dynamics.e_block_0.gcl_1.edge_mlp.2.weight"; `data` is a HOST pointer to fp32 in the reference's
 * own (out,in) row-major layout.  Blocking (copies immediately). */
dl_status dl_set_weight(dl_engine* e, const char* name, const float* data, int64_t numel);
/* Verifies that every parameter of the configured architecture was provided, repacks them for the
 * kernels (k-major fp32 + fp16 hi/lo UMMA tiles) and uploads. Blocking. */
dl_status dl_finalize_weights(dl_engine* e);
/* Number of parameters (floats) the configured architecture expects; for load_state_dict checks. */
int64_t dl_expected_param_count(const dl_engine* e);

/*
 * One Dynamics.forward (egnn.py:374-447 / 471-552). DEVICE pointers.
 *   t          (t_numel) floats, t_numel == B or 1
 *   xh         (B,N,3+F)
 *   node_mask  (B,N) int8
 *   linker_mask (B,N) fp32 or NULL (inpainting, edm.py:505,632)
 *   edge_mask  FC graphs: (B*N*N) int8 or NULL (= all ones); pocket graphs: ignored (edges never cross
 *              molecules here; the reference's batch-id vector egnn.py:557,573 is implied by the layout)
 *   context    (B,N,C) fp32 or NULL when C == 0
 *   out        (B,N,3+F)
 *   nan_flags  (B) int32, written (not accumulated): bit0 NaN in vel, bit1 NaN in h; may be NULL
 * Enqueued on `stream` (a cudaStream_t); returns immediately.
 */
dl_status dl_dynamics_forward(dl_engine* e, int32_t B, int32_t N, const float* t, int32_t t_numel, const float* xh,
                              const int8_t* node_mask, const float* linker_mask, const int8_t* edge_mask,
                              const float* context, float* out, int32_t* nan_flags, void* stream);

/* Same with HOST buffers; copies in, runs, copies out, synchronises; returns DL_NAN_DETECTED if any
 * nan_flags entry is non-zero (nan_flags, if given, is a host array of B int32). */
dl_status dl_dynamics_forward_host(dl_engine* e, int32_t B, int32_t N, const float* t, int32_t t_numel,
                                   const float* xh, const int8_t* node_mask, const float* linker_mask,
                                   const int8_t* edge_mask, const float* context, float* out, int32_t* nan_flags);

/*
 * The whole reverse-diffusion loop (edm.py:126-235), on device, one CUDA-graph replay per step.
 *   xh         (B,N,3+F) normalised input (x/norm0, (h-bias)/norm1), DEVICE
 *   fragment_mask, linker_mask (B,N) fp32 DEVICE; node_mask (B,N) int8; edge_mask, context as above
 *   noise      (T+2,B,N,3+F) UNMASKED standard normal draws, DEVICE: slab 0 initialises the linker,
 *              slab 1+r feeds reverse step r, slab T+1 the final p(x|z0) draw -- i.e. the reference's
 *              torch.randn call order (edm.py:328-345).
 *              DL_SAMPLER_INPAINT (edm.py:549-727): (2T+3,B,N,3+F) PREPARED draws in the order the reference consumes
 *              them -- slab 0 initial z; slabs 1+2r / 2+2r the p(z_s|z_t) (all atoms) and q(z_s|z_t,x) (fragment atoms)
 *              draws of reverse step r; slabs 2T+1 / 2T+2 the final p(x|z0) and q(x|z0,x) draws -- each already
 *              multiplied by its mask with the coordinate part projected to zero centre of mass
 *              (utils.sample_center_gravity_zero_gaussian_with_mask, utils.py:158-168).  The engine must have been
 *              created with centering = 1 (lightning.py:99); all atoms move (the dynamics get linker_mask = NULL),
 *              the latent is re-centred every step (edm.py:592-594) and chain[0] mixes the two final variants by
 *              linker_mask / fragment_mask (edm.py:603-608).
 *   coef       (T+1) dl_step_coef, HOST
 *   norm       {norm_values[0], norm_values[1], norm_biases[1]} HOST (edm.py:347-355)
 *   chain      (keep_frames,B,N,3+F) DEVICE out; chain[0] holds final x and one-hot h (edm.py:174)
 *   nan_flags  (B) int32 DEVICE out: sticky bits as above, OR'ed with (first_nan_row+1)<<8
 * Enqueued on `stream`; the caller synchronises and inspects nan_flags (FoundNaNException mapping).
 */
dl_status dl_sample_chain(dl_engine* e, int32_t sampler, int32_t B, int32_t N, int32_t T, int32_t keep_frames,
                          const float* xh, const int8_t* node_mask, const float* fragment_mask,
                          const float* linker_mask, const int8_t* edge_mask, const float* context,
                          const float* noise, const dl_step_coef* coef, const float* norm, float* chain,
                          int32_t* nan_flags, void* stream);

/* HOST-buffer variant (pinned or pageable): H2D of all inputs incl. noise, loop, D2H of chain and flags,
 * synchronises. Returns DL_NAN_DETECTED if any flag is set. */
/*
 * Same loop with the noise drawn ON THE DEVICE in the reference's stream order (edm.py:328-345, utils.py:189-192): per draw
 * torch.randn(B,N,3) then torch.randn(B,N,F). For a CUDA generator in state (seed, offset) those calls are Philox4x32-10
 * streams with a fixed thread -> element mapping (ATen DistributionTemplates.h); the kernels that consume the noise
 * regenerate exactly those numbers, so the result equals what `dl_sample_chain` returns for the tensor torch would have
 * drawn -- without the tensor ((T+2) B N (3+F) floats: 226 MB for B=256, N=40, T=500), its 2(T+2) launches and its
 * interleaving copy. A plain C caller can sample with nothing but a seed.
 *   seed, offset      the generator state on entry (torch.Generator.initial_seed() / get_offset(); offset % 4 == 0)
 *   offset_consumed   HOST out (may be NULL): what the (T+2) draws consumed -- advance the generator by it
 * DL_SAMPLER_LINKER only (the inpainting sampler needs centre-of-mass projected draws: pass prepared slabs).
 */
dl_status dl_sample_chain_rng(dl_engine* e, int32_t sampler, int32_t B, int32_t N, int32_t T, int32_t keep_frames,
                              const float* xh, const int8_t* node_mask, const float* fragment_mask,
                              const float* linker_mask, const int8_t* edge_mask, const float* context, uint64_t seed,
                              uint64_t offset, uint64_t* offset_consumed, const dl_step_coef* coef, const float* norm,
                              float* chain, int32_t* nan_flags, void* stream);
/* Strong scaling (SURVEY 8(e)): this engine samples molecules [b0, b0 + B) of a batch of B_full. The device-side noise of
 * the following dl_sample_chain_rng / dl_noise_fill calls is then the slice's ROWS of the full-batch draws (and
 * offset_consumed is the full batch's), so the gathered result is bit-identical to the single-GPU run whatever the split.
 * B_full = 0 switches it off. */
dl_status dl_set_noise_slice(dl_engine* e, int32_t B_full, int32_t b0);
/* The (n_draws,B,N,3+F) tensor the device-side stream of dl_sample_chain_rng stands for (tests, debugging). DEVICE out. */
dl_status dl_noise_fill(dl_engine* e, int32_t n_draws, int32_t B, int32_t N, uint64_t seed, uint64_t offset, float* out,
                        uint64_t* offset_consumed, void* stream);

/*
 * The diffusion objective of EDM.forward (edm.py:41-124) for a batch, evaluation only (no backward): what
 * DDPM.validation_step / test_step (lightning.py:228-268) compute through DDPM.forward(data, training=False).
 *   1. q(z_t | x, h) on the linker atoms (edm.py:64-75): z_t = xh*fragment_mask + (alpha_t*xh + sigma_t*eps_t)*linker_mask,
 *      eps_t = [randn(B,N,3), randn(B,N,F)] * linker_mask;
 *   2. one Dynamics.forward(z_t, t) with the per-molecule t (edm.py:78-85), FC or cut-off graph;
 *   3. per molecule, with eps_hat = out * linker_mask, the sums the loss is made of (edm.py:88-124, 244-318, 405-463).
 *   xh          (B,N,3+F) normalised input (x/norm0, (h-bias)/norm1), DEVICE
 *   fragment_mask, linker_mask (B,N) fp32; node_mask (B,N) int8; edge_mask, context as for dl_dynamics_forward. DEVICE
 *   coef        (DL_LOSS_COEFS, B) fp32 DEVICE, row k = coefficient k of every molecule (DL_LOSS_T ...): t = t_int/T, alpha_t,
 *               sigma_t of gamma(t), and alpha, sigma^2 and log(1/sigma) of gamma(1) for kl_prior -- computed by the caller
 *               with the reference's formulas (edm.py:49-62, 251-254), so they round as the reference's do
 *   eps         (B,N,3+F) UNMASKED standard normal draws, DEVICE, or NULL: then they are drawn on the device from (seed, offset)
 *               in the reference's order, randn(B,N,3) then randn(B,N,F), as dl_sample_chain_rng draws one noise sample;
 *               offset_consumed (HOST out, may be NULL) is what those two calls consume
 *   norm        {norm_values[0], norm_values[1], norm_biases[1]} HOST
 *   terms       (B, DL_LOSS_TERMS) fp32 DEVICE out, per molecule: DL_LOSS_ERROR_T = sum (eps_t - eps_hat)^2;
 *               DL_LOSS_NOISE = ||eps_hat||; DL_LOSS_LOG_P_X / DL_LOSS_LOG_P_H = the x and h parts of log p(x,h|z_0)
 *               without constants, evaluated at gamma_t (edm.py:272-318); DL_LOSS_KL_PRIOR = KL(q(z_1|x,h) || N(0,1))
 *               (edm.py:244-270; its h part sums every row, padding included, as the reference does);
 *               DL_LOSS_N_LINKER = number of linker atoms
 *   nan_flags   (B) int32 DEVICE out, as for dl_dynamics_forward
 * Sums are reduced in a fixed order: equal inputs give equal terms. Not for inpainting engines (centering = 1):
 * DL_ERR_UNSUPPORTED. Enqueued on `stream`; returns immediately.
 */
enum { DL_LOSS_T = 0, DL_LOSS_ALPHA_T = 1, DL_LOSS_SIGMA_T = 2, DL_LOSS_ALPHA_1 = 3, DL_LOSS_SIGMA2_1 = 4,
       DL_LOSS_LOG_INV_SIGMA_1 = 5, DL_LOSS_COEFS = 6 };
enum { DL_LOSS_ERROR_T = 0, DL_LOSS_NOISE = 1, DL_LOSS_LOG_P_X = 2, DL_LOSS_LOG_P_H = 3, DL_LOSS_KL_PRIOR = 4,
       DL_LOSS_N_LINKER = 5, DL_LOSS_TERMS = 6 };
dl_status dl_diffusion_loss(dl_engine* e, int32_t B, int32_t N, const float* xh, const int8_t* node_mask,
                            const float* fragment_mask, const float* linker_mask, const int8_t* edge_mask,
                            const float* context, const float* coef, const float* eps, uint64_t seed, uint64_t offset,
                            uint64_t* offset_consumed, const float* norm, float* terms, int32_t* nan_flags, void* stream);

dl_status dl_sample_chain_host(dl_engine* e, int32_t sampler, int32_t B, int32_t N, int32_t T, int32_t keep_frames,
                               const float* xh, const int8_t* node_mask, const float* fragment_mask,
                               const float* linker_mask, const int8_t* edge_mask, const float* context,
                               const float* noise, const dl_step_coef* coef, const float* norm, float* chain,
                               int32_t* nan_flags);

/* Instrumentation for bench.py: kernels launched by this engine since creation, and the device time (ms)
 * of the most recent dl_sample_chain loop / dl_dynamics_forward measured with CUDA events on `stream`
 * (valid after the stream has been synchronised). */
int64_t dl_launch_count(const dl_engine* e);
float dl_last_elapsed_ms(dl_engine* e);
/* Average device time (ms, CUDA events on the engine's loop stream) of the dominant kernel -- the layer-0 GCL
 * edge kernel -- relaunched `reps` times on the engine's current workspace (state of the last call; the
 * caller's mask tensors of that call must still be alive). Blocking. Negative on error. For bench.py's roofline. */
float dl_time_edge_kernel(dl_engine* e, int32_t reps);
/* Cut-off (pocket) graphs, tcgen05 path: what the neighbour-list kernel packed for the most recent forward call --
 * out[0] GCL tile records, out[1] GCL tiles (a row with more than 128 neighbours expands to several), out[2] GCL edges,
 * out[3] coordinate-update records.  All zero for FC graphs.  Blocking (device synchronise). For bench.py / tests. */
dl_status dl_cut_graph_stats(dl_engine* e, int64_t* out);
/* Self-test of the tcgen05 edge-MLP tile against the SIMT path on random data. Blocking.
 * Returns DL_OK and writes the max abs/rel error. */
dl_status dl_selftest_tc(dl_engine* e, float* max_abs_err, float* max_rel_err);
/* Same with the B operand in the MN-major canonical layout (b_mn_major == 1; instruction-descriptor bit 16), or with the
 * A operand in tensor memory (b_mn_major == 2: the TS form the third-generation GCL kernel uses for the stationary W2). */
dl_status dl_selftest_tc_layout(dl_engine* e, int32_t b_mn_major, float* max_abs_err, float* max_rel_err);

/*
 * Output stage (the step right after sample_chain in every generation script).
 *
 * dl_restore_frame -- generate.py:163-171, generate_with_pocket.py:272-280, sample.py:164-171: put the molecules back
 * to the input frame, x += (sum_n positions*com_mask / sum_n com_mask) * node_mask, in place on the first three columns
 * of `xh` (row stride `row_stride` floats: 3 for a packed x, 3+F for chain[0]).  DEVICE buffers, enqueued on `stream`.
 *   positions (B,N,3) fp32; com_mask (B,N) fp32 (fragment_mask or anchors); node_mask (B,N) int8
 */
dl_status dl_restore_frame(int32_t B, int32_t N, int32_t row_stride, float* xh, const float* positions,
                           const float* com_mask, const int8_t* node_mask, void* stream);
/* Same when the sampled batch was re-templated with sampled linker sizes (create_templates_for_linker_generation,
 * datasets.py:483-512): `xh` / `node_mask` have the template's padded length N while `positions` / `com_mask` keep the
 * input batch's padded length N_pos (generate.py:165-171 mixes exactly these two). */
dl_status dl_restore_frame2(int32_t B, int32_t N, int32_t N_pos, int32_t row_stride, float* xh, const float* positions,
                            const float* com_mask, const int8_t* node_mask, void* stream);

/*
 * dl_format_xyz -- visualizer.save_xyz_file (src/visualizer.py:14-31) for a whole batch: the text of the B .xyz files
 * ("%d\n\n" then one "%s %.9f %.9f %.9f\n" line per valid atom, symbol = symbols[argmax one_hot]) written
 * back to back into `out`; molecule b occupies out[offsets[b] .. offsets[b+1]).  HOST buffers.
 *   positions (B,N,>=3) fp32 with row stride pos_row_stride; one_hot (B,N,>=F) fp32 with row stride oh_row_stride
 *   symbols: n_symbols >= F NUL-terminated element symbols (const.IDX2ATOM / GEOM_IDX2ATOM, src/const.py:15,31)
 * Returns the number of bytes the full text needs (write again with a larger buffer if > out_cap; out may be NULL
 * for a sizing call), or a negative dl_status.
 */
int64_t dl_format_xyz(int32_t B, int32_t N, int32_t F, const float* positions, int32_t pos_row_stride,
                      const float* one_hot, int32_t oh_row_stride, const int8_t* node_mask,
                      const char* const* symbols, int32_t n_symbols, char* out, int64_t out_cap, int64_t* offsets);

/*
 * dl_bond_orders -- molecule_builder.build_xae_molecule / get_bond_order (src/molecule_builder.py:44-102) for a padded
 * batch: E[b][i][j] (i > j, both atoms valid) = 0..3 from the pair distance in pm against single / double / triple bond
 * length thresholds (table value + margin, src/const.py:66-146,180) of the type pair ordered by type index; the upper
 * triangle and masked rows are 0.  DEVICE buffers, enqueued on `stream`.
 *   x (B,N,>=3) fp32 with row stride x_row_stride; atom_types (B,N) int32; node_mask (B,N) int8
 *   thr1/thr2/thr3 (n_types,n_types) fp32 indexed [min type][max type]; negative = pair absent from that table
 *   E (B,N,N) int8 out
 */
dl_status dl_bond_orders(int32_t B, int32_t N, int32_t n_types, const float* x, int32_t x_row_stride,
                         const int32_t* atom_types, const int8_t* node_mask, const float* thr1, const float* thr2,
                         const float* thr3, int8_t* E, void* stream);

/*
 * SizeGNN (src/linker_size.py:45-91) as called by SizeClassifier.forward (src/linker_size_lightning.py:83-110): the
 * linker-size classifier that generate.py:88-99 runs once per batch before the sampler.
 *   out[b] = mean_n embedding_out( GCL_L(...GCL_1(embedding_in(one_hot*frag))) )     (B, out_node_nf) logits
 * with ReLU GCLs on the fragment atoms, edges = fragment pairs (self loops included) whose SQUARED distance is < 6
 * (linker_size_lightning.py:107-108), sum aggregation, normalization_factor 1.
 * Weight names: "embedding_in.{weight,bias}", "layer<l>.edge_mlp.{0,2}.{weight,bias}", "layer<l>.node_mlp.{0,2}.{weight,
 * bias}" (l = 0 is SizeGNN.gcl1, l >= 1 is gcl_layers[l-1]; with normalization='batch_norm' the caller folds the eval-mode
 * BatchNorm1d affine maps into node_mlp.0 / node_mlp.2), "embedding_out.{weight,bias}"; (out,in) row-major fp32, HOST.
 */
typedef struct dl_sizegnn dl_sizegnn; /* opaque */
typedef struct dl_sizegnn_config {
  int32_t in_node_nf;   /* one-hot width the network was trained with */
  int32_t hidden_nf;    /* 128 */
  int32_t out_node_nf;  /* number of linker-size classes */
  int32_t n_layers;     /* GCLs (train_size_gnn.py:20: 3) */
  int32_t device;
} dl_sizegnn_config;
dl_status dl_sizegnn_create(const dl_sizegnn_config* cfg, dl_sizegnn** out);
dl_status dl_sizegnn_destroy(dl_sizegnn* e);
dl_status dl_sizegnn_set_weight(dl_sizegnn* e, const char* name, const float* host_data, int64_t numel);
dl_status dl_sizegnn_finalize_weights(dl_sizegnn* e);
/* DEVICE buffers, enqueued on `stream`:
 *   xh            (B,N,3+in_node_nf) fp32: [positions | one_hot] (the kernel applies fragment_mask to both)
 *   fragment_mask (B,N) int8 0/1       (data['fragment_mask'], or 'fragment_only_mask' with pockets)
 *   edge_mask     (B,N,N) int8, non-zero = live pair (datasets.collate_with_fragment_edges, datasets.py:396-402), or NULL
 *   out           (B,out_node_nf) fp32 logits */
dl_status dl_sizegnn_forward(dl_sizegnn* e, int32_t B, int32_t N, const float* xh, const int8_t* fragment_mask,
                             const int8_t* edge_mask, float* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DIFFLINKER_B200_H_ */
