/*
 * foldingdiff_b200 - C ABI of the B200-native reverse-diffusion sampler.
 *
 * This is the drop-in boundary for ONE hot path of microsoft/foldingdiff: the
 * T-step p_sample loop around the BERT-style noise predictor.  The reference has
 * no FFI of its own (it is pure Python); each entry point below names the
 * reference interface it replaces (paths under /root/reference).
 *
 *   fd_create            <- modelling.BertForDiffusionBase.from_dir / __init__
 *                           (foldingdiff/modelling.py:239-291, 297-382): owns the weights
 *   fd_set_schedule      <- beta_schedules.compute_alphas as re-evaluated by every p_sample call
 *                           (foldingdiff/sampling.py:42-53, beta_schedules.py:45-62) + the
 *                           GaussianFourierProjection of every t (modelling.py:59-71)
 *   fd_set_batch         <- the per-batch attention-mask construction in
 *                           sampling.p_sample (foldingdiff/sampling.py:55-58)
 *   fd_forward           <- BertForDiffusionBase.forward (foldingdiff/modelling.py:384-484)
 *                           + transformers==4.11.3 BertEncoder (call site :473-480)
 *   fd_p_sample_steps    <- sampling.p_sample + the body of sampling.p_sample_loop
 *                           (foldingdiff/sampling.py:28-75, 102-131) and the inner loop of
 *                           sampling.get_reconstruction_error (:319-330)
 *   fd_p_sample_steps_philox  same steps, normals drawn inside the step kernel from the library's
 *                           counter-based stream (the throughput mode of SURVEY.md section 8b: no
 *                           per-step host work at all; NOT torch's stream)
 *   fd_sample_host       <- sampling.p_sample_loop as called with host tensors
 *                           (foldingdiff/sampling.py:79-132): host in, host out
 *   fd_destroy           <- (garbage collection of the nn.Module)
 *
 * Conventions
 *   - plain C: pointers, sizes, int status codes (0 = FD_OK).  No C++ exceptions and no
 *     torch types cross this boundary.  fd_last_error() returns a per-thread message for
 *     the last non-zero status.
 *   - all tensors are contiguous fp32, row-major.  Angles are (B, N, F) like the
 *     reference's `x`; lengths / timesteps are int32.
 *   - *_dev pointers are device pointers on the handle's device; work is enqueued on the
 *     given CUDA stream (a cudaStream_t passed as void*; NULL = legacy default stream) and
 *     the call returns without synchronising.  fd_sample_host synchronises.
 *   - a handle is bound to one device and is not re-entrant: one in-flight call per handle.
 *     Every entry point restores the caller's current CUDA device before it returns.
 *   - asynchronous failures: the tensor-core pipelines never spin forever - a bounded wait that
 *     expires (possible on a preempted / time-sliced GPU) ends the kernel and raises a
 *     device-side flag.  fd_forward / fd_p_sample_steps* copy that flag to the host behind
 *     their kernels; it is reported as FD_ERR_CUDA by the NEXT compute call on the handle, by
 *     fd_sample_host before it returns, and by fd_status() - call fd_status() after
 *     synchronising the stream and before trusting the results of an asynchronous call.
 *   - there is NO CPU fallback: every compute entry point returns FD_ERR_CUDA if no
 *     sm_100 device is usable.
 */
#ifndef FOLDINGDIFF_B200_H
#define FOLDINGDIFF_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FD_ABI_VERSION 2

enum {
  FD_OK = 0,
  FD_ERR_INVALID = 1, /* bad argument / shape */
  FD_ERR_CUDA = 2,    /* CUDA runtime error, or no usable device */
  FD_ERR_STATE = 3,   /* call order (e.g. no batch set) */
  FD_ERR_UNSUPPORTED = 4
};

/* GEMM arithmetic of the dense projections. */
enum {
  FD_GEMM_FP32_SIMT = 0, /* CUDA-core fp32 FMA: the in-GPU reference arithmetic          */
  FD_GEMM_TC_3X = 1,     /* tcgen05 tensor cores, error-compensated 3-pass split (parity)  */
  FD_GEMM_TC_1X = 2      /* tcgen05 tensor cores, single pass bf16 (throughput mode; does
                            NOT meet the 1e-4 parity gate - opt-in only)                   */
};

typedef struct fd_handle fd_handle;

/* Model dimensions: HF config.json + training_args.json of the reference model dir. */
typedef struct fd_dims {
  int32_t hidden;       /* config.hidden_size               (384)  */
  int32_t layers;       /* config.num_hidden_layers         (12)   */
  int32_t heads;        /* config.num_attention_heads       (12); head_dim must be 32 */
  int32_t intermediate; /* config.intermediate_size         (768)  */
  int32_t max_pos;      /* config.max_position_embeddings   (128)  */
  int32_t n_features;   /* len(ft_is_angular)               (6)    */
  int32_t timesteps;    /* training_args["timesteps"]       (1000) */
  float ln_eps;         /* config.layer_norm_eps            (1e-12) */
  float head_ln_eps;    /* AnglesPredictor eps              (1e-12, modelling.py:188) */
} fd_dims;

/*
 * Order of the host weight pointers given to fd_create (fp32, nn.Linear layout [out, in]):
 *   0 inputs_to_hidden_dim.weight (H,F)   1 .bias (H)
 *   2 embeddings.LayerNorm.weight (H)     3 .bias (H)
 *   then per layer l (FD_W_PER_LAYER = 17 entries), prefix encoder.layer.{l}. :
 *     +0 attention.self.query.weight (H,H)   +1 .bias
 *     +2 attention.self.key.weight   (H,H)   +3 .bias
 *     +4 attention.self.value.weight (H,H)   +5 .bias
 *     +6 attention.self.distance_embedding.weight (2*max_pos-1, 32)
 *     +7 attention.output.dense.weight (H,H) +8 .bias
 *     +9 attention.output.LayerNorm.weight   +10 .bias
 *     +11 intermediate.dense.weight (I,H)    +12 .bias
 *     +13 output.dense.weight (H,I)          +14 .bias
 *     +15 output.LayerNorm.weight            +16 .bias
 *   then: token_decoder.dense1.weight (H,H), .bias, token_decoder.layer_norm.weight, .bias,
 *         token_decoder.dense2.weight (F,H), .bias
 */
#define FD_W_HEAD 4
#define FD_W_PER_LAYER 17
#define FD_W_TAIL 6

/* Number of weight tensors fd_create expects for `layers` encoder layers. */
int32_t fd_num_weights(int32_t layers);

/*
 * Build a sampler on CUDA device `device`.  All inputs are HOST pointers; the library
 * copies and packs them.  `time_table` is (timesteps, hidden): row t is the reference's
 * GaussianFourierProjection(t) evaluated by the caller with the reference's exact fp32 op
 * order (modelling.py:69-70) - it is NOT recomputed on the device (sin/cos of ~1e4 rad).
 * `coef` is (timesteps, 4): {1/sqrt(alpha_t), beta_t, sqrt(1-alphabar_t), sqrt(posterior_var_t)}
 * from compute_alphas (beta_schedules.py:45-62, sampling.py:43-53,72).
 */
int32_t fd_create(const fd_dims* dims, const float* const* weights, int32_t n_weights,
                  const float* time_table, const float* coef, int32_t device, int32_t gemm_mode,
                  fd_handle** out);

void fd_destroy(fd_handle* h);

/* Message for the calling thread's last non-FD_OK status ("" if none). */
const char* fd_last_error(void);

/* ABI version and capability string of the loaded library. */
int32_t fd_abi_version(void);
const char* fd_build_info(void);

/*
 * Replace the schedule tables of an existing handle (weights stay resident): the loop may be run
 * with a different number of timesteps / beta schedule than the one given to fd_create
 * (sampling.p_sample_loop takes `timesteps` and `betas` as arguments, sampling.py:79-85).
 * time_table is (timesteps, hidden), coef is (timesteps, 4); both HOST, as for fd_create.
 */
int32_t fd_set_schedule(fd_handle* h, int32_t timesteps, const float* time_table, const float* coef);

/* Change the GEMM arithmetic of an existing handle (re-packs nothing: all formats are
 * prepared at create time). */
int32_t fd_set_gemm_mode(fd_handle* h, int32_t gemm_mode);

/*
 * Describe the batch the next calls operate on.
 *   batch, n_pad : x is (batch, n_pad, F), n_pad <= max_pos
 *   lengths      : HOST int32[batch], 1 <= lengths[b] <= n_pad. Keys >= lengths[b] are
 *                  masked exactly like the reference's additive -10000 (sampling.py:56-58,
 *                  modelling.py:450-452)
 *   all_rows     : 0 = only rows < lengths[b] are computed (sampling: the reference discards
 *                  the rest, sampling.py:201-203); 1 = every row of every chain is computed,
 *                  like the reference forward (padded query rows still see only valid keys)
 *   key_mask     : optional HOST float[batch*n_pad] of {0,1} for non-prefix masks (then
 *                  lengths[b] only bounds the computed rows); NULL = prefix mask from lengths
 * Reallocates the workspace if it has to grow; otherwise cheap.
 */
int32_t fd_set_batch(fd_handle* h, int32_t batch, int32_t n_pad, const int32_t* lengths,
                     int32_t all_rows, const float* key_mask, void* stream);

/*
 * eps_out[b, n, :] = model(x, t)[b, n, :] for computed rows; other rows are written as 0.
 *   x_dev    : (batch, n_pad, F)
 *   temb_dev : (batch, hidden) time embedding per chain (rows of the caller's table)
 */
int32_t fd_forward(fd_handle* h, const float* x_dev, const float* temb_dev, float* eps_out_dev,
                   void* stream);

/*
 * Run reverse steps t = t_hi-1, t_hi-2, ..., t_lo on x in place:
 *     eps = model(x, t);  x = c1_t * (x - beta_t * eps / s_t)  [+ sigma_t * z_t  if t > 0]
 *     x[..., j] = ((x[..., j] + pi) mod 2pi) - pi              if wrap_mask[j]
 *   x_dev       : (batch, n_pad, F) in/out.  Rows >= lengths[b] are left untouched.
 *   noise_dev   : (t_hi - t_lo, batch, n_pad, F) standard normals, slice k is used by the
 *                 k-th executed step (t = t_hi-1-k); the slice of t == 0 is never read.
 *                 The caller draws them (torch.randn_like on the reference's stream,
 *                 sampling.py:73) so that RNG state matches the reference.
 *   history_dev : NULL, or (t_hi - t_lo, batch, n_pad, F): slice k = x after step k
 *                 (the reference's imgs list, sampling.py:131-132)
 *   wrap_mask   : HOST uint8[F]
 * Execution: the first step of a new (batch, arithmetic, x buffer, wrap mask) combination is launched kernel by
 * kernel on `stream`; the step is then captured once into a CUDA graph on a stream the handle owns and every
 * further step is one graph launch (FOLDINGDIFF_B200_GRAPH=0 disables).  The handle's stream is ordered after
 * `stream` on entry and `stream` after it on exit, so the stream contract above holds unchanged.
 */
int32_t fd_p_sample_steps(fd_handle* h, float* x_dev, int32_t t_hi, int32_t t_lo,
                          const float* noise_dev, float* history_dev, const uint8_t* wrap_mask,
                          void* stream);

/*
 * fd_p_sample_steps with the library as the noise source: step k (t = t_hi-1-k) adds
 * sigma_t * z where z[b, n, f] is element  offset + k * batch * n_pad * F + (b * n_pad + n) * F + f
 * of the Philox4x32-10 / Box-Muller stream `seed` - the element fd_randn(seed, offset) writes at
 * that index, so pre-drawing with fd_randn and passing noise_dev gives the same bits.  A caller
 * that splits a chain into windows passes offset = (steps already done) * batch * n_pad * F.
 */
int32_t fd_p_sample_steps_philox(fd_handle* h, float* x_dev, int32_t t_hi, int32_t t_lo, uint64_t seed,
                                 uint64_t offset, float* history_dev, const uint8_t* wrap_mask,
                                 void* stream);

/*
 * Asynchronous-failure check (see Conventions): FD_OK, or FD_ERR_CUDA if a tensor-core pipeline
 * of a previous call on this handle timed out (its results are invalid).  Does not synchronise:
 * call it after synchronising the stream the work was enqueued on.  Reading clears the condition.
 */
int32_t fd_status(fd_handle* h);

/*
 * Host-buffer convenience for non-Python callers: the whole p_sample_loop.
 *   x0_host      : (batch, n_pad, F) initial noise            (HOST, read)
 *   noise_host   : (t_start, batch, n_pad, F) per-step normals (HOST, read) or NULL to have
 *                  the library draw them with its own Philox stream seeded by `seed`
 *   out_host     : full_history ? (t_start, batch, n_pad, F) : (batch, n_pad, F)  (HOST, written)
 * Runs t = t_start-1 .. 0; copies in, computes, copies out, synchronises.
 */
int32_t fd_sample_host(fd_handle* h, int32_t batch, int32_t n_pad, const int32_t* lengths,
                       const float* x0_host, int32_t t_start, const float* noise_host,
                       uint64_t seed, const uint8_t* wrap_mask, int32_t full_history,
                       float* out_host);

/*
 * Batched NeRF (SURVEY.md section 8f, rank 1 "next" row): internal angles -> backbone coordinates.
 * Replaces the per-chain Python loop of nerf.NERFBuilder.cartesian_coords / centered_cartesian_coords
 * (/root/reference/foldingdiff/nerf.py:79-128, place_dihedral :145-204) as called by
 * angles_and_coords.create_new_chain_nerf (/root/reference/foldingdiff/angles_and_coords.py:112-184).
 *   angles_dev     : (batch, n_pad, n_features) fp32, the sampler's output layout
 *   lengths        : HOST int32[batch], residues per chain
 *   columns        : HOST int32[6] = feature index of {phi, psi, omega, tau (N:CA:C), CA:C:1N, C:1N:1CA};
 *                    -1 for a bond angle means the reference's default (109 / 115 / 121 degrees)
 *   center         : 1 = subtract each chain's mean coordinate (the reference's default)
 *   coords_out_dev : (batch, 3 * n_pad, 3) fp32, atoms in N, CA, C order; rows >= 3 * lengths[b] are 0
 * Fixed bond lengths 1.34 / 1.46 / 1.54 A and the 1CRN start frame, like the reference. Synchronises.
 */
int32_t fd_nerf_build(const float* angles_dev, int32_t batch, int32_t n_pad, int32_t n_features,
                      const int32_t* lengths, const int32_t* columns, int32_t center, float* coords_out_dev,
                      void* stream);

/* ---- forward half of the training step (SURVEY.md section 8f, rank 3) ------------------------------------------
 * Device pointers, fp32 unless stated, work enqueued on `stream`, no synchronisation; bad shapes / arguments return
 * FD_ERR_INVALID.  Together with fd_forward they evaluate BertForDiffusion._get_loss_terms
 * (/root/reference/foldingdiff/modelling.py:553-677) on the device.
 *
 * fd_q_sample <- NoisedAnglesDataset.sample_noise + __getitem__ (/root/reference/foldingdiff/datasets.py:772-799,
 *   :801-886), for a whole batch:
 *     known_noise = scale_f * z,                              wrapped into [-pi, pi) where angular[f]
 *     corrupted   = sqrt_abar_b * x0 + sqrt_1m_abar_b * known_noise,   wrapped where angular[f]
 *   in torch's fp32 op order, bit-identical to the host mirror given the same z.
 *     x0_dev (batch, n_pad, F); sqrt_abar_dev / sqrt_1m_abar_dev (batch); var_scale HOST float[F]; angular HOST
 *     uint8[F]; z_dev (batch, n_pad, F) standard normals, or NULL: element i = (b * n_pad + n) * F + f then is element
 *     offset + i of the library's Philox stream `seed` (what fd_randn(seed, offset) writes at index i).
 */
int32_t fd_q_sample(const float* x0_dev, int32_t batch, int32_t n_pad, int32_t n_features, const float* sqrt_abar_dev,
                    const float* sqrt_1m_abar_dev, const float* var_scale, const uint8_t* angular, const float* z_dev,
                    uint64_t seed, uint64_t offset, float* known_noise_dev, float* corrupted_dev, void* stream);

/* Loss kinds of fd_loss_terms (BertForDiffusion's `loss` argument, modelling.py:224-237). */
enum {
  FD_LOSS_SMOOTH_L1 = 0, /* angular: radian_smooth_l1_loss, beta = pi/10; other: F.smooth_l1_loss (beta = 1) */
  FD_LOSS_L1 = 1         /* angular: radian_l1_loss;                       other: F.l1_loss                  */
};

/*
 * fd_loss_terms <- the per-feature loop of _get_loss_terms (modelling.py:571-604, losses.py:12-62): terms_dev[f] =
 * mean over the tokens with attn_mask != 0 of the feature-f loss between eps_hat and known_noise, plus
 * circle_penalty * mean(trunc(|eps_hat| / pi)) on angular features when loss == FD_LOSS_SMOOTH_L1.
 *   eps_hat_dev, known_noise_dev (batch, n_pad, F); attn_mask_dev (batch, n_pad); angular HOST uint8[F]
 *   chain_sums_dev (batch, 2F + 1) fp64, written: per chain the loss sums of each feature, the circle sums of each
 *                  feature and the valid-token count (what a per-timestep table is built from)
 *   terms_dev      (F), written
 * Every sum is taken in one fixed order in fp64 (no atomics): two runs give the same bits.
 */
int32_t fd_loss_terms(const float* eps_hat_dev, const float* known_noise_dev, const float* attn_mask_dev, int32_t batch,
                      int32_t n_pad, int32_t n_features, const uint8_t* angular, int32_t loss, float circle_penalty,
                      double* chain_sums_dev, float* terms_dev, void* stream);

/*
 * fd_pdist_loss <- the pairwise-distance branch of _get_loss_terms (modelling.py:616-677, losses.py:66-150):
 *   denoised = (corrupted - sqrt_1m_abar_b * eps_hat) / sqrt_abar_b   (not wrapped, the reference's fp32 op order)
 *   both denoised and known_angles go through the NeRF of fd_nerf_build (uncentred); over the CA atoms of chain b,
 *   pairs i < j < lengths[b]:  loss = sum_b coef_b * sum (|a_i - a_j| - |k_i - k_j|)^2 / (number of pairs in the batch)
 *   known_angles_dev is the batch's "angles": the reference builds the known structure from the zero-centred angles.
 *   corrupted_dev, eps_hat_dev, known_angles_dev (batch, n_pad, F); sqrt_* and coef_dev (batch) fp32
 *   lengths HOST int32[batch] in [1, n_pad]; columns HOST int32[6] as for fd_nerf_build; n_pad <= 128
 *   denoised_dev   (batch, n_pad, F) written, or NULL
 *   chain_sums_dev (batch, 2) fp64 written (weighted squared-difference sum, pair count), or NULL
 *   loss_dev       (1) written
 * Scratch is stream-ordered (cudaMallocAsync / cudaFreeAsync); distances and sums in fp64, fixed order.
 */
int32_t fd_pdist_loss(const float* corrupted_dev, const float* eps_hat_dev, const float* known_angles_dev,
                      const float* sqrt_abar_dev, const float* sqrt_1m_abar_dev, const float* coef_dev, int32_t batch,
                      int32_t n_pad, int32_t n_features, const int32_t* lengths, const int32_t* columns,
                      float* denoised_dev, double* chain_sums_dev, float* loss_dev, void* stream);

/* Fill dst_dev[0..n) with standard normals from the library's Philox4x32-10 stream
 * (seed, offset).  Used by fd_sample_host(noise_host == NULL) and the throughput mode. */
int32_t fd_randn(float* dst_dev, int64_t n, uint64_t seed, uint64_t offset, void* stream);

/* Number of kernels this handle has launched since creation (bench's gpu_launches). */
int64_t fd_launch_count(const fd_handle* h);

/*
 * Built-in kernel timer (used by bench.py for the roofline figures).  Between begin and end every
 * kernel launch of this handle is bracketed by a CUDA-event pair on its launch stream; end
 * synchronises and returns, per kernel category, the summed device time in ms and the launch count
 * (arrays of fd_profile_num_categories() entries; names from fd_profile_category_name).
 */
int32_t fd_profile_begin(fd_handle* h);
int32_t fd_profile_end(fd_handle* h, float* ms_out, int64_t* launches_out);
int32_t fd_profile_num_categories(void);
const char* fd_profile_category_name(int32_t i);

/* Debug / test hooks: run one projection  C = A * W^T (+bias)  with the given arithmetic.
 * A (rows, k), W (n, k), bias (n) or NULL, C (rows, n); all device fp32; rows % 128 == 0. */
int32_t fd_debug_gemm(int32_t gemm_mode, const float* a_dev, const float* w_dev,
                      const float* bias_dev, float* c_dev, int32_t rows, int32_t n, int32_t k,
                      void* stream);

/* Debug / test hook: one relative-key attention layer in isolation.  qkv_dev is packed rows x 3H fp32
 * (q | k | v, rows of chain b start at sum of the computed rows before it), dist_dev the (255, 32)
 * distance embedding, ctx_out_dev packed rows x H fp32.  mode: FD_GEMM_FP32_SIMT = CUDA-core kernel,
 * FD_GEMM_TC_3X / _1X = mma.sync kernel on fp16 hi / lo planes.  Synchronises. */
int32_t fd_debug_attention(int32_t mode, const float* qkv_dev, int32_t batch, int32_t n_pad,
                           const int32_t* lengths, int32_t all_rows, const float* dist_dev, int32_t heads,
                           float* ctx_out_dev, void* stream);

/* ---- output writers (host only, no device work; SURVEY section 8f rank 2) --------------------------------
 * fd_write_angles_csv_gz: one chain's angle table as the gzip-compressed CSV pandas writes for a float32
 *   DataFrame - replaces `s.to_csv(sampled_angles_folder / f"generated_{i}.csv.gz")`,
 *   /root/reference/bin/sample.py:365-370: header ",name,name,..." , one "row_index,v,v,..." line per residue,
 *   numbers spelled as numpy str(float32).  angles_host is [n_rows][row_stride] fp32, the first n_features
 *   columns of each row are written.  gz_level 0..9 (pandas uses 9; -1 = zlib default).
 * fd_write_backbone_pdb: N / CA / C backbone as PDB v3.3 ATOM records of GLY residues in chain A, occupancy
 *   1.00, B factor 5.00, followed by CONECT records for the inter-residue C-N bonds (what biotite emits for the
 *   reference's bond list) - replaces angles_and_coords.write_coords_to_pdb,
 *   /root/reference/foldingdiff/angles_and_coords.py:187-253.  coords_host is [n_atoms][3] fp32, n_atoms = 3N.
 * fd_write_batch: the per-chain fan-out of bin/sample.py:105-128 (multiprocessing.Pool + pandas / biotite) as
 *   one call: chain i has lengths[i] residues, its angles at angles_host[i][n_pad][n_features] and its
 *   coordinates at coords_host[i][atoms_pad][3]; csv_paths / pdb_paths give one file name per chain and either
 *   may be NULL to skip that output.  Work is spread over n_threads host threads. */
int32_t fd_write_angles_csv_gz(const float* angles_host, int32_t n_rows, int32_t n_features, int32_t row_stride,
                               const char* const* feature_names, const char* path, int32_t gz_level);
int32_t fd_write_backbone_pdb(const float* coords_host, int32_t n_atoms, const char* path);
int32_t fd_write_batch(int32_t n_chains, const float* angles_host, int32_t n_pad, int32_t n_features,
                       const char* const* feature_names, const float* coords_host, int32_t atoms_pad,
                       const int32_t* lengths, const char* const* csv_paths, const char* const* pdb_paths,
                       int32_t n_threads, int32_t gz_level);

/* Debug / test hook: synchronise the current device and return (then clear) the tensor-core
 * pipeline error flag: 0 = healthy; 101..104 = a bounded mbarrier wait in the TMA producer /
 * MMA issuer / epilogue timed out (the kernels never spin forever). Negative = CUDA error. */
int32_t fd_debug_tc_status(void);

/* Debug / test hook: 1 = the reverse step of the current batch is being replayed as a CUDA graph (fd_p_sample_steps*
 * capture it after the first step of a window), 0 = not (yet) captured, -1 = a capture failed and the handle stays on
 * kernel-by-kernel launches (FOLDINGDIFF_B200_GRAPH=0 also keeps it at 0). */
int32_t fd_debug_graph_state(const fd_handle* h);

/* Debug / test hook for the tcgen05 attention kernel (FOLDINGDIFF_B200_ATT=tc): while dump_dev is
 * non-NULL every launch also writes, per (chain, head) item and query row, 290 floats
 * {S raw [128], S + relative-key term [128], O unnormalised [32], row max (log2 units), row sum} to
 * dump_dev[(chain * heads + head) * 128 + row]. Pass NULL to switch the dump off again. */
int32_t fd_debug_attention_dump(float* dump_dev);

#ifdef __cplusplus
}
#endif
#endif /* FOLDINGDIFF_B200_H */
