/*
 * diffsbdd_b200 — C ABI of the B200-native DiffSBDD denoiser hot path.
 *
 * The reference has no FFI: its "plugin point" is the Python call
 *     EGNNDynamics.forward(xh_atoms, xh_residues, t, mask_atoms, mask_residues)
 * (reference equivariant_diffusion/dynamics.py:87-167) made once per DDPM step from
 * ConditionalDDPM.sample_p_zs_given_zt (conditional_model.py:445) and
 * EnVariationalDiffusion.sample_p_zs_given_zt (en_diffusion.py:503-557).
 * The entry points below are what a ctypes binding of that call needs: plain device pointers and
 * sizes, no torch types.  INTEGRATION.md shows the reference-side stub.
 *
 * All `const float*` / `float*` / `int64_t*` arguments are DEVICE pointers unless stated otherwise.
 * Every function returns 0 on success or a negative dsb_status; dsb_last_error() gives the text.
 * All kernels are launched on the caller's stream; no function synchronises the stream except
 * dsb_dynamics_create/destroy (weight packing) — forward is CUDA-graph capturable.
 */
#ifndef DIFFSBDD_B200_H_
#define DIFFSBDD_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
  DSB_OK = 0,
  DSB_ERR_INVALID_ARGUMENT = -1,
  DSB_ERR_UNSUPPORTED_CONFIG = -2, /* mode 'gnn_dynamics', H not in {64..256 step 64}, tensor-core math modes with sin_embedding */
  DSB_ERR_CUDA = -3,
  DSB_ERR_WORKSPACE_TOO_SMALL = -4
} dsb_status;

/* Constructor arguments of EGNNDynamics (dynamics.py:11-19); same names, C types.
 * Cut-offs: a negative value means "None" (no cut-off for that block, dynamics.py:174-181). */
typedef struct {
  int32_t atom_nf;               /* dynamics.py:11 */
  int32_t residue_nf;
  int32_t n_dims;                /* must be 3 */
  int32_t joint_nf;
  int32_t hidden_nf;
  int32_t n_layers;
  int32_t inv_sublayers;
  int32_t attention;             /* bool */
  int32_t tanh;                  /* bool */
  int32_t condition_time;        /* bool */
  int32_t update_pocket_coords;  /* bool: joint model (dynamics.py:130-132, :161-164) */
  int32_t reflection_equivariant;/* bool: 0 -> cross-product MLP active (egnn_new.py:86-92) */
  int32_t edge_embedding_dim;    /* 0 = None (dynamics.py:51-53) */
  float norm_constant;           /* egnn_new.py:301, :315 */
  float normalization_factor;    /* egnn_new.py:327-328 ('sum' aggregation) */
  float coords_range;            /* 15.0: the undivided value the blocks receive (egnn_new.py:218) */
  float edge_cutoff_ligand;
  float edge_cutoff_pocket;
  float edge_cutoff_interaction;
  int32_t aggregation_mean;      /* bool: aggregation_method == 'mean' (egnn_new.py:330-334: sums divided by the receiver's edge count,
                                  * 1 for a receiver without edges) instead of 'sum' (divided by normalization_factor) */
  int32_t sin_embedding;         /* bool: the two squared distances of an edge enter the MLPs as 2 x 12 sinusoidal features
                                  * (egnn_new.py:282-293); fp32 FFMA kernels only (math mode 0) */
} dsb_config;

typedef struct dsb_dynamics dsb_dynamics; /* opaque: packed weights for one EGNNDynamics module */

/* ---- parameter table: the reference state-dict entries, in the order dsb_dynamics_create wants them.
 * Names are the reference's state_dict keys ("egnn.e_block_0.gcl_0.edge_mlp.0.weight", ...;
 * egnn_new.py:15-29, :78-92, :212-222; dynamics.py:27-53).  cross_product_mlp.4.weight is NOT listed:
 * it aliases coord_mlp.4.weight (egnn_new.py:78, :85, :91). */
int dsb_param_count(const dsb_config* cfg);
/* writes the NUL-terminated key of parameter i into buf; returns its element count, or <0. */
int64_t dsb_param_name(const dsb_config* cfg, int i, char* buf, size_t buflen);

/* ---- module lifetime.  `params[i]` is a device pointer to parameter i (fp32, contiguous, the
 * reference's own [out,in] layout).  The library copies/re-packs them into its own device buffer
 * (k-major GEMM operands, factorised first layers) — the caller's tensors are not referenced after
 * the call returns.  Replaces: EGNNDynamics.__init__ + load_state_dict (dynamics.py:11-85). */
int dsb_dynamics_create(const dsb_config* cfg, const float* const* params, int n_params,
                        dsb_dynamics** out);
void dsb_dynamics_destroy(dsb_dynamics* dyn);

/* Upper bound of directed edges incl. self loops for a batch: sum_g (n_lig_g + n_pocket_g)^2.
 * Host helper (host pointers). */
int64_t dsb_edge_capacity(const int64_t* n_lig_per_graph, const int64_t* n_pocket_per_graph,
                          int n_graphs);

/* Scratch the forward needs (activations, CSR edge list).  The caller owns the buffer (so that a
 * caching allocator / CUDA graph pool can provide it); contents need not be preserved between calls. */
size_t dsb_dynamics_workspace_bytes(const dsb_dynamics* dyn, int64_t n_atoms, int64_t n_residues,
                                    int64_t n_graphs, int64_t edge_capacity);

/* ---- the hot path.  Replaces EGNNDynamics.forward (dynamics.py:87-167), eval mode:
 *   xh_atoms    [n_atoms, 3+atom_nf]      xh_residues [n_residues, 3+residue_nf]   (row-major fp32)
 *   t           [t_numel]; t_numel == n_graphs (one per graph) or 1 (shared, dynamics.py:105-107)
 *   mask_atoms  [n_atoms] int64, mask_residues [n_residues] int64: non-decreasing graph ids in
 *               [0, n_graphs) (utils.py:146-154)
 *   out_atoms   [n_atoms, 3+atom_nf]      out_residues [n_residues, 3+residue_nf]
 *   status      device int32[4]: [0] |= 1 if a NaN reached the coordinate output (the reference raises
 *               ValueError("NaN detected in EGNN output"), dynamics.py:155-159 — the host wrapper
 *               turns the flag into that exception); [1] = number of edges of this call;
 *               [2] |= 1 if the edge list would not fit edge_capacity (outputs invalid); [3] reserved (always 0).
 *               Sticky: the library only ORs into [0] and [2]; the caller clears them.  (3xFP16 mode: an activation
 *               beyond the fp16 range becomes inf and reaches the output as NaN, i.e. flag [0].)
 * Inputs are not modified.  Asynchronous on `stream` (a cudaStream_t passed as void*). */
int dsb_dynamics_forward(dsb_dynamics* dyn,
                         const float* xh_atoms, const float* xh_residues,
                         const float* t, int64_t t_numel,
                         const int64_t* mask_atoms, const int64_t* mask_residues,
                         int64_t n_atoms, int64_t n_residues, int64_t n_graphs,
                         int64_t edge_capacity,
                         float* out_atoms, float* out_residues,
                         void* workspace, size_t workspace_bytes,
                         int32_t* status, void* stream);

/* ---- edge list only.  Replaces EGNNDynamics.get_edges (dynamics.py:169-187): same-graph pairs within
 * the per-block cut-offs, self loops kept, sorted by (row, col).  rows/cols: device int32[edge_capacity];
 * n_edges: device int32[1].  Uses `workspace` (same size contract as forward). */
int dsb_dynamics_edges(dsb_dynamics* dyn,
                       const float* xh_atoms, const float* xh_residues,
                       const int64_t* mask_atoms, const int64_t* mask_residues,
                       int64_t n_atoms, int64_t n_residues, int64_t n_graphs,
                       int64_t edge_capacity,
                       int32_t* rows, int32_t* cols, int32_t* n_edges,
                       void* workspace, size_t workspace_bytes, void* stream);

/* Number of kernel launches (memsets excluded) the last dsb_dynamics_forward on this module enqueued. */
int dsb_dynamics_last_launch_count(const dsb_dynamics* dyn);

/* Process-wide switch for programmatic dependent launch of the forward's kernels (each kernel's launch and prologue
 * overlap its predecessor's tail; every kernel executes griddepcontrol.wait before touching data a predecessor may
 * have written).  enable: 1 on, 0 off, negative = query only.  Returns the previous setting.  Initial value: the
 * environment variable DSB_PDL (default on).  No effect on results. */
int dsb_set_programmatic_launch(int enable);

/* Process-wide selection among equivalent kernel forms of the 3xFP16 path (same results within the parity tolerance).
 * Bit 0: the edge kernels run as CTA pairs (tcgen05 cta_group::2) with the second-layer weights resident in shared memory
 * instead of single CTAs that stream them; bit 1: node_model and the merged first-layer GEMM of a block run as one fused
 * CTA-pair kernel instead of two launches.  Higher bits are ignored.  variants < 0 = query only.  Returns the previous
 * setting.  Initial value: 3, minus bit 0 / 1 if the environment has DSB_EDGE_PAIR=0 / DSB_NODE_BLOCK=0. */
int dsb_set_kernel_variants(int variants);

/* ---- arithmetic path.  mode is a bitmask: 1 = node GEMMs, 2 = edge (GCL) kernel, 4 = coordinate edge kernel run on
 * the tensor pipe (tcgen05.mma, accumulators in TMEM) as 3-product split contractions with fp32 accumulation
 * (x.w ~= x_lo.w_hi + x_hi.w_lo + x_hi.w_hi: fp32-grade accuracy, inside the atol 1e-5 / rtol 1e-4 parity tolerance);
 * 8 selects the operand format of those kernels: 0 = 3xTF32 (kind::tf32, 8-bit exponent, any range),
 * 8 = 3xFP16 (kind::f16: half the shared-memory operand traffic, twice the MMA rate; weights are pre-scaled per matrix
 * with an exact power of two; an activation beyond the fp16 range turns into NaN at the output and raises through
 * status[0]).  0 = fp32 FFMA kernels everywhere.  Only hidden_nf == 256 has tensor-core kernels. */
int dsb_dynamics_set_math_mode(dsb_dynamics* dyn, int mode);

/* ---- measurement hook (bench.py's live roofline).  When enabled, every non-captured forward brackets
 * its launches with CUDA events on the launch stream, grouped into 7 kernel classes:
 *   0 setup (plan, encoders+embedding, edge list)  1 node GEMMs  2 memsets  3 edge_gcl_kernel
 *   4 edge_coord_kernel  5 coord finish/centroid  6 decoders/output.
 * collect() synchronises the recorded events and returns accumulated milliseconds and interval counts per
 * class (host arrays of 7); reset != 0 clears the accumulators. */
int dsb_dynamics_set_profiling(dsb_dynamics* dyn, int enabled);
int dsb_dynamics_collect_profile(dsb_dynamics* dyn, double* ms_by_class, int64_t* count_by_class, int reset);

/* ---- fused DDPM ligand update (one launch). Replaces the element-wise tail of
 * ConditionalDDPM.sample_p_zs_given_zt (conditional_model.py:451-460) + sample_normal_zero_com
 * (:140-160) + remove_mean_batch (:688-696):
 *   mu   = z/alpha_ts[g] - coef1[g] * eps_hat
 *   z'   = mu + sigma[g] * noise ;   com_g = mean over ligand atoms of graph g of z'[:, :3]
 *   z_out[:, :3] = z'[:, :3] - com_g ; z_out[:, 3:] = z'[:, 3:]
 *   pocket_out[:, :3] = pocket[:, :3] - com_g ; pocket_out[:, 3:] = pocket[:, 3:]
 * coef: device fp32 [n_graphs, 3] = (alpha_ts, sigma2_ts/alpha_ts/sigma_t, sigma) per graph (z is DIVIDED by
 * alpha_ts, exactly as conditional_model.py:451 does).
 * In-place allowed (z_out == z, pocket_out == pocket). */
int dsb_ddpm_ligand_update(const float* z_lig, const float* eps_hat, const float* noise,
                           const float* coef, const int64_t* mask_atoms, const int64_t* mask_residues,
                           const float* xh_pocket, int64_t n_atoms, int64_t n_residues,
                           int64_t n_graphs, int32_t atom_nf, int32_t residue_nf,
                           float* z_out, float* xh_pocket_out, void* stream);

/* ---- fused RePaint iteration of ConditionalDDPM.inpaint (one launch; conditional_model.py:636-666), run right after
 * dsb_ddpm_ligand_update, in place on its outputs (z_lig = z_unknown, xh_pocket):
 *   xk      = xh_known, coordinates shifted by (COM(pocket) - com_pocket0[g])                         (:636-640)
 *   z_known = alpha_s xk + sigma_s noise_known ; ligand COM of z_known removed from z_known and pocket   (:162-183)
 *   dx      = COM_fixed(z_unknown) - COM_fixed(z_known) ; z_known.x += dx ; pocket.x += dx               (:645-656)
 *   z       = z_known * fixed + z_unknown * (1 - fixed)                                                  (:659)
 *   if noise_renoise != NULL:  z = alpha_ts z + sigma_ts noise_renoise, ligand COM removed from z and pocket  (:420-430, :662-666)
 * xh_known [n_atoms, 3+atom_nf] (normalised known ligand), com_pocket0 [n_graphs, 3] (pocket COM before sampling),
 * lig_fixed [n_atoms] (0/1 as fp32), coef [n_graphs, 4] = (alpha_s, sigma_s, alpha_{t|s}, sigma_{t|s}). */
int dsb_ddpm_inpaint_update(float* z_lig, float* xh_pocket, const float* xh_known, const float* com_pocket0,
                            const float* lig_fixed, const float* noise_known, const float* noise_renoise,
                            const float* coef, const int64_t* mask_atoms, const int64_t* mask_residues,
                            int64_t n_atoms, int64_t n_residues, int64_t n_graphs, int32_t atom_nf,
                            int32_t residue_nf, void* stream);

/* ---- joint model (EnVariationalDiffusion, update_pocket_coords = 1): the same two fusions for ligand AND pocket.
 * noise_x is ONE tensor [n_atoms + n_residues, 3] (ligand rows first) as sample_center_gravity_zero_gaussian_batch draws it
 * (en_diffusion.py:559-578); its per-graph mean over ligand+pocket nodes is removed inside the kernel (:940-944).
 * dsb_ddpm_joint_update  = tail of EnVariationalDiffusion.sample_p_zs_given_zt (en_diffusion.py:540-557):
 *   z' = z/alpha_ts - coef1 * eps_hat + sigma * eps ; joint COM of z'.x removed.  coef [n_graphs, 3] as dsb_ddpm_ligand_update.
 * dsb_ddpm_joint_inpaint_update = one RePaint iteration of EnVariationalDiffusion.inpaint after that step (:741-807):
 *   z_known = alpha_s xh0 + sigma_s eps ; COM of the fixed nodes aligned noised -> denoised ; blend by lig_fixed / pocket_fixed ;
 *   if renoise_x != NULL: jump back z = alpha_{t|s} z + sigma_{t|s} eps' with the joint COM removed (sample_p_zt_given_zs).
 *   coef [n_graphs, 4] = (alpha_s, sigma_s, alpha_{t|s}, sigma_{t|s}); xh0_* = known data, normalised and centred as :707-717. */
int dsb_ddpm_joint_update(float* z_lig, float* z_pocket, const float* eps_lig, const float* eps_pocket,
                          const float* noise_x, const float* noise_h_lig, const float* noise_h_pocket,
                          const float* coef, const int64_t* mask_atoms, const int64_t* mask_residues,
                          int64_t n_atoms, int64_t n_residues, int64_t n_graphs, int32_t atom_nf,
                          int32_t residue_nf, void* stream);
int dsb_ddpm_joint_inpaint_update(float* z_lig, float* z_pocket, const float* xh0_lig, const float* xh0_pocket,
                                  const float* lig_fixed, const float* pocket_fixed, const float* noise_x,
                                  const float* noise_h_lig, const float* noise_h_pocket, const float* renoise_x,
                                  const float* renoise_h_lig, const float* renoise_h_pocket, const float* coef,
                                  const int64_t* mask_atoms, const int64_t* mask_residues, int64_t n_atoms,
                                  int64_t n_residues, int64_t n_graphs, int32_t atom_nf, int32_t residue_nf,
                                  void* stream);

const char* dsb_last_error(void);
const char* dsb_version(void);

/* ---- diagnostics of the tensor-core kernels (profiles/tc_ablate.py; no reference counterpart).  The product library is
 * built without instrumentation: dsb_debug_set_tc_flags(flags != 0) returns -4 and the counters stay 0.  The instrumented
 * build (-DDSB_TC_INSTRUMENT=1, libdiffsbdd_b200_instr.so) takes a bitmask that disables individual roles of the kernels
 * (results are then garbage) and, with bit 512, accumulates in-kernel clock64 counters that dsb_debug_read_tc_prof copies
 * into out64[64] and clears. */
int dsb_debug_set_tc_flags(int flags);
int dsb_debug_read_tc_prof(unsigned long long* out64);

#ifdef __cplusplus
}
#endif
#endif /* DIFFSBDD_B200_H_ */
