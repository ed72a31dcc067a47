/* mlcg.h -- C ABI of libmlcg_b200.so: the sm_100a implementation of ml_conformer_generator's data-parallel hot path
 * (batched EDM reverse diffusion with the EGNN denoiser, then the AdjMatSeer bond-order GCN).
 *
 * The reference (Membrizard/ml_conformer_generator) is pure Python/torch and has no FFI layer; its seams for this
 * path are Python call sites.  Each entry point below names the reference call it replaces (file:line relative to the
 * reference root).  INTEGRATION.md shows the ctypes binding a maintainer adds on the reference side.
 *
 * Conventions
 *  - plain pointers and sizes only; no torch types.  Unless a parameter says "host", pointers are DEVICE pointers
 *    owned by the caller; the library never frees caller memory.
 *  - every call enqueues its work on `stream` (a cudaStream_t passed as void*) and returns without synchronising,
 *    except mlcg_generate / mlcg_generate_fragment(_jobs) / mlcg_load_* / mlcg_set_batch which are synchronous.
 *  - return value: 0 = ok, < 0 = argument / state error (see mlcg_last_error), > 0 = cudaError_t.
 *  - one handle per (device, stream); a handle is thread-compatible, not thread-safe.
 *  - layouts are the reference's: z / eps / noise are (B, N, 11) float32 row-major with N = the call's max_n_nodes
 *    (3 coordinates, then 8 atom-class channels); atoms of a sample occupy the first n_nodes[b] slots ("prefix"
 *    node mask, reference utils/mol_utils.py:241-243); padded slots are written as exact zeros.
 *  - there is no CPU fallback: every function fails loudly (MLCG_E_NO_DEVICE) if no sm_100 device is present.
 */
#ifndef MLCG_H_
#define MLCG_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct mlcg_handle mlcg_handle;

/* precision of the EGNN edge / node GEMMs */
enum {
  MLCG_PREC_FP32 = 0, /* exact fp32 SIMT kernels (on-GPU reference mode; edge tensors staged through HBM) */
  MLCG_PREC_TF32 = 1, /* tcgen05 kind::tf32, fp32 accumulate -- parity mode (eps within 1e-3 relative) */
  MLCG_PREC_BF16 = 2, /* tcgen05 kind::f16 (bf16 operands), fp32 accumulate, fp32 residual stream */
  MLCG_PREC_FP16 = 3  /* tcgen05 kind::f16 (fp16 operands: tf32's 10-bit mantissa at bf16's rate), fp32 accumulate, fp32
                         residual stream; every 16-bit quantity carries an exact power-of-two range scale whose inverse is
                         folded into the packed weights -- the fast mode that also meets the tf32 parity numbers */
};

enum {
  MLCG_OK = 0,
  MLCG_E_ARG = -1,       /* bad argument / shape */
  MLCG_E_STATE = -2,     /* weights or batch not set */
  MLCG_E_NO_DEVICE = -3, /* no sm_100 CUDA device: this library has no fallback */
  MLCG_E_WEIGHT = -4     /* missing / mis-shaped state_dict entry */
};

/* One state_dict entry: reference key name, fp32 DEVICE pointer, shape (rows = size(0), cols = numel/size(0)). */
typedef struct {
  const char* name;
  const float* data;
  int rows;
  int cols;
} mlcg_weight_desc;

/* Noise source for one draw of sample_combined_position_feature_noise (equivariant_diffusion.py:341-363).
 * raw != NULL : (B, N, 11) raw N(0,1) draws injected by the caller (parity mode; x-part first, then h-part);
 * raw == NULL : device Philox4x32-10 keyed by (seed, global sample id, atom, draw) -- results do not depend on how a
 *               batch is sharded across GPUs.  The global id of sample b is sample_ids[b] when sample_ids (a DEVICE
 *               array of B int64) is given, else sample_offset + b.  key = {seed lo, seed hi}, counter =
 *               {3*draw + k, atom, id lo, id hi} for k = 0..2: 12 uint32 -> 6 Box-Muller pairs -> 11 normals, so no
 *               two (sample, atom, draw) triples share a random bit (restated on the host in oracle/philox_oracle.py). */
typedef struct {
  const float* raw;
  uint64_t seed;
  uint64_t draw;
  int64_t sample_offset;
  const int64_t* sample_ids;
} mlcg_noise;

/* Scalars of one reverse step, computed on the host exactly as the reference does in float32 torch
 * (equivariant_diffusion.py:224-247, 305-326): z_s = z_t/alpha_ts - c_eps*eps + c_sigma*noise. */
typedef struct {
  float t;        /* (s+1)/T, fed to the denoiser */
  float alpha_ts; /* alpha_{t|s} */
  float c_eps;    /* sigma2_{t|s} / alpha_{t|s} / sigma_t */
  float c_sigma;  /* sigma_{t|s} * sigma_s / sigma_t */
  float alpha_s;  /* forward-diffusion of the fixed fragment (inpaint / merge) */
  float sigma_s;
  float blend;    /* (1 - s/T)^blend_power */
} mlcg_step_scalars;

const char* mlcg_version(void);

/* Replaces: module construction + .to(device) in MLConformerGenerator.__init__ (conformer_generator.py:67-123). */
int mlcg_create(mlcg_handle** out, int device, int precision);
void mlcg_destroy(mlcg_handle* h);
const char* mlcg_last_error(mlcg_handle* h);

/* Replaces: generative_model.load_state_dict(...) (conformer_generator.py:90-95).  Keys: "dynamics.egnn.*" exactly as
 * in EquivariantDiffusion.state_dict(); "gamma.gamma" is ignored (the schedule is rebuilt on the host for the
 * requested step count, conformer_generator.py:104-113).  Repacks / pads / casts once; synchronous. */
int mlcg_load_egnn(mlcg_handle* h, const mlcg_weight_desc* w, int n);
/* Replaces: adj_mat_seer.load_state_dict(...) (conformer_generator.py:97-102). */
int mlcg_load_seer(mlcg_handle* h, const mlcg_weight_desc* w, int n);

/* Replaces: prepare_masks (utils/mol_utils.py:226-252) + EGNNDynamics.get_adj_matrix (egnn.py:515-541): fixes the
 * batch geometry (n_nodes_host[b] atoms in sample b, padded to N slots), builds the edge-tile table and sizes the
 * workspaces.  n_nodes_host is a HOST array.  1 <= n_nodes[b] <= N <= 39. */
int mlcg_set_batch(mlcg_handle* h, const int32_t* n_nodes_host, int B, int N);

/* Replaces: EGNNDynamics.forward (egnn.py:472-513), i.e. `dynamics(t, xh, node_mask, edge_mask, context)`.
 * t: (B) per-sample time; z: (B,N,11); ctx: (B,3) normalised context per sample; eps out: (B,N,11). */
int mlcg_egnn_forward(mlcg_handle* h, const float* t, const float* z, const float* ctx, float* eps, void* stream);

/* Replaces: sample_combined_position_feature_noise as used for the initial latent (equivariant_diffusion.py:384). */
int mlcg_noise_init(mlcg_handle* h, float* z, const mlcg_noise* noise, void* stream);
/* Replaces: the arithmetic of sample_p_zs_given_zt after the network call (equivariant_diffusion.py:320-338). */
int mlcg_step(mlcg_handle* h, float* z, const float* eps, const mlcg_step_scalars* sc, const mlcg_noise* noise,
              void* stream);
/* Replaces: fragment re-injection of inpaint / merge_fragments (equivariant_diffusion.py:473-493, 79-105).
 * z_known: (B,N,11); fixed_mask: (B,N) float 0/1. */
int mlcg_reinject(mlcg_handle* h, float* z, const float* z_known, const float* fixed_mask, const mlcg_step_scalars* sc,
                  const mlcg_noise* noise, void* stream);
/* Replaces: z = alpha*z_known + sigma*eps at diffusion_level (equivariant_diffusion.py:549-559). */
int mlcg_forward_diffuse(mlcg_handle* h, float* z, const float* z_known, float alpha, float sigma,
                         const mlcg_noise* noise, void* stream);
/* Replaces: sample_p_xh_given_z0 after the network call (equivariant_diffusion.py:269-285).
 * x out: (B,N,3); atom_class out: (B,N) int32 in 0..6, -1 for padded slots. */
int mlcg_decode(mlcg_handle* h, const float* z0, const float* eps0, float sigma_0, float alpha_0, float sigma_x,
                const mlcg_noise* noise, float* x, int32_t* atom_class, void* stream);

/* Whole reverse loop on the device.  mode 0 = EquivariantDiffusion.forward (equivariant_diffusion.py:365-421),
 * 1 = .inpaint (:423-513), 2 = .merge_fragments (:515-607).  steps: HOST array of T entries, steps[s] for integer
 * step s (s = T-1 .. 0 are executed; merge skips s > diffusion_level).  ctx: (B,3).  noise_tape: NULL (device
 * Philox, seed; sample_ids: NULL or a DEVICE array of B global sample ids, see mlcg_noise) or (n_draws, B, N, 11) raw
 * draws consumed in the reference's order.  z_work: (B,N,11) scratch that
 * holds z_0 on return.  trace_z / trace_eps: optional (n_forwards, B, N, 11) outputs recording every denoiser
 * input / output (parity tests), or NULL. */
int mlcg_sample(mlcg_handle* h, int mode, int T, const mlcg_step_scalars* steps, int resample_steps,
                int diffusion_level, float merge_alpha, float merge_sigma, float sigma_0, float alpha_0, float sigma_x,
                const float* ctx, const float* z_known, const float* fixed_mask, const float* noise_tape,
                uint64_t seed, int64_t sample_offset, const int64_t* sample_ids, float* z_work, float* x_out,
                int32_t* atom_class_out, float* trace_z, float* trace_eps, void* stream);

/* Replaces (tensor part, declared connectivity rule -- see DESIGN.md): prepare_adj_mat_seer_input
 * (utils/mol_utils.py:159-191).  x: (B,N,3), atom_class: (B,N) -> elements (B,42) int32, dist (B,42,42), adj (B,42,42). */
int mlcg_seer_inputs(mlcg_handle* h, const float* x, const int32_t* atom_class, int32_t* elements, float* dist,
                     float* adj, void* stream);
/* Replaces: AdjMatSeer.forward (adj_mat_seer.py:104-165) + the argmax of redefine_bonds (utils/mol_utils.py:210-211).
 * elements (B,42) int32; dist, adj (B,42,42) incl. +I; logits out (B,42,42,5) or NULL; bonds out (B,42,42) int8 or
 * NULL (lower triangle, zero diagonal).  B here is independent of mlcg_set_batch. */
int mlcg_seer_forward(mlcg_handle* h, const int32_t* elements, const float* dist, const float* adj, float* logits,
                      int8_t* bonds, int B, void* stream);

/* End-to-end call with HOST inputs (what MLConformerGenerator.generate_tensors and the multi-GPU driver use): uploads
 * n_nodes / context / sample ids, runs mlcg_set_batch (only when the geometry changed) + mlcg_sample(mode 0) +
 * mlcg_seer_inputs + mlcg_seer_forward -- replayed as one CUDA graph from the second call with the same geometry on --
 * and copies the results out.  n_nodes_host (B), ctx_host (B,3), sample_ids_host (B int64 global ids, or NULL =
 * sample_offset + b) are HOST arrays.  x_out (B,N,3), atom_class_out (B,N) int32, bonds_out (B,42,42) int8 may be
 * pinned HOST or DEVICE buffers (copied with cudaMemcpyDefault).  Synchronous. */
int mlcg_generate(mlcg_handle* h, const int32_t* n_nodes_host, int B, int N, const float* ctx_host, int T,
                  const mlcg_step_scalars* steps, int resample_steps, float sigma_0, float alpha_0, float sigma_x,
                  uint64_t seed, int64_t sample_offset, const int64_t* sample_ids_host, float* x_out,
                  int32_t* atom_class_out, int8_t* bonds_out, void* stream);

/* The fixed fragment of mlcg_generate_fragment (the reference's `fixed_fragment=`; one fragment per call).  All HOST
 * pointers. */
typedef struct {
  int mode;                          /* 1 = inpainting (EquivariantDiffusion.inpaint, equivariant_diffusion.py:423-513);
                                        2 = inertial fragment matching (inertial_fragment_matching=True, the reference's
                                        default; conformer_generator.py:178-236): a forward loop on the n - n_ff atoms still
                                        to be generated (padded to N - n_ff), the mlcg_ifm_merge_inputs step, then the
                                        merge_fragments loop on the whole molecules */
  int n_ff;                          /* fixed atoms, 1 <= n_ff < min(n_nodes) */
  const float* ff_x_host;            /* (n_ff,3) fragment coordinates */
  const float* ff_h_host;            /* (n_ff,8) raw 0/1 one-hot atom classes */
  int diffusion_level;               /* mode 2: merge_fragments' diffusion_level */
  float merge_alpha, merge_sigma;    /* mode 2: alpha / sigma of that level (mlcg_sample's merge_alpha / merge_sigma) */
  const float* moi_gen_origin_host;  /* mode 2: 3x3, exactly as mlcg_ifm_context takes it */
  const float* ff_weighted_com_host; /* mode 2: 3, exactly as mlcg_ifm_context takes it */
  const float* norm_mean_host;       /* mode 2: 3, CONTEXT_NORMS mean */
  const float* norm_mad_host;        /* mode 2: 3, CONTEXT_NORMS mad */
} mlcg_fragment;

/* Fragment-conditioned counterpart of mlcg_generate: same inputs, outputs, synchronous behaviour and CUDA-graph replay
 * (from the second call with the same key on), plus the fragment.  ctx_host (B,3) is the normalised reference context
 * of every sample.  The device sequence is the eager composition of MLConformerGenerator.edm_sample_tensors followed by
 * the GCN -- mode 1: z_known / fixed_mask from the fragment (prepare_fragment, utils/mol_utils.py:298-342),
 * mlcg_sample(mode 1); mode 2: mlcg_ifm_context on the whole atom counts, mlcg_sample(mode 0) on the atoms still to be
 * generated with the context it wrote, mlcg_ifm_merge_inputs, mlcg_sample(mode 2) -- then mlcg_seer_inputs +
 * mlcg_seer_forward, with the same noise keys and draw numbers; the results equal that composition bit for bit.  The
 * fragment, its prologue, context, sample ids and {seed, sample_offset} are uploaded on every call, so a replay never sees
 * a previous call's inputs, and another fragment or reference context of the same size replays the captured graph.  A
 * call of mlcg_generate and one of mlcg_generate_fragment(_jobs) invalidate each other's graph.  This is the one-job case
 * of mlcg_generate_fragment_jobs.  Returns MLCG_E_ARG for a mode other than 1 or 2, n_ff < 1, n_ff >= min(n_nodes),
 * N - n_ff < 1, a null pointer or weights not loaded. */
int mlcg_generate_fragment(mlcg_handle* h, const mlcg_fragment* frag, const int32_t* n_nodes_host, int B, int N,
                           const float* ctx_host, int T, const mlcg_step_scalars* steps, int resample_steps, float sigma_0,
                           float alpha_0, float sigma_x, uint64_t seed, int64_t sample_offset,
                           const int64_t* sample_ids_host, float* x_out, int32_t* atom_class_out, int8_t* bonds_out,
                           void* stream);

/* Many fragment jobs of one mode in one call of mlcg_generate_fragment_jobs: every job has its own fixed fragment (and,
 * mode 2, its own reference context); the loop settings are shared.  All HOST pointers. */
typedef struct {
  int mode;                          /* 1 = inpainting, 2 = inertial fragment matching (as mlcg_fragment.mode) */
  int n_jobs;                        /* >= 1 */
  const int32_t* job_of_sample_host; /* (B) the job of every sample, 0 <= job < n_jobs */
  const int32_t* n_ff_host;          /* (n_jobs) fixed atoms of every job, 1 <= n_ff[job[b]] < n_nodes[b] */
  const float* ff_x_host;            /* (sum n_ff,3) the jobs' fragment coordinates back to back, in job order */
  const float* ff_h_host;            /* (sum n_ff,8) their raw 0/1 one-hot atom classes, in the same order */
  int diffusion_level;               /* mode 2: merge_fragments' diffusion_level, shared */
  float merge_alpha, merge_sigma;    /* mode 2: alpha / sigma of that level, shared */
  const float* moi_gen_origin_host;  /* mode 2: (n_jobs,3,3), per job as mlcg_ifm_context takes it */
  const float* ff_weighted_com_host; /* mode 2: (n_jobs,3), per job as mlcg_ifm_context takes it */
  const float* norm_mean_host;       /* mode 2: 3, CONTEXT_NORMS mean, shared */
  const float* norm_mad_host;        /* mode 2: 3, CONTEXT_NORMS mad, shared */
} mlcg_fragment_jobs;

/* mlcg_generate_fragment for many jobs at once: sample b runs with the fragment (and, mode 2, the prologue) of job
 * job_of_sample[b]; every other input and output is that of mlcg_generate_fragment.  Mode 2 generates the atoms still to
 * be generated, n_nodes[b] - n_ff[job[b]], padded to N - min(n_ff over the samples).  Every kernel works on each sample
 * alone and the noise is keyed by the global sample id, so a sample's result equals that of a call holding only its own
 * job with the same id, bit for bit.  The graph key is the geometry (mode, B, N, per-sample n_nodes and n_ff, the job
 * count and the packed fragment length) and the shared scalars; the fragments, the job table, the job of every sample,
 * the context, the ids and the seed are uploaded on every call, so other references or fragments of the same sizes
 * replay the captured graph.  Returns MLCG_E_ARG for a mode other than 1 or 2, n_jobs < 1, a job index out of range,
 * n_ff < 1 or N - n_ff < 1 for any job, n_ff[job[b]] >= n_nodes[b] for any sample, a null pointer or weights not
 * loaded. */
int mlcg_generate_fragment_jobs(mlcg_handle* h, const mlcg_fragment_jobs* jobs, const int32_t* n_nodes_host, int B, int N,
                                const float* ctx_host, int T, const mlcg_step_scalars* steps, int resample_steps,
                                float sigma_0, float alpha_0, float sigma_x, uint64_t seed, int64_t sample_offset,
                                const int64_t* sample_ids_host, float* x_out, int32_t* atom_class_out, int8_t* bonds_out,
                                void* stream);

/* ---- Inertial fragment matching (the default fragment mode) between the two reverse loops ---------------------------
 * Replaces: ifm_prepare_gen_fragment_context (utils/mol_utils.py:373-457) after its batch-independent prologue.  The
 * caller computes once, on the host and in float32 as the reference does, moi_gen_origin_host (3x3 row-major) =
 * diag(reference_context) - MOI(fixed fragment) (:396-409) and ff_weighted_com_host (3) = n_ff * mean(fixed fragment
 * coordinates) (:411); norm_mean_host / norm_mad_host (3 each) are CONTEXT_NORMS.  Per sample b (n_nodes[b] = total atoms,
 * DEVICE int32): n_gen = n_nodes - n_ff, shift = ff_weighted_com / n_gen, the inverse parallel-axis shift
 * (shift_moi_to_com_batch, :527-550), the symmetric 3x3 eigen-decomposition (torch.linalg.eigh in the reference; cyclic
 * Jacobi here, eigenvalues ascending, each eigenvector signed so that its largest component is positive -- an eigenvector's
 * sign is the solver's choice) and the normalised context.  Outputs (DEVICE): ctx (B,3), shift (B,3), rot (B,3,3, columns
 * = eigenvectors), n_gen (B) int32. */
int mlcg_ifm_context(mlcg_handle* h, const float* moi_gen_origin_host, const float* ff_weighted_com_host, int n_ff,
                     const float* norm_mean_host, const float* norm_mad_host, const int32_t* n_nodes, int B, float* ctx_out,
                     float* shift_out, float* rot_out, int32_t* n_gen_out, void* stream);
/* Replaces: inverse_coord_transform (utils/mol_utils.py:508-524) + ifm_prepare_fragments_for_merge (:460-505) on the
 * device outputs of the first loop.  x_gen (B,Ng,3), cls_gen (B,Ng) int32 (-1 = padding), shift (B,3), rot (B,3,3),
 * ff_x (n_ff,3), ff_h (n_ff,8) raw 0/1 one-hot -> z_known (B,N,11), fixed_mask (B,N) float; N >= n_ff, atoms beyond
 * n_ff + Ng are zero.  All DEVICE pointers. */
int mlcg_ifm_merge_inputs(mlcg_handle* h, const float* x_gen, const int32_t* cls_gen, const float* shift, const float* rot,
                          const float* ff_x, const float* ff_h, int n_ff, int B, int Ng, int N, float* z_known,
                          float* fixed_mask, void* stream);

/* ---- Gaussian shape similarity (the tensor part of the reference's evaluate_samples) -------------------------------
 * Replaces get_shape_quadrupole_for_molecule (cheminformatics/shape_similarity.py:18-203: clique enumeration :267-311 and
 * the inclusion-exclusion moment series) up to the 3x3 eigen-decomposition, which stays on the host (torch.linalg.eigh,
 * as the reference, :139), and tanimoto_score / rotate_coord (:422-492) for all samples and orientations at once.
 * These entry points use the handle only for its device and error slot; no weights or batch plan are needed. */

/* coords (B,N,3) fp32 device, n_nodes (B) int32 device, 1 <= n_nodes[b] <= 64.  out (B,16) fp32 device:
 * [0] Gaussian volume, [1..3] first moments (relative to the atom mean), [4..12] second-moment tensor about the first
 * moment divided by the volume (row-major 3x3; s_mom_tensor_0 of :126-135), [13..15] atom mean.
 * amplitude / atom_radius / n_terms: the reference's AMPLITUDE 2.70, ATOM_RADIUS 1.60, 6. */
int mlcg_shape_moments(mlcg_handle* h, const float* coords, const int32_t* n_nodes, int B, int N, float amplitude,
                       float atom_radius, int n_terms, float* out, void* stream);

/* Grid Tanimoto of every (sample, orientation) against a reference molecule.
 * ref_pts (n_ref,3): reference atoms in their principal frame; coords (B,N,3), n_nodes (B): raw sample coordinates;
 * frames (B,12): per sample {shift (3), rotation (3x3 row-major)} so that principal = (x - shift) . rotation;
 * orient (n_orient,9): orientation matrices applied as principal . O (entry 0 is ignored: the unrotated frame, as
 * pipeline.py:76); axes (3,G): grid coordinates per axis (Grid of :381-403, built by the caller), G <= 48;
 * workspace: G^3 + 1 floats (reference density and its squared sum).  Outputs: scores (B,n_orient) =
 * sum(f g) / (sum f^2 + sum g^2 - sum(f g)); aligned (B,n_orient,N,3) final coordinates, or NULL. All device pointers. */
int mlcg_shape_tanimoto(mlcg_handle* h, const float* ref_pts, int n_ref, const float* coords, const int32_t* n_nodes, int B,
                        int N, const float* frames, const float* orient, int n_orient, const float* axes, int G,
                        float amplitude, float atom_radius, float* workspace, float* scores, float* aligned, void* stream);

/* Host-only (no device, no handle): the plan of the fused edge kernel for a batch.  tiles_out receives 8 int32 per tile
 * {molecule, rows of the first target that precede the tile, rows, atoms, first target, targets touched, state of the
 * first target, state of the last target} with state -1 = whole, -2 = carried in shared memory between two consecutive
 * tiles of one CTA, >= 0 = side-buffer id (cut between two CTAs); owner_out the CTA (of min(tiles, num_sms) CTAs, paired
 * as the kernel pairs them) that processes each tile; *n_fix_out the number of side-buffer targets.  Returns the number
 * of tiles (at most max_tiles entries are written) or a negative error code. */
int mlcg_plan_edge_tiles(const int32_t* n_nodes_host, int B, int N, int num_sms, int32_t* tiles_out, int32_t* owner_out,
                         int max_tiles, int32_t* n_fix_out);

/* Host-only (no device, no handle): the order in which k_tc_edge3 -- the fused edge kernel of the 16-bit modes -- streams
 * and multiplies the 21 (third of the output channels, K chunk) weight blocks of a tile.  out receives 21 values
 * third * 8 + chunk.  equivariant = 0: GCL sub-layers (third 0, 1, 2, chunks ascending); 1: EquivariantUpdate sub-layers (the
 * second third interleaved with the first while the A operand is generated).  Producer and MMA issuer both follow this
 * table.  Returns 21. */
int mlcg_edge_block_order(int equivariant, int32_t* out);

/* 1 if any mlcg_decode since the last call produced a non-finite coordinate, else 0; clears the flag; synchronises `stream`.
 * A trajectory can diverge (random-init weights in inpaint mode do, in every precision -- the reference's own fp32 path goes
 * NaN too); in MLCG_PREC_FP16 it also happens when pairwise distances exceed ~1.6e4 (pre-activations leave the fp16 range;
 * ordinary molecules stay below 1e2).  The Python host turns this into a RuntimeWarning. */
int mlcg_nonfinite(mlcg_handle* h, void* stream);

/* Introspection for benches / tests. */
int mlcg_num_edge_tiles(mlcg_handle* h);
int64_t mlcg_num_edges(mlcg_handle* h);          /* sum_b n_b (n_b - 1) */
int64_t mlcg_kernel_launches(mlcg_handle* h);    /* kernels launched by this handle since creation */
int64_t mlcg_graph_captures(mlcg_handle* h);     /* CUDA graphs captured by mlcg_generate / mlcg_generate_fragment(_jobs)
                                                    since creation: a replay leaves it unchanged */
/* Times the dominant kernel (the fused edge kernel) with CUDA events on `stream`: runs one sub-layer launch `iters`
 * times on the current batch state and returns the mean milliseconds per launch (< 0 on error). */
float mlcg_time_edge_kernel(mlcg_handle* h, int layer, int iters, void* stream);

/* Measurement: one EGNN forward (same arguments as mlcg_egnn_forward) with a CUDA event after every launch.
 * out_ms[c] = milliseconds in kernel class c: 0 prepare (k_egnn_prepare), 1 P/Q projection GEMMs, 2 fused edge kernel
 * (GCL sub-layers), 3 fused edge kernel (equivariant sub-layers), 4 split-target fix-ups, 5 first node-MLP GEMM,
 * 6 second node-MLP GEMM (residual), 7 readout; out_ms[8] = the whole forward; out_ms[9 + c] = launches of class c.
 * out_ms must hold 17 doubles.  Synchronous. */
int mlcg_egnn_forward_breakdown(mlcg_handle* h, const float* t, const float* z, const float* ctx, float* eps,
                                double* out_ms, void* stream);

/* Diagnostics: mean cycles per 128-row tile spent in each phase of the fused edge kernel for `layer` on the current
 * batch: out[0] row-info + P/Q wait, [1] A generation, [2] MMA tail, [3] epilogue pass 1, [4] pass 2 / coordinate
 * update, [5] A-ring back-pressure (part of [1]), [6] tiles profiled, [7..10] pass-2 sub-phases (wait for the
 * segment-sum MMAs incl. the next tile's early A generation, unused, selector + publish, readout), [11] A-operand
 * hand-off (tcgen05.st + publish, part of [1]).  out must hold 16 doubles.  Synchronous. */
int mlcg_edge_phase_profile(mlcg_handle* h, int layer, double* out, void* stream);

/* Diagnostics: cycle counters of one node-GEMM launch on the current batch, averaged over CTAs.  which: 0 = P/Q projection
 * of layer 0, 1 = first node-MLP GEMM (SiLU epilogue), 2 = second node-MLP GEMM (residual epilogue; adds a second copy of
 * the update to the residual stream -- call it on a scratch state only).  out[0] producer waits for a free ring slot,
 * [1] MMA issuer waits for operands, [2] MMA issuer waits for the epilogue, [3] epilogue waits for the accumulator,
 * [4] epilogue proper, [5] tiles per CTA, [6] CTA lifetime (all but [5] in cycles per CTA), [7] launch ms.  Synchronous. */
int mlcg_gemm_phase_profile(mlcg_handle* h, int which, double* out, void* stream);

/* Test hook: C[M x N] = A[M x K] . W[N x K]^T + bias through the tcgen05 GEMM kernel (row-major fp32 in / out,
 * converted to operand format internally).  mode = MLCG_PREC_TF32, MLCG_PREC_BF16 or MLCG_PREC_FP16; bn = 448 or 256. */
int mlcg_test_gemm(mlcg_handle* h, int mode, int bn, const float* a, const float* w, const float* bias, float* c,
                   int M, int N, int K, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MLCG_H_ */
