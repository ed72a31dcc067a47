// Inertial fragment matching (IFM) on the device: the tensor math between the two reverse loops of the reference's
// default fragment mode (conformer_generator.py:178-236), which the reference runs in torch on the host:
//   k_ifm_context       ifm_prepare_gen_fragment_context (utils/mol_utils.py:373-457): per-sample moment-of-inertia tensor
//                       of the fragment still to be generated (inverse parallel-axis theorem, :527-550), its 3x3 symmetric
//                       eigen-decomposition (torch.linalg.eigh there; cyclic Jacobi here) and the normalised context
//   k_ifm_merge_inputs  inverse_coord_transform (:508-524) + ifm_prepare_fragments_for_merge (:460-505): z_known and
//                       fixed_mask of the merge loop, built straight from the first loop's device outputs
#pragma once
#include "mlcg_common.cuh"

namespace mlcg {

// One job of a fragment call (mlcg_generate_fragment_jobs): its fixed fragment's rows in the packed ff_x / ff_h and,
// for inertial fragment matching, the per-job part of the moment-of-inertia prologue.  Sample b reads jobs[job[b]].
struct FragJob {
  float moi0[9];   // diag(reference context) - MOI(fixed fragment): the generated fragment's MOI about the origin
  float ffsum[3];  // n_ff * mean(fixed fragment coordinates)
  int n_ff;        // fixed atoms
  int ff_off;      // row of the fragment's first atom in the packed ff_x / ff_h
};

struct IfmNorms {
  float mean[3], mad[3];  // context normalisation (utils/config.py CONTEXT_NORMS), shared by all jobs
};

// Symmetric 3x3 eigen-decomposition, cyclic Jacobi in double precision (converges to machine precision in <= 6 sweeps
// for 3x3).  Eigenvalues ascending (as torch.linalg.eigh), eigenvectors in the columns of v.  An eigenvector is defined
// up to its sign; LAPACK's choice (what the reference gets on the CPU) follows no rule, so the convention is fixed here:
// the component of largest magnitude is positive.
__device__ inline void eigh3(const double a_in[3][3], double w[3], double v[3][3]) {
  double a[3][3];
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) { a[i][j] = a_in[i][j]; v[i][j] = (i == j) ? 1.0 : 0.0; }
  for (int sweep = 0; sweep < 12; ++sweep) {
    const double off = a[0][1] * a[0][1] + a[0][2] * a[0][2] + a[1][2] * a[1][2];
    const double diag = a[0][0] * a[0][0] + a[1][1] * a[1][1] + a[2][2] * a[2][2];
    if (off <= 1e-30 * (diag + 1e-300)) break;
    for (int p = 0; p < 2; ++p)
      for (int q = p + 1; q < 3; ++q) {
        if (a[p][q] == 0.0) continue;
        const double theta = (a[q][q] - a[p][p]) / (2.0 * a[p][q]);
        const double t = (theta >= 0.0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
        const double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
        for (int k = 0; k < 3; ++k) {  // A <- A J
          const double akp = a[k][p], akq = a[k][q];
          a[k][p] = c * akp - s * akq;
          a[k][q] = s * akp + c * akq;
        }
        for (int k = 0; k < 3; ++k) {  // A <- J^T A
          const double apk = a[p][k], aqk = a[q][k];
          a[p][k] = c * apk - s * aqk;
          a[q][k] = s * apk + c * aqk;
        }
        for (int k = 0; k < 3; ++k) {  // V <- V J
          const double vkp = v[k][p], vkq = v[k][q];
          v[k][p] = c * vkp - s * vkq;
          v[k][q] = s * vkp + c * vkq;
        }
      }
  }
  int order[3] = {0, 1, 2};
  for (int i = 0; i < 2; ++i)
    for (int j = 0; j < 2 - i; ++j)
      if (a[order[j]][order[j]] > a[order[j + 1]][order[j + 1]]) { const int t = order[j]; order[j] = order[j + 1]; order[j + 1] = t; }
  double vs[3][3];
  for (int c = 0; c < 3; ++c) {
    w[c] = a[order[c]][order[c]];
    int big = 0;
    for (int k = 1; k < 3; ++k)
      if (fabs(v[k][order[c]]) > fabs(v[big][order[c]])) big = k;
    const double sgn = v[big][order[c]] < 0.0 ? -1.0 : 1.0;
    for (int k = 0; k < 3; ++k) vs[k][c] = sgn * v[k][order[c]];
  }
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) v[i][j] = vs[i][j];
}

// one thread per sample.  n_nodes: total atoms of the sample (fixed + generated); job (B): the sample's entry of `jobs`
// (nullptr: every sample reads jobs[0]).
__global__ void k_ifm_context(const int* __restrict__ n_nodes, const int* __restrict__ job, const FragJob* __restrict__ jobs,
                              int B, IfmNorms nrm, float* __restrict__ ctx_out, float* __restrict__ shift_out,
                              float* __restrict__ rot_out, int* __restrict__ n_gen_out) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const FragJob p = jobs[job ? job[b] : 0];
  const float n_gen = (float)(n_nodes[b] - p.n_ff);
  // shift = (n_ff * mean(ff_x)) / n_gen   (reference :411-412; fp32 as there)
  float s[3];
  for (int c = 0; c < 3; ++c) s[c] = __fdiv_rn(p.ffsum[c], n_gen);
  // shift_moi_to_com_batch (:527-550): I_com = I_origin - m * (|r|^2 E - r r^T)
  const float r2 = __fadd_rn(__fadd_rn(__fmul_rn(s[0], s[0]), __fmul_rn(s[1], s[1])), __fmul_rn(s[2], s[2]));
  double m[3][3];
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) {
      const float term = __fsub_rn((i == j) ? r2 : 0.0f, __fmul_rn(s[i], s[j]));
      m[i][j] = (double)__fsub_rn(p.moi0[i * 3 + j], __fmul_rn(n_gen, term));
    }
  double w[3], v[3][3];
  eigh3(m, w, v);
  for (int c = 0; c < 3; ++c) {
    ctx_out[b * 3 + c] = __fdiv_rn(__fsub_rn((float)w[c], nrm.mean[c]), nrm.mad[c]);
    shift_out[b * 3 + c] = s[c];
    for (int k = 0; k < 3; ++k) rot_out[b * 9 + k * 3 + c] = (float)v[k][c];
  }
  n_gen_out[b] = n_nodes[b] - p.n_ff;
}

// z_known (B,N,11) and fixed_mask (B,N) of the merge loop.  Sample b has the fixed fragment of jobs[job[b]] (nullptr: of
// jobs[0]): n_ff atoms at rows ff_off.. of the packed ff_x / ff_h.  Atom i < n_ff: the fixed fragment (coordinates + raw
// 0/1 one-hot).  Atom n_ff + j (j < Ng, the packed stride of x_gen / cls_gen): generated atom j of the first loop moved
// back to the reference frame, x R^T - shift, with the one-hot of its class.  As in the reference, padded generated rows
// (x = 0) come out as -shift with an all-zero one-hot.
__global__ void k_ifm_merge_inputs(const float* __restrict__ x_gen, const int* __restrict__ cls_gen, const float* __restrict__ shift,
                                   const float* __restrict__ rot, const float* __restrict__ ff_x, const float* __restrict__ ff_h,
                                   const int* __restrict__ job, const FragJob* __restrict__ jobs, int Ng, int N,
                                   float* __restrict__ z_known, float* __restrict__ fixed_mask) {
  const int b = blockIdx.x;
  const int jb = job ? job[b] : 0;
  const int n_ff = jobs[jb].n_ff, ff_off = jobs[jb].ff_off;
  for (int i = threadIdx.x; i < N; i += blockDim.x) {
    float out[ZC];
#pragma unroll
    for (int c = 0; c < ZC; ++c) out[c] = 0.f;
    if (i < n_ff) {
      for (int c = 0; c < 3; ++c) out[c] = ff_x[(size_t)(ff_off + i) * 3 + c];
      for (int c = 0; c < 8; ++c) out[3 + c] = ff_h[(size_t)(ff_off + i) * 8 + c];
    } else if (i - n_ff < Ng) {
      const int j = i - n_ff;
      const float* xg = x_gen + ((size_t)b * Ng + j) * 3;
      const float* R = rot + (size_t)b * 9;
      for (int c = 0; c < 3; ++c) {
        // bmm(coord, R^T)[c] = sum_k coord[k] * R[c][k], accumulated in k order like the reference's matmul
        float acc = __fmul_rn(xg[0], R[c * 3 + 0]);
        acc = fmaf(xg[1], R[c * 3 + 1], acc);
        acc = fmaf(xg[2], R[c * 3 + 2], acc);
        out[c] = __fsub_rn(acc, shift[b * 3 + c]);
      }
      const int cls = cls_gen[(size_t)b * Ng + j];
      if (cls >= 0 && cls < 8) out[3 + cls] = 1.0f;
    }
    float* dst = z_known + ((size_t)b * N + i) * ZC;
#pragma unroll
    for (int c = 0; c < ZC; ++c) dst[c] = out[c];
    fixed_mask[(size_t)b * N + i] = (i < n_ff) ? 1.0f : 0.0f;
  }
}

}  // namespace mlcg
