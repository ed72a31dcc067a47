// Gaussian shape similarity of generated conformers against a reference (SURVEY 8f-4): the tensor part of the reference's
// evaluate_samples (cheminformatics/pipeline.py:37-86, cheminformatics/shape_similarity.py).
//
//  k_shape_moments : per molecule, the inclusion-exclusion series (orders 1..6) of Gaussian volume, first and second
//                    moments over all cliques of mutually neighbouring atoms (shape_similarity.py:18-125).  The reference
//                    enumerates the cliques with a recursive Python backtracker and evaluates the series three times
//                    (raw, centred, rotated coordinates); here one depth-first walk with 64-bit neighbour masks carries
//                    the running coordinate sums, every clique costs one exp, and the centred tensor follows from the
//                    raw sums algebraically.
//  k_shape_grid    : Tanimoto overlap of the Gaussian densities on the reference's 40^3 grid (shape_similarity.py:
//                    406-492) for every (sample, orientation).  exp(-a|p-c|^2) is separable, so each block builds three
//                    40 x n tables and a grid point costs two multiplies and an FMA per atom -- no MUFU work.
//
// Both are small next to the generation itself (about a millisecond for 1024 samples x 4 orientations); the point is that
// the reference needs 1.5 - 4 s of CPU per sample for the same numbers.
#pragma once
#include "mlcg_common.cuh"

namespace mlcg {

constexpr int SHAPE_MAX_ATOMS = 64;   // 64-bit neighbour masks
constexpr int SHAPE_MAX_GRID = 48;    // grid points per axis (reference: 40)
constexpr int SHAPE_MAX_TERMS = 6;    // clique order (reference n_terms = 6)

struct ShapeConsts {
  float amplitude, alpha, threshold;
  int n_terms;
  float amp_k[SHAPE_MAX_TERMS + 1];    // amplitude^k
  float vol_k[SHAPE_MAX_TERMS + 1];    // (pi / (k alpha))^(3/2)
  float inv2ka[SHAPE_MAX_TERMS + 1];   // 1 / (2 k alpha)
};

// out[b][16] = {volume, first moment (3), pre-rotation second-moment tensor row-major (9), coordinate mean (3)}
__global__ void __launch_bounds__(128) k_shape_moments(const float* __restrict__ coords, const int* __restrict__ n_nodes, int N,
                                                       const ShapeConsts k, float* __restrict__ out) {
  __shared__ float cx[SHAPE_MAX_ATOMS], cy[SHAPE_MAX_ATOMS], cz[SHAPE_MAX_ATOMS];
  __shared__ unsigned long long adj[SHAPE_MAX_ATOMS];
  __shared__ float mean_s[3];
  __shared__ double red[4][11];
  const int b = blockIdx.x, tid = threadIdx.x;
  const int n = n_nodes[b];
  const float* x = coords + (size_t)b * N * 3;
  if (tid < 3) {  // centre of the atoms (pipeline.py:39-40 / 68-69)
    float s = 0.f;
    for (int i = 0; i < n; ++i) s += x[i * 3 + tid];
    mean_s[tid] = s / (float)n;
  }
  __syncthreads();
  if (tid < n) {
    cx[tid] = x[tid * 3 + 0] - mean_s[0];
    cy[tid] = x[tid * 3 + 1] - mean_s[1];
    cz[tid] = x[tid * 3 + 2] - mean_s[2];
  }
  __syncthreads();
  if (tid < n) {  // neighbours: 0 < distance < threshold (shape_similarity.py:243-257)
    unsigned long long m = 0;
    for (int j = 0; j < n; ++j) {
      const float dx = cx[tid] - cx[j], dy = cy[tid] - cy[j], dz = cz[tid] - cz[j];
      const float d = sqrtf(dx * dx + dy * dy + dz * dz);
      if (d > 0.f && d < k.threshold) m |= 1ull << j;
    }
    adj[tid] = m;
  }
  __syncthreads();

  // accumulators: V, F(3), M2 (xx, yy, zz, xy, xz, yz), K = sum sign * v / (2 k alpha)
  double acc[11];
#pragma unroll
  for (int i = 0; i < 11; ++i) acc[i] = 0.0;
  // one clique of `order` atoms with coordinate sum (sx, sy, sz) and sum of squared norms r2 (shape_similarity.py:206-230)
  auto contrib = [&](int order, float sx, float sy, float sz, float r2) {
    const float inv = 1.0f / (float)order;
    const float gamma = r2 - (sx * sx + sy * sy + sz * sz) * inv;
    const float v = k.amp_k[order] * __expf(-k.alpha * gamma) * k.vol_k[order];
    const double sv = (order & 1) ? (double)v : -(double)v;  // (-1)^(order-1)
    const double px = sx * inv, py = sy * inv, pz = sz * inv;
    acc[0] += sv;
    acc[1] += sv * px; acc[2] += sv * py; acc[3] += sv * pz;
    acc[4] += sv * px * px; acc[5] += sv * py * py; acc[6] += sv * pz * pz;
    acc[7] += sv * px * py; acc[8] += sv * px * pz; acc[9] += sv * py * pz;
    acc[10] += sv * (double)k.inv2ka[order];
  };
  auto above = [](int v) { return v >= 63 ? 0ull : ~((2ull << v) - 1ull); };
  auto n2 = [&](int a) { return cx[a] * cx[a] + cy[a] * cy[a] + cz[a] * cz[a]; };
  for (int i = tid; i < n; i += blockDim.x) contrib(1, cx[i], cy[i], cz[i], n2(i));
  // cliques of order >= 2: one depth-first walk per neighbouring pair (i < j), members in increasing index order
  for (int pr = tid; pr < n * n; pr += blockDim.x) {
    const int i = pr / n, j = pr - i * n;
    if (j <= i || !((adj[i] >> j) & 1ull) || k.n_terms < 2) continue;
    const float s2x = cx[i] + cx[j], s2y = cy[i] + cy[j], s2z = cz[i] + cz[j], r2 = n2(i) + n2(j);
    contrib(2, s2x, s2y, s2z, r2);
    if (k.n_terms < 3) continue;
    unsigned long long m3 = adj[i] & adj[j] & above(j);
    while (m3) {
      const int a = __ffsll((long long)m3) - 1;
      m3 &= m3 - 1;
      const float s3x = s2x + cx[a], s3y = s2y + cy[a], s3z = s2z + cz[a], r3 = r2 + n2(a);
      contrib(3, s3x, s3y, s3z, r3);
      if (k.n_terms < 4) continue;
      unsigned long long m4 = adj[i] & adj[j] & adj[a] & above(a);
      while (m4) {
        const int c = __ffsll((long long)m4) - 1;
        m4 &= m4 - 1;
        const float s4x = s3x + cx[c], s4y = s3y + cy[c], s4z = s3z + cz[c], r4 = r3 + n2(c);
        contrib(4, s4x, s4y, s4z, r4);
        if (k.n_terms < 5) continue;
        unsigned long long m5 = adj[i] & adj[j] & adj[a] & adj[c] & above(c);
        while (m5) {
          const int d = __ffsll((long long)m5) - 1;
          m5 &= m5 - 1;
          const float s5x = s4x + cx[d], s5y = s4y + cy[d], s5z = s4z + cz[d], r5 = r4 + n2(d);
          contrib(5, s5x, s5y, s5z, r5);
          if (k.n_terms < 6) continue;
          unsigned long long m6 = adj[i] & adj[j] & adj[a] & adj[c] & adj[d] & above(d);
          while (m6) {
            const int e = __ffsll((long long)m6) - 1;
            m6 &= m6 - 1;
            contrib(6, s5x + cx[e], s5y + cy[e], s5z + cz[e], r5 + n2(e));
          }
        }
      }
    }
  }
  // block reduction (fixed order: deterministic)
#pragma unroll
  for (int i = 0; i < 11; ++i) {
    double v = acc[i];
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    if ((tid & 31) == 0) red[tid >> 5][i] = v;
  }
  __syncthreads();
  if (tid == 0) {
    double s[11];
    for (int i = 0; i < 11; ++i) s[i] = (red[0][i] + red[1][i]) + (red[2][i] + red[3][i]);
    const double V = s[0];
    const double m[3] = {s[1] / V, s[2] / V, s[3] / V};
    // second moments about the first moment: sum sv (c - m)(c - m)^T = M2 - m F^T, plus the 1/(2 k alpha) diagonal term
    const double xx = s[4] - m[0] * s[1] + s[10], yy = s[5] - m[1] * s[2] + s[10], zz = s[6] - m[2] * s[3] + s[10];
    const double xy = s[7] - m[0] * s[2], xz = s[8] - m[0] * s[3], yz = s[9] - m[1] * s[3];
    float* o = out + (size_t)b * 16;
    o[0] = (float)V;
    o[1] = (float)m[0]; o[2] = (float)m[1]; o[3] = (float)m[2];
    o[4] = (float)(xx / V); o[5] = (float)(xy / V); o[6] = (float)(xz / V);
    o[7] = (float)(xy / V); o[8] = (float)(yy / V); o[9] = (float)(yz / V);
    o[10] = (float)(xz / V); o[11] = (float)(yz / V); o[12] = (float)(zz / V);
    o[13] = mean_s[0]; o[14] = mean_s[1]; o[15] = mean_s[2];
  }
}

// Density overlap on the grid.  block = (sample b, orientation o); final coordinates = ((x - shift_b) . R_b) . O_o.
//  kRef = true : one block, writes the density of the reference molecule to dens[G^3] and sum f^2 to dens[G^3].
//  kRef = false: reads them, writes scores[b][o] = fg / (f2 + gg - fg) and (optionally) the final coordinates.
//  kJobs = true: many references in one launch.  Reference j owns axes + j*3*G and dens + j*(G^3+1).  The reference pass
//  runs one block per reference (b = j, its points at coords + j*N*3, its atom count n_nodes[j]); the sample pass scores
//  sample b against reference job[b].  Everything else -- and so every bit of a score -- is the single-reference code.
template <bool kRef, bool kJobs = false>
__global__ void __launch_bounds__(256) k_shape_grid(const float* __restrict__ coords, const int* __restrict__ n_nodes, int n_fixed,
                                                    int N, const float* __restrict__ frames, const float* __restrict__ orient,
                                                    int n_orient, const float* __restrict__ axes, int G, float amplitude,
                                                    float alpha, float* dens, float* __restrict__ scores,
                                                    float* __restrict__ aligned, const int* __restrict__ job = nullptr) {
  __shared__ float tx[SHAPE_MAX_ATOMS][SHAPE_MAX_GRID], ty[SHAPE_MAX_ATOMS][SHAPE_MAX_GRID], tz[SHAPE_MAX_ATOMS][SHAPE_MAX_GRID];
  __shared__ float px[SHAPE_MAX_ATOMS], py[SHAPE_MAX_ATOMS], pz[SHAPE_MAX_ATOMS];
  __shared__ float red[2][8];
  const int b = blockIdx.x, o = blockIdx.y, tid = threadIdx.x;
  const int n = (kRef && !kJobs) ? n_fixed : n_nodes[b];
  if (kJobs) {
    const size_t j = kRef ? (size_t)b : (size_t)job[b];
    axes += j * 3 * G;
    dens += j * ((size_t)G * G * G + 1);
  }
  if (tid < n) {
    const float* x = coords + ((size_t)b * N + tid) * 3;
    float v[3] = {x[0], x[1], x[2]};
    if (!kRef) {
      const float* f = frames + (size_t)b * 12;
      const float c0 = v[0] - f[0], c1 = v[1] - f[1], c2 = v[2] - f[2];
      // principal frame: row vector times the (column-permuted) eigenvector matrix (shape_similarity.py:139-140, 199)
      const float r0 = c0 * f[3] + c1 * f[6] + c2 * f[9];
      const float r1 = c0 * f[4] + c1 * f[7] + c2 * f[10];
      const float r2 = c0 * f[5] + c1 * f[8] + c2 * f[11];
      if (o == 0) {  // the first orientation is the unrotated principal frame (pipeline.py:76)
        v[0] = r0; v[1] = r1; v[2] = r2;
      } else {
        const float* q = orient + (size_t)o * 9;
        v[0] = r0 * q[0] + r1 * q[3] + r2 * q[6];
        v[1] = r0 * q[1] + r1 * q[4] + r2 * q[7];
        v[2] = r0 * q[2] + r1 * q[5] + r2 * q[8];
      }
      if (aligned != nullptr) {
        float* a = aligned + (((size_t)b * n_orient + o) * N + tid) * 3;
        a[0] = v[0]; a[1] = v[1]; a[2] = v[2];
      }
    }
    px[tid] = v[0]; py[tid] = v[1]; pz[tid] = v[2];
  }
  __syncthreads();
  // separable Gaussian tables: t?[a][i] = exp(-alpha (axis_i - c_a)^2)
  for (int e = tid; e < n * G; e += blockDim.x) {
    const int a = e / G, i = e - a * G;
    const float dx = axes[i] - px[a], dy = axes[G + i] - py[a], dz = axes[2 * G + i] - pz[a];
    tx[a][i] = __expf(-alpha * dx * dx);
    ty[a][i] = __expf(-alpha * dy * dy);
    tz[a][i] = __expf(-alpha * dz * dz);
  }
  __syncthreads();
  float fg = 0.f, gg = 0.f;
  // thread = column (ix, iy); the G products along z stay in registers
  for (int col = tid; col < G * G; col += blockDim.x) {
    const int ix = col / G, iy = col - ix * G;
    float prod[SHAPE_MAX_GRID];
#pragma unroll
    for (int z = 0; z < SHAPE_MAX_GRID; ++z) prod[z] = 1.0f;
    for (int a = 0; a < n; ++a) {
      const float exy = amplitude * tx[a][ix] * ty[a][iy];
#pragma unroll
      for (int z = 0; z < SHAPE_MAX_GRID; ++z)
        if (z < G) prod[z] *= fmaf(-exy, tz[a][z], 1.0f);  // 1 - A exp(-alpha d^2)   (shape_similarity.py:415-417)
    }
    float* drow = dens + (size_t)col * G;
#pragma unroll
    for (int z = 0; z < SHAPE_MAX_GRID; ++z) {
      if (z < G) {
        const float g = 1.0f - prod[z];
        if (kRef) {
          drow[z] = g;
          gg += g * g;
        } else {
          const float f = drow[z];
          fg += f * g;
          gg += g * g;
        }
      }
    }
  }
  for (int s = 16; s > 0; s >>= 1) {
    fg += __shfl_down_sync(0xffffffffu, fg, s);
    gg += __shfl_down_sync(0xffffffffu, gg, s);
  }
  if ((tid & 31) == 0) { red[0][tid >> 5] = fg; red[1][tid >> 5] = gg; }
  __syncthreads();
  if (tid == 0) {
    float sfg = 0.f, sgg = 0.f;
    for (int w = 0; w < 8; ++w) { sfg += red[0][w]; sgg += red[1][w]; }
    if (kRef) {
      dens[(size_t)G * G * G] = sgg;
    } else {
      const float f2 = dens[(size_t)G * G * G];
      scores[(size_t)b * n_orient + o] = sfg / (f2 + sgg - sfg);  // shape_similarity.py:486-490
    }
  }
}

}  // namespace mlcg
