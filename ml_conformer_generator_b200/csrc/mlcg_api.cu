// C-ABI of libmlcg_b200.so (see include/mlcg.h).  Host-side orchestration only: weight repacking at load time, batch
// plan (edge-tile table), kernel sequencing of one EGNN forward / the reverse-diffusion loop / the AdjMatSeer GCN.
#include <algorithm>
#include <cstddef>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include "mlcg.h"
#include "mlcg_kernels.cuh"
#include "mlcg_tc.cuh"
#include "mlcg_tc3.cuh"
#include "mlcg_shape.cuh"
#include "mlcg_ifm.cuh"

using namespace mlcg;

namespace {

struct Wt {
  float* d = nullptr;
  int rows = 0, cols = 0;
};

struct DevBuf {
  void* p = nullptr;
  size_t bytes = 0;
  cudaError_t ensure(size_t need, bool zero = true) {
    if (need <= bytes) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr;
    bytes = 0;
    cudaError_t e = cudaMalloc(&p, need);
    if (e != cudaSuccess) return e;
    bytes = need;
    return zero ? cudaMemset(p, 0, need) : cudaSuccess;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    bytes = 0;
  }
  template <class T>
  T* as() const { return reinterpret_cast<T*>(p); }
};

struct LayerW {
  bool equiv = false;
  Wt w1, b1, w2, b2, w3, b3, w4, b4, wv;  // raw fp32 (owned copies)
  float att_bias = 0.f;
  DevBuf w1ab_op, w2_op, w3_op, w4_op;  // operand-format (tensor-core modes)
  DevBuf bias_pq, wc, wd, wvp, b3p, b4p;  // padded fp32 vectors
  float h_wc[HP], h_wd[HP], h_wv[HP];     // host copies passed to the edge kernel through the constant bank
};

struct SeerLayer {
  Wt w, b;
  DevBuf w_op, b_pad;
  int k = 0, n = 0;
};

struct SimtChunk { int node_begin, node_end, edge_base, edge_rows; };

// Batch plan: the geometry of one batch (atom counts, edge-tile table, split targets) and its device copies.  The kernels
// read the handle's active plan; the workspaces they write are shared by all plans and sized to the largest.
struct BatchPlan {
  int B = 0, N = 0, M = 0, n_mtiles = 0, n_etiles = 0;
  long long n_edges = 0;
  std::vector<int> h_n_nodes, h_node_off;
  std::vector<SimtChunk> simt_chunks;
  DevBuf d_n_nodes, d_node_off, d_node_mol, d_node_edge_off, d_tiles, d_fix_node;
  DevBuf fix_agg, fix_dx;  // side buffers of the split targets: zero between edge-kernel launches
  int n_fix = 0;           // target nodes whose neighbour list is split over two edge tiles
  void release() {
    for (DevBuf* b : {&d_n_nodes, &d_node_off, &d_node_mol, &d_node_edge_off, &d_tiles, &d_fix_node, &fix_agg, &fix_dx})
      b->release();
  }
};

}  // namespace

struct mlcg_handle {
  int device = 0, precision = 0, num_sms = 148;
  std::string err;
  long long launches = 0;
  bool egnn_loaded = false, seer_loaded = false, batch_set = false;
  std::map<std::string, Wt> egnn_w, seer_w;
  std::vector<void*> owned;
  Wt w_emb, b_emb, w_out, b_out;
  LayerW layers[27];
  SeerLayer seer_gcn[7];  // gcn1_dm gcn2_dm gcn3_dm gcn1 gcn2 gcn3 gcn4
  SeerLayer seer_resize;
  // batch plans: plans[0] is the one mlcg_set_batch builds; mlcg_generate_fragment keeps the geometry of its first loop
  // (inertial fragment matching: the atoms still to be generated) in plans[1] and switches `pl` between launches
  BatchPlan plans[2];
  BatchPlan* pl = &plans[0];
  // EGNN workspaces
  DevBuf x0, xa, xb, h_res, pq, h_op, agg_op, t_op, agg_f32, t_f32, a1, m2, t_dev, eps_dev;
  // seer workspaces
  DevBuf s_ld, s_la, s_rowd, s_rowa, s_x64, s_y_op, s_x, s_emb, s_add, s_raw, s_y_f32;
  // mlcg_generate device buffers
  DevBuf g_ctx, g_z, g_x, g_cls, g_el, g_dist, g_adj, g_bonds, g_ids;
  // mlcg_generate_fragment(_jobs) device buffers: packed fragments, job table, job of every sample, z_known / fixed_mask,
  // and the first IFM loop's context and outputs
  DevBuf f_ffx, f_ffh, f_jobs, f_job, f_zk, f_fm, f_ctx, f_shift, f_rot, f_ngen, f_xg, f_clsg;
  DevBuf hook_job;  // the one-job table of the eager hooks mlcg_ifm_context / mlcg_ifm_merge_inputs
  DevBuf nf_flag;  // set by k_decode when a generated coordinate is not finite (mlcg_nonfinite)
  std::vector<int64_t> ids_stage;
  // test gemm
  DevBuf tg_a, tg_w, tg_b, tg_c;
  // CUDA-graph replay of mlcg_generate (whole reverse loop + GCN as one graph)
  DevBuf noise_ctl;               // {seed, sample_offset} read by the noise kernels when use_noise_ctl is set
  bool use_noise_ctl = false;
  cudaGraphExec_t gen_graph = nullptr;
  std::vector<long long> gen_key;  // geometry / schedule the graph was captured for
  int gen_key_hits = 0;            // calls seen with the current key (1st runs eagerly, 2nd captures)
  long long gen_graph_launches = 0;
  long long graph_captures = 0;    // CUDA graphs captured by mlcg_generate / mlcg_generate_fragment(_jobs)
  cudaStream_t own_stream = nullptr;  // used by mlcg_generate when the caller passes the NULL stream (not capturable)
  // mlcg_egnn_forward_breakdown: events recorded after every launch of one forward, tagged with a kernel class
  bool bd_on = false;
  std::vector<std::pair<int, cudaEvent_t>> bd_ev;
  int kc448() const { return HP / epc(is16(precision) ? PREC_BF16 : PREC_TF32); }
};

#define CK(call)                                                                              \
  do {                                                                                        \
    cudaError_t _e = (call);                                                                  \
    if (_e != cudaSuccess) {                                                                  \
      h->err = std::string(#call) + ": " + cudaGetErrorString(_e);                            \
      return (int)_e;                                                                         \
    }                                                                                         \
  } while (0)
#define KCHECK()                                 \
  do {                                           \
    h->launches++;                               \
    CK(cudaGetLastError());                      \
  } while (0)
#define FAIL(code, msg) \
  do {                  \
    h->err = (msg);     \
    return (code);      \
  } while (0)

static thread_local std::string g_create_err;

// kernel classes of one EGNN forward (mlcg_egnn_forward_breakdown)
enum { BD_START = -1, BD_PREPARE = 0, BD_PQ = 1, BD_EDGE_GCL = 2, BD_EDGE_EQUIV = 3, BD_FIXUP = 4, BD_MLP1 = 5, BD_MLP2 = 6,
       BD_READOUT = 7, BD_NCLASS = 8 };
static void bd_mark(mlcg_handle* h, int cls, cudaStream_t st) {
  if (!h->bd_on) return;
  cudaEvent_t e;
  if (cudaEventCreate(&e) != cudaSuccess) return;
  cudaEventRecord(e, st);
  h->bd_ev.emplace_back(cls, e);
}

// ---------------------------------------------------------------------------------------------------------------
// kernel launch helpers
// ---------------------------------------------------------------------------------------------------------------
template <int kMode, int BN, int kEpi>
static cudaError_t launch_gemm(const GemmArgs& a, int n_mtiles, int n_ntiles, cudaStream_t st) {
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(k_tc_gemm<kMode, BN, kEpi>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         GemmCfg<BN>::SMEM_BYTES);
    if (e != cudaSuccess) return e;
    attr_set = true;
  }
  static int num_sms = 0;
  if (num_sms == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev);
    if (num_sms <= 0) num_sms = 148;
  }
  GemmArgs b = a;
  b.n_mtiles = n_mtiles;
  b.n_ntiles = n_ntiles;
  k_tc_gemm<kMode, BN, kEpi><<<std::min(n_mtiles * n_ntiles, num_sms), GEMM_THREADS, GemmCfg<BN>::SMEM_BYTES, st>>>(b);
  return cudaGetLastError();
}
template <int BN, int kEpi>
static cudaError_t launch_gemm_mode(int mode, const GemmArgs& a, int n_mtiles, int n_ntiles, cudaStream_t st) {
  if (mode == PREC_FP16) return launch_gemm<PREC_FP16, BN, kEpi>(a, n_mtiles, n_ntiles, st);
  return mode == PREC_BF16 ? launch_gemm<PREC_BF16, BN, kEpi>(a, n_mtiles, n_ntiles, st)
                           : launch_gemm<PREC_TF32, BN, kEpi>(a, n_mtiles, n_ntiles, st);
}
template <int kMode, bool kEquiv, bool kPair, bool kDistF32 = false, bool kProf = false>
static cudaError_t launch_edge(const EdgeArgs& a, int grid, cudaStream_t st) {
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(k_tc_edge<kMode, kEquiv, kPair, kDistF32, kProf>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         EdgeSmemT<kMode>::ALLOC);
    if (e != cudaSuccess) return e;
    attr_set = true;
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(EDGE_THREADS);
  cfg.dynamicSmemBytes = EdgeSmemT<kMode>::ALLOC;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = kPair ? 2 : 1;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, k_tc_edge<kMode, kEquiv, kPair, kDistF32, kProf>, a);
}
// Edge tiles are 128-row ranges of a molecule's edge list that may split a target node's neighbours over two tiles
// (default); MLCG_EDGE_SPLIT=0 keeps whole targets per tile (lower row occupancy, no fix-up kernel).
static bool edge_split_mode() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("MLCG_EDGE_SPLIT");
    v = (e == nullptr) ? 1 : (atoi(e) != 0);
  }
  return v != 0;
}
// The 16-bit modes evaluate the first-layer distance terms d2 * wc + d0^2 * wd either packed (bf16x2 / f16x2 FMAs) or in
// fp32 (one rounding of the whole pre-activation; ~4.5 % slower).  It only matters when the distance terms dominate the
// pre-activation and cancel -- the random-weight trajectories of the parity tests, where |x| grows to ~1e3.  Default: fp32
// in fp16 mode (the parity mode: per-step eps and argmax agreement on a par with tf32, profiles/r2_parity.txt), packed in
// bf16 mode.  MLCG_EDGE_DIST_FP32=0/1 overrides either default.
static bool edge_dist_fp32(int mode) {
  static int v = -2;
  if (v == -2) {
    const char* e = getenv("MLCG_EDGE_DIST_FP32");
    v = (e == nullptr) ? -1 : (atoi(e) != 0);
  }
  return v < 0 ? (mode == PREC_FP16) : (v != 0);
}
// AdjMatSeer GEMMs: error-compensated 3xTF32 (default) or plain tf32 (MLCG_SEER_3XTF32=0: a third of the GEMM time, logits
// to ~1e-4 instead of ~1e-6; the bond argmax of a random-init GCN then flips on ties below that error).
static bool seer_split3() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("MLCG_SEER_3XTF32");
    v = (e == nullptr) ? 1 : (atoi(e) != 0);
  }
  return v != 0;
}
// CTA-pair mode (default) needs an even grid; MLCG_EDGE_PAIR=0 selects the single-CTA kernel.
static bool edge_pair_mode() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("MLCG_EDGE_PAIR");
    v = (e == nullptr) ? 1 : (atoi(e) != 0);
  }
  return v != 0;
}
// grid of the persistent edge kernel: one CTA per SM (MLCG_EDGE_GRID overrides it for scaling experiments)
static int edge_grid_for(int n_tiles, int num_sms) {
  int g = std::min(n_tiles, num_sms);
  if (const char* e = getenv("MLCG_EDGE_GRID")) g = std::max(1, std::min(g, atoi(e)));
  return g;
}
// which CTA processes tile t: the same contiguous ranges k_tc_edge computes from (blockIdx, gridDim, n_tiles)
static void edge_tile_owner(int num_sms, int n_tiles, std::vector<int>& owner) {
  owner.assign(n_tiles, 0);
  int grid = edge_grid_for(n_tiles, num_sms);
  const bool pair = edge_pair_mode() && grid >= 2;
  if (pair) grid &= ~1;
  if (grid <= 0) return;
  if (pair) {
    const int npairs = grid / 2;
    for (int pr = 0; pr < npairs; ++pr) {
      const int T0 = (int)(((long long)pr * n_tiles) / npairs), T1 = (int)(((long long)(pr + 1) * n_tiles) / npairs);
      const int n_iter = (T1 - T0 + 1) >> 1;
      for (int t = T0; t < T1; ++t) owner[t] = 2 * pr + (t >= T0 + n_iter ? 1 : 0);
    }
  } else {
    for (int b = 0; b < grid; ++b) {
      const int t0 = (int)(((long long)b * n_tiles) / grid), t1 = (int)(((long long)(b + 1) * n_tiles) / grid);
      for (int t = t0; t < t1; ++t) owner[t] = b;
    }
  }
}
// k_tc_edge3 (mlcg_tc3.cuh): resident A operand + two ping-pong 144-column accumulators.  16-bit modes, CTA pairs.
template <int kMode, bool kEquiv, bool kDistF32, bool kProf = false>
static cudaError_t launch_edge3(const EdgeArgs& a, int grid, cudaStream_t st) {
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(k_tc_edge3<kMode, kEquiv, kDistF32, kProf>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         Edge3Smem<kMode, kEquiv>::ALLOC);
    if (e != cudaSuccess) return e;
    attr_set = true;
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(EDGE_THREADS);
  cfg.dynamicSmemBytes = Edge3Smem<kMode, kEquiv>::ALLOC;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, k_tc_edge3<kMode, kEquiv, kDistF32, kProf>, a);
}
// MLCG_EDGE_V3=0 selects the single-accumulator kernel k_tc_edge in the 16-bit modes (A/B measurements); default: k_tc_edge3
static bool edge_v3_mode() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("MLCG_EDGE_V3");
    v = (e == nullptr) ? 1 : (atoi(e) != 0);
  }
  return v != 0;
}
static cudaError_t launch_edge_mode(int mode, bool equiv, const EdgeArgs& a, int grid, cudaStream_t st, bool prof = false) {
  const bool pair = edge_pair_mode() && grid >= 2;
  if (pair) grid &= ~1;
  if (prof && pair && is16(mode) && edge_v3_mode() && a.n_kc == E3_NKC) {
    // instrumented instantiations of the default variant of each mode
    if (edge_dist_fp32(mode) != (mode == PREC_FP16)) return cudaErrorNotSupported;
    if (mode == PREC_FP16)
      return equiv ? launch_edge3<PREC_FP16, true, true, true>(a, grid, st) : launch_edge3<PREC_FP16, false, true, true>(a, grid, st);
    return equiv ? launch_edge3<PREC_BF16, true, false, true>(a, grid, st) : launch_edge3<PREC_BF16, false, false, true>(a, grid, st);
  }
  if (!prof && pair && is16(mode) && edge_v3_mode() && a.n_kc == E3_NKC) {
    const bool df = edge_dist_fp32(mode);
    if (mode == PREC_FP16) {
      if (df) return equiv ? launch_edge3<PREC_FP16, true, true>(a, grid, st) : launch_edge3<PREC_FP16, false, true>(a, grid, st);
      return equiv ? launch_edge3<PREC_FP16, true, false>(a, grid, st) : launch_edge3<PREC_FP16, false, false>(a, grid, st);
    }
    if (df) return equiv ? launch_edge3<PREC_BF16, true, true>(a, grid, st) : launch_edge3<PREC_BF16, false, true>(a, grid, st);
    return equiv ? launch_edge3<PREC_BF16, true, false>(a, grid, st) : launch_edge3<PREC_BF16, false, false>(a, grid, st);
  }
  if (prof) {
    // instrumented instantiations exist for the default variant of each mode only (CTA pairs, default distance terms)
    if (!pair || edge_dist_fp32(mode) != (mode == PREC_FP16)) return cudaErrorNotSupported;
    if (mode == PREC_FP16)
      return equiv ? launch_edge<PREC_FP16, true, true, true, true>(a, grid, st) : launch_edge<PREC_FP16, false, true, true, true>(a, grid, st);
    if (mode == PREC_BF16)
      return equiv ? launch_edge<PREC_BF16, true, true, false, true>(a, grid, st) : launch_edge<PREC_BF16, false, true, false, true>(a, grid, st);
    return equiv ? launch_edge<PREC_TF32, true, true, false, true>(a, grid, st) : launch_edge<PREC_TF32, false, true, false, true>(a, grid, st);
  }
  if (mode == PREC_FP16 && edge_dist_fp32(mode)) {
    if (pair)
      return equiv ? launch_edge<PREC_FP16, true, true, true>(a, grid, st) : launch_edge<PREC_FP16, false, true, true>(a, grid, st);
    return equiv ? launch_edge<PREC_FP16, true, false, true>(a, grid, st) : launch_edge<PREC_FP16, false, false, true>(a, grid, st);
  }
  if (mode == PREC_FP16) {
    if (pair) return equiv ? launch_edge<PREC_FP16, true, true>(a, grid, st) : launch_edge<PREC_FP16, false, true>(a, grid, st);
    return equiv ? launch_edge<PREC_FP16, true, false>(a, grid, st) : launch_edge<PREC_FP16, false, false>(a, grid, st);
  }
  if (mode == PREC_BF16 && edge_dist_fp32(mode)) {
    if (pair)
      return equiv ? launch_edge<PREC_BF16, true, true, true>(a, grid, st) : launch_edge<PREC_BF16, false, true, true>(a, grid, st);
    return equiv ? launch_edge<PREC_BF16, true, false, true>(a, grid, st) : launch_edge<PREC_BF16, false, false, true>(a, grid, st);
  }
  if (mode == PREC_BF16) {
    if (pair) return equiv ? launch_edge<PREC_BF16, true, true>(a, grid, st) : launch_edge<PREC_BF16, false, true>(a, grid, st);
    return equiv ? launch_edge<PREC_BF16, true, false>(a, grid, st) : launch_edge<PREC_BF16, false, false>(a, grid, st);
  }
  if (pair) return equiv ? launch_edge<PREC_TF32, true, true>(a, grid, st) : launch_edge<PREC_TF32, false, true>(a, grid, st);
  return equiv ? launch_edge<PREC_TF32, true, false>(a, grid, st) : launch_edge<PREC_TF32, false, false>(a, grid, st);
}
// second half of an edge layer: completes the targets whose neighbour list is split over two tiles
static cudaError_t launch_edge_fixup(mlcg_handle* h, int mode, bool equiv, const EdgeArgs& a, cudaStream_t st) {
  if (h->pl->n_fix == 0) return cudaSuccess;
  const int* fn = h->pl->d_fix_node.as<int>();
  if (equiv) {
    const int grid = (h->pl->n_fix * 4 + 127) / 128;
    if (is16(mode))  // the coordinate fix-up does not depend on the operand format
      k_edge_fixup<PREC_BF16, true><<<grid, 128, 0, st>>>(fn, h->pl->n_fix, a.fix_agg, a.fix_dx, a.agg_op, a.agg_chunks, a.x_cur, a.x_next);
    else
      k_edge_fixup<PREC_TF32, true><<<grid, 128, 0, st>>>(fn, h->pl->n_fix, a.fix_agg, a.fix_dx, a.agg_op, a.agg_chunks, a.x_cur, a.x_next);
  } else {
    if (mode == PREC_FP16) {
      const int grid = (h->pl->n_fix * (HP / epp(PREC_FP16)) + 127) / 128;
      k_edge_fixup<PREC_FP16, false><<<grid, 128, 0, st>>>(fn, h->pl->n_fix, a.fix_agg, a.fix_dx, a.agg_op, a.agg_chunks, a.x_cur, a.x_next);
    } else if (mode == PREC_BF16) {
      const int grid = (h->pl->n_fix * (HP / epp(PREC_BF16)) + 127) / 128;
      k_edge_fixup<PREC_BF16, false><<<grid, 128, 0, st>>>(fn, h->pl->n_fix, a.fix_agg, a.fix_dx, a.agg_op, a.agg_chunks, a.x_cur, a.x_next);
    } else {
      const int grid = (h->pl->n_fix * (HP / epp(PREC_TF32)) + 127) / 128;
      k_edge_fixup<PREC_TF32, false><<<grid, 128, 0, st>>>(fn, h->pl->n_fix, a.fix_agg, a.fix_dx, a.agg_op, a.agg_chunks, a.x_cur, a.x_next);
    }
  }
  h->launches++;
  return cudaGetLastError();
}

static cudaError_t launch_pack(int mode, const PackArgs& a, int n_ntiles, cudaStream_t st) {
  dim3 grid(a.n_kc, n_ntiles);
  if (mode == PREC_FP16) k_pack_weight<PREC_FP16><<<grid, 256, 0, st>>>(a);
  else if (mode == PREC_BF16) k_pack_weight<PREC_BF16><<<grid, 256, 0, st>>>(a);
  else k_pack_weight<PREC_TF32><<<grid, 256, 0, st>>>(a);
  return cudaGetLastError();
}
__global__ void k_fill_f32(float* p, float v, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}

static NoiseSrc to_src(const mlcg_handle* h, const mlcg_noise* n) {
  NoiseSrc s;
  s.raw = n->raw;
  s.seed = n->seed;
  s.draw = n->draw;
  s.sample_offset = n->sample_offset;
  s.ids = reinterpret_cast<const long long*>(n->sample_ids);
  s.ctl = (h->use_noise_ctl && n->raw == nullptr) ? h->noise_ctl.as<unsigned long long>() : nullptr;
  return s;
}

// ---------------------------------------------------------------------------------------------------------------
// create / destroy
// ---------------------------------------------------------------------------------------------------------------
extern "C" const char* mlcg_version(void) { return "mlcg_b200 0.1 (sm_100a)"; }

extern "C" int mlcg_create(mlcg_handle** out, int device, int precision) {
  if (out == nullptr || precision < 0 || precision > 3) return MLCG_E_ARG;
  *out = nullptr;
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0 || device >= count) return MLCG_E_NO_DEVICE;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return MLCG_E_NO_DEVICE;
  if (prop.major != 10) return MLCG_E_NO_DEVICE;  // sm_100a cubins only
  if (cudaSetDevice(device) != cudaSuccess) return MLCG_E_NO_DEVICE;
  mlcg_handle* h = new mlcg_handle();
  h->device = device;
  h->precision = precision;
  h->num_sms = prop.multiProcessorCount;
  *out = h;
  return MLCG_OK;
}

extern "C" void mlcg_destroy(mlcg_handle* h) {
  if (!h) return;
  cudaSetDevice(h->device);
  for (void* p : h->owned) cudaFree(p);
  for (auto& l : h->layers) {
    for (DevBuf* b : {&l.w1ab_op, &l.w2_op, &l.w3_op, &l.w4_op, &l.bias_pq, &l.wc, &l.wd, &l.wvp, &l.b3p, &l.b4p}) b->release();
  }
  for (auto& s : h->seer_gcn) { s.w_op.release(); s.b_pad.release(); }
  h->seer_resize.w_op.release();
  h->seer_resize.b_pad.release();
  if (h->gen_graph) cudaGraphExecDestroy(h->gen_graph);
  if (h->own_stream) cudaStreamDestroy(h->own_stream);
  h->noise_ctl.release();
  for (BatchPlan& p : h->plans) p.release();
  for (DevBuf* b : {&h->x0, &h->xa, &h->xb,
                    &h->h_res, &h->pq, &h->h_op, &h->agg_op, &h->t_op, &h->agg_f32, &h->t_f32, &h->a1, &h->m2, &h->t_dev,
                    &h->eps_dev, &h->s_ld, &h->s_la, &h->s_rowd, &h->s_rowa, &h->s_x64, &h->s_y_op, &h->s_x, &h->s_emb,
                    &h->s_add, &h->s_raw, &h->s_y_f32, &h->g_ctx, &h->g_z, &h->g_x, &h->g_cls, &h->g_el, &h->g_dist,
                    &h->g_adj, &h->g_bonds, &h->g_ids, &h->f_ffx, &h->f_ffh, &h->f_jobs, &h->f_job, &h->hook_job, &h->f_zk, &h->f_fm, &h->f_ctx, &h->f_shift,
                    &h->f_rot, &h->f_ngen, &h->f_xg, &h->f_clsg, &h->nf_flag, &h->tg_a, &h->tg_w, &h->tg_b, &h->tg_c})
    b->release();
  delete h;
}

extern "C" const char* mlcg_last_error(mlcg_handle* h) { return h ? h->err.c_str() : "null handle"; }

// ---------------------------------------------------------------------------------------------------------------
// weights
// ---------------------------------------------------------------------------------------------------------------
static int copy_weights(mlcg_handle* h, const mlcg_weight_desc* w, int n, std::map<std::string, Wt>& dst) {
  // new weights invalidate a captured generation graph (it holds the old buffers' addresses); nothing may be in flight
  CK(cudaDeviceSynchronize());
  if (h->gen_graph) { cudaGraphExecDestroy(h->gen_graph); h->gen_graph = nullptr; }
  h->gen_key.clear();
  h->gen_key_hits = 0;
  for (int i = 0; i < n; ++i) {
    if (!w[i].name || !w[i].data || w[i].rows <= 0 || w[i].cols <= 0) FAIL(MLCG_E_ARG, "bad weight descriptor");
    Wt t;
    t.rows = w[i].rows;
    t.cols = w[i].cols;
    const size_t bytes = (size_t)t.rows * t.cols * sizeof(float);
    auto old = dst.find(w[i].name);
    if (old != dst.end()) {  // reloading: release the previous copy
      h->owned.erase(std::remove(h->owned.begin(), h->owned.end(), (void*)old->second.d), h->owned.end());
      cudaFree(old->second.d);
    }
    CK(cudaMalloc((void**)&t.d, bytes));
    h->owned.push_back(t.d);
    CK(cudaMemcpy(t.d, w[i].data, bytes, cudaMemcpyDeviceToDevice));
    dst[w[i].name] = t;
  }
  return MLCG_OK;
}
static int need(mlcg_handle* h, std::map<std::string, Wt>& m, const std::string& key, int rows, int cols, Wt* out) {
  auto it = m.find(key);
  if (it == m.end()) FAIL(MLCG_E_WEIGHT, "missing state_dict entry: " + key);
  if (it->second.rows != rows || it->second.cols != cols)
    FAIL(MLCG_E_WEIGHT, "bad shape for " + key + ": got (" + std::to_string(it->second.rows) + "," +
                            std::to_string(it->second.cols) + ")");
  *out = it->second;
  return MLCG_OK;
}
static int pad_vec(mlcg_handle* h, DevBuf& dst, const float* src, int stride, int n_real, int n_pad, int dst_off = 0,
                   int alloc = -1, float scale = 1.0f) {
  CK(dst.ensure((size_t)(alloc < 0 ? n_pad : alloc) * sizeof(float)));
  k_pad_vector<<<(n_pad + 127) / 128, 128>>>(src, stride, n_real, dst.as<float>() + dst_off, n_pad, scale);
  KCHECK();
  return MLCG_OK;
}

extern "C" int mlcg_load_egnn(mlcg_handle* h, const mlcg_weight_desc* w, int n) {
  if (!h) return MLCG_E_ARG;
  CK(cudaSetDevice(h->device));
  int rc = copy_weights(h, w, n, h->egnn_w);
  if (rc) return rc;
  auto& m = h->egnn_w;
  const std::string p = "dynamics.egnn.";
  if ((rc = need(h, m, p + "embedding.weight", HID, IN_NF, &h->w_emb))) return rc;
  if ((rc = need(h, m, p + "embedding.bias", HID, 1, &h->b_emb))) return rc;
  if ((rc = need(h, m, p + "embedding_out.weight", IN_NF, HID, &h->w_out))) return rc;
  if ((rc = need(h, m, p + "embedding_out.bias", IN_NF, 1, &h->b_out))) return rc;
  const int mode = h->precision;
  const int kc = h->kc448();
  // bf16 fast mode evaluates SiLU as h + h*tanh(h) with h = x/2: the exact factor 1/2 is folded into the packed first
  // and second edge-layer weights, their biases and the distance columns (tensor-core path only).
  const float es = is16(mode) ? 0.5f : 1.0f;
  // fp16 mode: power-of-two range scales (mlcg_common.cuh): ACT on the edge pre-activations, OP on the node-level GEMM
  // operands; the inverses are folded into the packed weights here.  Both are 1 in the other modes.
  const float s_act = act_scale(mode), s_op = op_scale(mode);
  for (int l = 0; l < 27; ++l) {
    LayerW& L = h->layers[l];
    const int blk = l / 3, sub = l % 3;
    L.equiv = (sub == 2);
    const std::string q = p + "e_block_" + std::to_string(blk) + (L.equiv ? ".gcl_equiv." : (sub == 0 ? ".gcl_0." : ".gcl_1."));
    const std::string e = L.equiv ? "coord_mlp." : "edge_mlp.";
    if ((rc = need(h, m, q + e + "0.weight", HID, 2 * HID + 2, &L.w1))) return rc;
    if ((rc = need(h, m, q + e + "0.bias", HID, 1, &L.b1))) return rc;
    if ((rc = need(h, m, q + e + "2.weight", HID, HID, &L.w2))) return rc;
    if ((rc = need(h, m, q + e + "2.bias", HID, 1, &L.b2))) return rc;
    if (L.equiv) {
      if ((rc = need(h, m, q + "coord_mlp.4.weight", 1, HID, &L.wv))) return rc;
      L.att_bias = 0.f;
    } else {
      if ((rc = need(h, m, q + "node_mlp.0.weight", HID, 2 * HID, &L.w3))) return rc;
      if ((rc = need(h, m, q + "node_mlp.0.bias", HID, 1, &L.b3))) return rc;
      if ((rc = need(h, m, q + "node_mlp.2.weight", HID, HID, &L.w4))) return rc;
      if ((rc = need(h, m, q + "node_mlp.2.bias", HID, 1, &L.b4))) return rc;
      if ((rc = need(h, m, q + "att_mlp.0.weight", 1, HID, &L.wv))) return rc;
      Wt ab;
      if ((rc = need(h, m, q + "att_mlp.0.bias", 1, 1, &ab))) return rc;
      CK(cudaMemcpy(&L.att_bias, ab.d, sizeof(float), cudaMemcpyDeviceToHost));
    }
    // padded vectors (all modes)
    if ((rc = pad_vec(h, L.wc, L.w1.d + 2 * HID, 2 * HID + 2, HID, HP, 0, -1, es * s_act))) return rc;
    if ((rc = pad_vec(h, L.wd, L.w1.d + 2 * HID + 1, 2 * HID + 2, HID, HP, 0, -1, es * s_act))) return rc;
    if ((rc = pad_vec(h, L.wvp, L.wv.d, 1, HID, HP))) return rc;
    if ((rc = pad_vec(h, L.bias_pq, L.b1.d, 1, HID, HP, HP, 2 * HP, es))) return rc;  // [0 | b1]
    CK(cudaMemcpy(L.h_wc, L.wc.p, HP * sizeof(float), cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(L.h_wd, L.wd.p, HP * sizeof(float), cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(L.h_wv, L.wvp.p, HP * sizeof(float), cudaMemcpyDeviceToHost));
    if (!L.equiv) {
      if ((rc = pad_vec(h, L.b3p, L.b3.d, 1, HID, HP))) return rc;
      if ((rc = pad_vec(h, L.b4p, L.b4.d, 1, HID, HP))) return rc;
    }
    if (mode == PREC_FP32_SIMT) continue;
    const size_t blk448 = (size_t)HP * CHUNK_BYTES;
    // W1 split into the P (cols 0..419) and Q (cols 420..839) projections: N = 896 as two 448-row tiles
    CK(L.w1ab_op.ensure(2 * kc * blk448));
    for (int half = 0; half < 2; ++half) {
      PackArgs a{};
      a.src = L.w1.d; a.ld = 2 * HID + 2; a.n_real = HID; a.n_src_off = 0; a.bn = HP; a.n_kc = kc;
      a.seg_len = HP; a.kreal0 = HID; a.kofs0 = half * HID; a.kreal1 = 0; a.kofs1 = 0;
      a.bias = nullptr; a.bias_k = -1; a.scale = es / s_op;  // the operand h arrives scaled by OP
      a.dst = L.w1ab_op.as<uint8_t>() + (size_t)half * kc * blk448;
      CK(launch_pack(mode, a, 1, 0));
      h->launches++;
    }
    {  // W2 with b2 folded into K column 420
      CK(L.w2_op.ensure(kc * blk448));
      PackArgs a{};
      a.src = L.w2.d; a.ld = HID; a.n_real = HID; a.bn = HP; a.n_kc = kc; a.seg_len = HP; a.kreal0 = HID;
      a.bias = L.b2.d; a.bias_k = BIAS_COL; a.dst = L.w2_op.as<uint8_t>(); a.scale = es;
      CK(launch_pack(mode, a, 1, 0));
      h->launches++;
    }
    if (!L.equiv) {
      CK(L.w3_op.ensure(2 * kc * blk448));
      PackArgs a{};
      a.src = L.w3.d; a.ld = 2 * HID; a.n_real = HID; a.bn = HP; a.n_kc = 2 * kc; a.seg_len = HP;
      a.kreal0 = HID; a.kofs0 = 0; a.kreal1 = HID; a.kofs1 = HID; a.bias = nullptr; a.bias_k = -1;
      a.scale = 1.0f / s_op;  // both operand halves (h, agg) arrive scaled by OP
      a.dst = L.w3_op.as<uint8_t>();
      CK(launch_pack(mode, a, 1, 0));
      h->launches++;
      CK(L.w4_op.ensure(kc * blk448));
      PackArgs b{};
      b.src = L.w4.d; b.ld = HID; b.n_real = HID; b.bn = HP; b.n_kc = kc; b.seg_len = HP; b.kreal0 = HID;
      b.bias = nullptr; b.bias_k = -1; b.dst = L.w4_op.as<uint8_t>();
      b.scale = 1.0f / s_op;  // the hidden operand t arrives scaled by OP
      CK(launch_pack(mode, b, 1, 0));
      h->launches++;
    }
  }
  CK(cudaDeviceSynchronize());
  h->egnn_loaded = true;
  return MLCG_OK;
}

extern "C" int mlcg_load_seer(mlcg_handle* h, const mlcg_weight_desc* w, int n) {
  if (!h) return MLCG_E_ARG;
  CK(cudaSetDevice(h->device));
  int rc = copy_weights(h, w, n, h->seer_w);
  if (rc) return rc;
  auto& m = h->seer_w;
  const char* names[7] = {"gcn1_dm", "gcn2_dm", "gcn3_dm", "gcn1", "gcn2", "gcn3", "gcn4"};
  const int seer_mode = PREC_TF32;  // the GCN always runs kind::tf32 in tensor-core modes (0.2 % of the FLOPs)
  const int ksplit = seer_split3() ? 3 : 1;  // error-compensated 3xTF32 (default): logits to fp32 accuracy
  auto prep = [&](SeerLayer& S, const std::string& key, int nn, int kk) -> int {
    int r;
    if ((r = need(h, m, key + ".weight", nn, kk, &S.w))) return r;
    if ((r = need(h, m, key + ".bias", nn, 1, &S.b))) return r;
    S.n = nn;
    S.k = kk;
    const int npad = ((nn + 255) / 256) * 256;
    if ((r = pad_vec(h, S.b_pad, S.b.d, 1, nn, npad))) return r;
    if (h->precision == PREC_FP32_SIMT) return MLCG_OK;
    const int kc = (kk + epc(seer_mode) - 1) / epc(seer_mode);
    CK(S.w_op.ensure((size_t)(npad / 256) * ksplit * kc * 256 * CHUNK_BYTES));
    PackArgs a{};
    a.src = S.w.d; a.ld = kk; a.n_real = nn; a.bn = 256; a.n_kc = ksplit * kc; a.seg_len = kc * epc(seer_mode);
    a.kreal0 = kk; a.kofs0 = 0; a.bias = nullptr; a.bias_k = -1; a.dst = S.w_op.as<uint8_t>();
    a.split3 = (ksplit == 3);
    CK(launch_pack(seer_mode, a, npad / 256, 0));
    h->launches++;
    return MLCG_OK;
  };
  for (int i = 0; i < 7; ++i) {
    const bool first = (i == 0 || i == 3);
    if ((rc = prep(h->seer_gcn[i], std::string(names[i]) + ".linear", SEER_H, first ? SEER_E : SEER_H))) return rc;
  }
  if ((rc = prep(h->seer_resize, "resize", SEER_D * SEER_NB, SEER_H))) return rc;
  Wt t;
  if ((rc = need(h, m, "nodes_embedding.weight", 36, SEER_E, &t))) return rc;
  if ((rc = need(h, m, "dm_nodes_embedding.weight", 36, SEER_E, &t))) return rc;
  if ((rc = need(h, m, "nodes_coord_fc.weight", SEER_D * SEER_E, SEER_D, &t))) return rc;
  if ((rc = need(h, m, "nodes_coord_fc.bias", SEER_D * SEER_E, 1, &t))) return rc;
  if ((rc = need(h, m, "dm_resize.weight", 1, SEER_H, &t))) return rc;
  if ((rc = need(h, m, "dm_resize.bias", 1, 1, &t))) return rc;
  CK(cudaDeviceSynchronize());
  h->seer_loaded = true;
  return MLCG_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// batch plan
// ---------------------------------------------------------------------------------------------------------------
// Host-only plan of the fused edge kernel for a batch: the tile table (section 4.1 of DESIGN.md) and the targets that go
// through the side buffer.  Pure function of (atom counts, SM count, environment switches); also exported for tests.
static int plan_edge_tiles(const int32_t* n_nodes, int B, int N, int num_sms, std::vector<EdgeTile>& tiles,
                           std::vector<int>& fix_node, std::vector<int>& node_off, std::string& err) {
  tiles.clear();
  fix_node.clear();
  node_off.assign(B + 1, 0);
  for (int b = 0; b < B; ++b) {
    const int n = n_nodes[b];
    if (n < 1 || n > N) { err = "set_batch: n_nodes[b] must be in [1, N]"; return MLCG_E_ARG; }
    node_off[b + 1] = node_off[b] + n;
    const int nm1 = n - 1, node0 = node_off[b];
    if (nm1 < EDGE_MAXG || !edge_split_mode()) {
      // few neighbours per target: whole targets per tile (a 128-row window could touch more than EDGE_MAXG targets)
      const int gmax = std::min(EDGE_MAXG, n > 1 ? TILE_M / nm1 : EDGE_MAXG);
      for (int i0 = 0; i0 < n; i0 += gmax) {
        const int ng = std::min(gmax, n - i0);
        tiles.push_back(EdgeTile{b, 0, ng * nm1, n, i0, ng, EDGE_WHOLE, EDGE_WHOLE});
      }
    } else {
      // cut the n(n-1) target-major edge rows into near-equal ranges of at most 128 rows
      const int E = n * nm1, T = (E + TILE_M - 1) / TILE_M;
      for (int k = 0; k < T; ++k) {
        const int ra = (int)((long long)k * E / T), rb = (int)((long long)(k + 1) * E / T);
        const int i_first = ra / nm1, i_last = (rb - 1) / nm1;
        // provisional: fixb = node whose neighbour list is cut at the end of this tile (resolved below)
        tiles.push_back(EdgeTile{b, ra - i_first * nm1, rb - ra, n, i_first, i_last - i_first + 1, EDGE_WHOLE,
                                 (rb % nm1 != 0) ? node0 + i_last : EDGE_WHOLE});
      }
    }
  }
  // Resolve the split targets.  The edge kernel gives every CTA a contiguous tile range (edge_tile_owner mirrors it): a
  // target cut between two tiles of one CTA is carried in shared memory, one cut between two CTAs goes through the
  // side buffer + k_edge_fixup.
  std::vector<int> owner;
  edge_tile_owner(num_sms, (int)tiles.size(), owner);
  for (size_t t = 0; t + 1 < tiles.size(); ++t) {
    if (tiles[t].fixb == EDGE_WHOLE) continue;
    const int node = tiles[t].fixb;
    if (owner[t] == owner[t + 1]) {
      tiles[t].fixb = tiles[t + 1].fixa = EDGE_CARRY;
    } else {
      tiles[t].fixb = tiles[t + 1].fixa = (int)fix_node.size();
      fix_node.push_back(node);
    }
  }
  return MLCG_OK;
}

/* Test / introspection hook (no device needed): the edge-tile plan for a batch as 8 ints per tile (EdgeTile) and the
 * CTA that owns each tile.  Returns the number of tiles (or < 0); fills at most max_tiles entries. */
extern "C" int mlcg_edge_block_order(int equivariant, int32_t* out) {
  if (!out) return MLCG_E_ARG;
  for (int b = 0; b < 3 * E3_NKC; ++b) out[b] = e3_blk(equivariant != 0, b);
  return 3 * E3_NKC;
}

extern "C" int mlcg_plan_edge_tiles(const int32_t* n_nodes, int B, int N, int num_sms, int32_t* tiles_out, int32_t* owner_out,
                                    int max_tiles, int32_t* n_fix_out) {
  if (!n_nodes || B <= 0 || N <= 0 || N > EDGE_MAXN || num_sms <= 0) return MLCG_E_ARG;
  std::vector<EdgeTile> tiles;
  std::vector<int> fix_node, node_off, owner;
  std::string err;
  const int rc = plan_edge_tiles(n_nodes, B, N, num_sms, tiles, fix_node, node_off, err);
  if (rc) return rc;
  edge_tile_owner(num_sms, (int)tiles.size(), owner);
  for (int t = 0; t < (int)tiles.size() && t < max_tiles; ++t) {
    if (tiles_out) memcpy(tiles_out + 8 * t, &tiles[t], sizeof(EdgeTile));
    if (owner_out) owner_out[t] = owner[t];
  }
  if (n_fix_out) *n_fix_out = (int)fix_node.size();
  return (int)tiles.size();
}

// Builds plan `p` for a batch (n_nodes HOST, 1 <= n_nodes[b] <= N) and grows the shared workspaces to fit it.  Synchronous
// copies on the NULL stream: the caller drains the device first and never calls it inside a stream capture.
static int build_plan(mlcg_handle* h, BatchPlan& p, const int32_t* n_nodes, int B, int N) {
  p.B = B;
  p.N = N;
  p.h_n_nodes.assign(n_nodes, n_nodes + B);
  p.h_node_off.assign(B + 1, 0);
  std::vector<int> node_mol, node_edge_off;
  std::vector<EdgeTile> tiles;
  std::vector<int> fix_node;
  {
    std::string perr;
    const int prc = plan_edge_tiles(n_nodes, B, N, h->num_sms, tiles, fix_node, p.h_node_off, perr);
    if (prc) FAIL(prc, perr.c_str());
  }
  long long edges = 0;
  for (int b = 0; b < B; ++b) {
    const int n = n_nodes[b];
    for (int i = 0; i < n; ++i) {
      node_mol.push_back(b);
      if (edges + (long long)i * (n - 1) > 0x7fffffffLL) FAIL(MLCG_E_ARG, "set_batch: too many edges for one batch");
      node_edge_off.push_back((int)(edges + (long long)i * (n - 1)));
    }
    edges += (long long)n * (n - 1);
  }
  p.n_etiles = (int)tiles.size();
  p.n_edges = edges;
  p.M = p.h_node_off[B];
  p.n_mtiles = (p.M + TILE_M - 1) / TILE_M;
  p.n_etiles = (int)tiles.size();
  const size_t mpad = (size_t)p.n_mtiles * TILE_M;
  CK(p.d_n_nodes.ensure(B * sizeof(int)));
  CK(p.d_node_off.ensure((B + 1) * sizeof(int)));
  CK(p.d_node_mol.ensure(p.M * sizeof(int)));
  CK(p.d_node_edge_off.ensure(p.M * sizeof(int)));
  CK(p.d_tiles.ensure(tiles.size() * sizeof(EdgeTile)));
  p.n_fix = (int)fix_node.size();
  CK(p.d_fix_node.ensure(std::max<size_t>(fix_node.size(), 1) * sizeof(int)));
  CK(p.fix_agg.ensure(std::max<size_t>(fix_node.size(), 1) * HP * sizeof(float)));
  CK(p.fix_dx.ensure(std::max<size_t>(fix_node.size(), 1) * 4 * sizeof(float)));
  CK(cudaMemcpy(p.d_n_nodes.p, n_nodes, B * sizeof(int), cudaMemcpyHostToDevice));
  CK(cudaMemcpy(p.d_node_off.p, p.h_node_off.data(), (B + 1) * sizeof(int), cudaMemcpyHostToDevice));
  CK(cudaMemcpy(p.d_node_mol.p, node_mol.data(), p.M * sizeof(int), cudaMemcpyHostToDevice));
  CK(cudaMemcpy(p.d_node_edge_off.p, node_edge_off.data(), p.M * sizeof(int), cudaMemcpyHostToDevice));
  CK(cudaMemcpy(p.d_tiles.p, tiles.data(), tiles.size() * sizeof(EdgeTile), cudaMemcpyHostToDevice));
  if (p.n_fix) CK(cudaMemcpy(p.d_fix_node.p, fix_node.data(), fix_node.size() * sizeof(int), cudaMemcpyHostToDevice));
  // the side buffers of split targets are zero between edge-kernel launches (k_edge_fixup re-zeroes what it consumes)
  CK(cudaMemset(p.fix_agg.p, 0, std::max<size_t>(fix_node.size(), 1) * HP * sizeof(float)));
  CK(cudaMemset(p.fix_dx.p, 0, std::max<size_t>(fix_node.size(), 1) * 4 * sizeof(float)));
  // workspaces (zero-initialised on growth; padded rows / columns are never written afterwards)
  CK(h->x0.ensure(mpad * 3 * sizeof(float)));
  CK(h->xa.ensure(mpad * 3 * sizeof(float)));
  CK(h->xb.ensure(mpad * 3 * sizeof(float)));
  CK(h->h_res.ensure(mpad * HP * sizeof(float)));
  CK(h->pq.ensure(mpad * 2 * HP * sizeof(float)));
  CK(h->t_dev.ensure(B * sizeof(float)));
  CK(h->nf_flag.ensure(sizeof(int)));
  CK(h->eps_dev.ensure((size_t)B * N * ZC * sizeof(float)));
  if (h->precision == PREC_FP32_SIMT) {
    CK(h->agg_f32.ensure(mpad * HP * sizeof(float)));
    CK(h->t_f32.ensure(mpad * HP * sizeof(float)));
    // chunk the edge list so the materialised edge activations stay bounded
    const int cap = 49152;
    p.simt_chunks.clear();
    int nb = 0;
    while (nb < p.M) {
      SimtChunk c{nb, nb, node_edge_off[nb], 0};
      while (c.node_end < p.M) {
        const int b = node_mol[c.node_end];
        const int deg = n_nodes[b] - 1;
        if (c.edge_rows + deg > cap && c.edge_rows > 0) break;
        c.edge_rows += deg;
        c.node_end++;
      }
      p.simt_chunks.push_back(c);
      nb = c.node_end;
    }
    CK(h->a1.ensure((size_t)(cap + 64) * HP * sizeof(float)));
    CK(h->m2.ensure((size_t)(cap + 64) * HP * sizeof(float)));
  } else {
    const size_t opb = (size_t)p.n_mtiles * h->kc448() * A_CHUNK_BYTES;
    CK(h->h_op.ensure(opb));
    CK(h->agg_op.ensure(opb));
    CK(h->t_op.ensure(opb));
  }
  return MLCG_OK;
}

extern "C" int mlcg_set_batch(mlcg_handle* h, const int32_t* n_nodes, int B, int N) {
  if (!h) return MLCG_E_ARG;
  if (!n_nodes || B <= 0 || N <= 0 || N > EDGE_MAXN) FAIL(MLCG_E_ARG, "set_batch: need B > 0 and 1 <= N <= 39");
  CK(cudaSetDevice(h->device));
  // The plan buffers below are rewritten with synchronous copies on the NULL stream while earlier calls may still be
  // running on the caller's (possibly non-blocking) streams: drain the device first.  set_batch is documented synchronous.
  CK(cudaDeviceSynchronize());
  // any change of the batch plan invalidates the graph captured by mlcg_generate / mlcg_generate_fragment
  if (h->gen_graph) { cudaGraphExecDestroy(h->gen_graph); h->gen_graph = nullptr; }
  h->gen_key.clear();
  h->gen_key_hits = 0;
  h->batch_set = false;
  h->pl = &h->plans[0];
  const int rc = build_plan(h, h->plans[0], n_nodes, B, N);
  if (rc) return rc;
  h->batch_set = true;
  return MLCG_OK;
}

/* 1 if any decode since the last call produced a non-finite coordinate (the trajectory diverged, or -- fp16 mode -- left the
 * fp16 range, see DESIGN.md section 3), else 0; clears the flag.  Synchronises `stream`. */
extern "C" int mlcg_nonfinite(mlcg_handle* h, void* stream) {
  if (!h || !h->nf_flag.p) return 0;
  int v = 0;
  if (cudaStreamSynchronize((cudaStream_t)stream) != cudaSuccess) return 0;
  if (cudaMemcpy(&v, h->nf_flag.p, sizeof(int), cudaMemcpyDeviceToHost) != cudaSuccess) return 0;
  if (v) cudaMemset(h->nf_flag.p, 0, sizeof(int));
  return v != 0;
}
extern "C" int mlcg_num_edge_tiles(mlcg_handle* h) { return h ? h->pl->n_etiles : -1; }
extern "C" int64_t mlcg_num_edges(mlcg_handle* h) { return h ? h->pl->n_edges : -1; }
extern "C" int64_t mlcg_kernel_launches(mlcg_handle* h) { return h ? h->launches : -1; }
extern "C" int64_t mlcg_graph_captures(mlcg_handle* h) { return h ? h->graph_captures : -1; }

// ---------------------------------------------------------------------------------------------------------------
// EGNN forward
// ---------------------------------------------------------------------------------------------------------------
static int edge_grid(mlcg_handle* h) { return edge_grid_for(h->pl->n_etiles, h->num_sms); }

static EdgeArgs edge_args(mlcg_handle* h, const LayerW& L, const float* x_cur, float* x_next) {
  EdgeArgs a{};
  a.tiles = h->pl->d_tiles.as<int4>();
  a.n_tiles = h->pl->n_etiles;
  a.fix_agg = h->pl->fix_agg.as<float>();
  a.fix_dx = h->pl->fix_dx.as<float>();
  a.node_off = h->pl->d_node_off.as<int>();
  a.pq = h->pq.p;
  a.x_cur = x_cur;
  a.x0 = h->x0.as<float>();
  a.x_next = x_next;
  a.w2 = L.w2_op.as<uint8_t>();
  a.n_kc = h->kc448();
  memcpy(a.wc, L.h_wc, sizeof(a.wc));
  memcpy(a.wd, L.h_wd, sizeof(a.wd));
  memcpy(a.wv, L.h_wv, sizeof(a.wv));
  if (is16(h->precision)) {
    const bool f16 = (h->precision == PREC_FP16);
    const float dinv = 1.0f / dist_scale(h->precision);  // the packed squared distances carry dist_scale
    auto bf = [f16, dinv](float f) -> uint32_t {  // round-to-nearest-even 16-bit pattern of the distance-column weight
      f *= dinv;
      if (f16) {
        const __half hv = __float2half_rn(f);
        unsigned short us;
        memcpy(&us, &hv, 2);
        return us;
      }
      uint32_t u;
      memcpy(&u, &f, 4);
      return (u + 0x7fffu + ((u >> 16) & 1u)) >> 16;
    };
    for (int k2 = 0; k2 < HP / 2; ++k2) {
      a.wcd_h[4 * (k2 / 2) + (k2 & 1)] = bf(L.h_wc[2 * k2]) | (bf(L.h_wc[2 * k2 + 1]) << 16);
      a.wcd_h[4 * (k2 / 2) + 2 + (k2 & 1)] = bf(L.h_wd[2 * k2]) | (bf(L.h_wd[2 * k2 + 1]) << 16);
    }
  }
  a.att_bias = L.att_bias;
  a.agg_op = h->agg_op.as<uint8_t>();
  a.agg_chunks = h->kc448();
  a.prof = nullptr;
  return a;
}

static int egnn_forward_tc(mlcg_handle* h, cudaStream_t st) {
  const int mode = h->precision, kc = h->kc448();
  const int grid_e = edge_grid(h);
  auto gemm_pq = [&](const LayerW& L) -> cudaError_t {
    GemmArgs a{};
    a.a0 = h->h_op.as<uint8_t>(); a.a0_chunks = kc; a.a0_per_tile = kc; a.n_kc = kc;
    a.w = L.w1ab_op.as<uint8_t>(); a.bias = L.bias_pq.as<float>(); a.m_rows = h->pl->M;
    a.out_f32 = h->pq.as<float>(); a.ldo = 2 * HP; a.n_valid = 2 * HP; a.rowscale = nullptr; a.relu = 0;
    // bf16 mode keeps the P/Q projections in bf16 (halves their HBM and shared-memory traffic; no accuracy cost)
    a.out_scale = act_scale(mode);  // fp16: P/Q rows are stored scaled by ACT
    if (mode == PREC_FP16) return launch_gemm<PREC_FP16, HP, EPI_BF16>(a, h->pl->n_mtiles, 2, st);
    if (mode == PREC_BF16) return launch_gemm<PREC_BF16, HP, EPI_BF16>(a, h->pl->n_mtiles, 2, st);
    return launch_gemm<PREC_TF32, HP, EPI_F32>(a, h->pl->n_mtiles, 2, st);
  };
  float* xa = h->xa.as<float>();
  float* xb = h->xb.as<float>();
  CK(gemm_pq(h->layers[0]));
  h->launches++;
  bd_mark(h, BD_PQ, st);
  for (int l = 0; l < 27; ++l) {
    const LayerW& L = h->layers[l];
    const int blk = l / 3;
    const float* x_cur = (blk & 1) ? xb : xa;
    float* x_next = (blk & 1) ? xa : xb;
    EdgeArgs ea = edge_args(h, L, x_cur, x_next);
    CK(launch_edge_mode(mode, L.equiv, ea, grid_e, st));
    h->launches++;
    bd_mark(h, L.equiv ? BD_EDGE_EQUIV : BD_EDGE_GCL, st);
    CK(launch_edge_fixup(h, mode, L.equiv, ea, st));
    bd_mark(h, BD_FIXUP, st);
    if (!L.equiv) {
      GemmArgs a{};
      a.a0 = h->h_op.as<uint8_t>(); a.a0_chunks = kc; a.a0_per_tile = kc;
      a.a1 = h->agg_op.as<uint8_t>(); a.a1_per_tile = kc; a.n_kc = 2 * kc;
      a.w = L.w3_op.as<uint8_t>(); a.bias = L.b3p.as<float>(); a.m_rows = h->pl->M;
      a.out_op = h->t_op.as<uint8_t>(); a.out_op_chunks = kc; a.out_scale = op_scale(mode);
      CK((launch_gemm_mode<HP, EPI_SILU_OP>(mode, a, h->pl->n_mtiles, 1, st)));
      h->launches++;
      bd_mark(h, BD_MLP1, st);
      GemmArgs b{};
      b.a0 = h->t_op.as<uint8_t>(); b.a0_chunks = kc; b.a0_per_tile = kc; b.n_kc = kc;
      b.w = L.w4_op.as<uint8_t>(); b.bias = L.b4p.as<float>(); b.m_rows = h->pl->M;
      b.out_op = h->h_op.as<uint8_t>(); b.out_op_chunks = kc; b.resid = h->h_res.as<float>(); b.ldr = 0;  // tiled residual layout
      b.out_scale = op_scale(mode);
      CK((launch_gemm_mode<HP, EPI_RESID_OP>(mode, b, h->pl->n_mtiles, 1, st)));
      h->launches++;
      bd_mark(h, BD_MLP2, st);
    }
    if (l + 1 < 27) {
      CK(gemm_pq(h->layers[l + 1]));
      h->launches++;
      bd_mark(h, BD_PQ, st);
    }
  }
  return MLCG_OK;
}

static int simt_gemm(mlcg_handle* h, const float* A, int lda, const float* W, int ldw, const float* bias, float* C, int ldc,
                     int M, int N, int K, int flags, const float* rowscale, cudaStream_t st) {
  if (M <= 0) return MLCG_OK;
  dim3 grid((N + 63) / 64, (M + 63) / 64);
  k_simt_gemm<<<grid, 256, 0, st>>>(A, lda, W, ldw, bias, rowscale, C, ldc, M, N, K, flags);
  KCHECK();
  return MLCG_OK;
}

static int egnn_forward_simt(mlcg_handle* h, cudaStream_t st) {
  float* xa = h->xa.as<float>();
  float* xb = h->xb.as<float>();
  float* hres = h->h_res.as<float>();
  float* pq = h->pq.as<float>();
  const int* node_mol = h->pl->d_node_mol.as<int>();
  const int* node_off = h->pl->d_node_off.as<int>();
  const int* neo = h->pl->d_node_edge_off.as<int>();
  int rc;
  for (int l = 0; l < 27; ++l) {
    const LayerW& L = h->layers[l];
    const int blk = l / 3;
    const float* x_cur = (blk & 1) ? xb : xa;
    float* x_next = (blk & 1) ? xa : xb;
    // P = h.W1[:, :420]^T ; Q = h.W1[:, 420:840]^T + b1
    if ((rc = simt_gemm(h, hres, HP, L.w1.d, 2 * HID + 2, nullptr, pq, 2 * HP, h->pl->M, HID, HID, 0, nullptr, st))) return rc;
    if ((rc = simt_gemm(h, hres, HP, L.w1.d + HID, 2 * HID + 2, L.b1.d, pq + HP, 2 * HP, h->pl->M, HID, HID, SG_BIAS, nullptr, st)))
      return rc;
    for (const SimtChunk& c : h->pl->simt_chunks) {
      const int nn = c.node_end - c.node_begin;
      k_simt_build_a1<<<nn, HP, 0, st>>>(pq, x_cur, h->x0.as<float>(), node_mol, node_off, neo, c.node_begin, c.edge_base,
                                         L.w1.d, h->a1.as<float>());
      KCHECK();
      if ((rc = simt_gemm(h, h->a1.as<float>(), HP, L.w2.d, HID, L.b2.d, h->m2.as<float>(), HP, c.edge_rows, HID, HID,
                          SG_BIAS | SG_SILU, nullptr, st)))
        return rc;
      if (L.equiv)
        k_simt_gate_agg<true><<<nn, HP, 0, st>>>(h->m2.as<float>(), L.wv.d, 0.f, node_mol, node_off, neo, c.node_begin,
                                                 c.edge_base, nullptr, 0, x_cur, x_next);
      else
        k_simt_gate_agg<false><<<nn, HP, 0, st>>>(h->m2.as<float>(), L.wv.d, L.att_bias, node_mol, node_off, neo,
                                                  c.node_begin, c.edge_base, h->agg_f32.as<float>(), HP, x_cur, x_next);
      KCHECK();
    }
    if (!L.equiv) {
      float* t = h->t_f32.as<float>();
      if ((rc = simt_gemm(h, hres, HP, L.w3.d, 2 * HID, L.b3.d, t, HP, h->pl->M, HID, HID, SG_BIAS, nullptr, st))) return rc;
      if ((rc = simt_gemm(h, h->agg_f32.as<float>(), HP, L.w3.d + HID, 2 * HID, nullptr, t, HP, h->pl->M, HID, HID,
                          SG_ACC | SG_SILU, nullptr, st)))
        return rc;
      if ((rc = simt_gemm(h, t, HP, L.w4.d, HID, L.b4.d, hres, HP, h->pl->M, HID, HID, SG_BIAS | SG_ACC, nullptr, st))) return rc;
    }
  }
  return MLCG_OK;
}

extern "C" int mlcg_egnn_forward(mlcg_handle* h, const float* t, const float* z, const float* ctx, float* eps, void* stream) {
  if (!h) return MLCG_E_ARG;
  if (!h->egnn_loaded || !h->batch_set) FAIL(MLCG_E_STATE, "egnn_forward: load weights and set the batch first");
  if (!t || !z || !ctx || !eps) FAIL(MLCG_E_ARG, "egnn_forward: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  const int kc = h->kc448();
  bd_mark(h, BD_START, st);
  if (h->precision == PREC_FP16)
    k_egnn_prepare<PREC_FP16><<<(h->pl->M + PREP_NPB - 1) / PREP_NPB, HP, 0, st>>>(z, t, ctx, h->pl->d_node_mol.as<int>(), h->pl->d_node_off.as<int>(), h->pl->N, h->pl->M, h->w_emb.d,
                                                  h->b_emb.d, h->h_res.as<float>(), 0, h->h_op.as<uint8_t>(), kc,
                                                  h->x0.as<float>(), h->xa.as<float>());
  else if (h->precision == PREC_BF16)
    k_egnn_prepare<PREC_BF16><<<(h->pl->M + PREP_NPB - 1) / PREP_NPB, HP, 0, st>>>(z, t, ctx, h->pl->d_node_mol.as<int>(), h->pl->d_node_off.as<int>(), h->pl->N, h->pl->M, h->w_emb.d,
                                                  h->b_emb.d, h->h_res.as<float>(), 0, h->h_op.as<uint8_t>(), kc,
                                                  h->x0.as<float>(), h->xa.as<float>());
  else if (h->precision == PREC_TF32)
    k_egnn_prepare<PREC_TF32><<<(h->pl->M + PREP_NPB - 1) / PREP_NPB, HP, 0, st>>>(z, t, ctx, h->pl->d_node_mol.as<int>(), h->pl->d_node_off.as<int>(), h->pl->N, h->pl->M, h->w_emb.d,
                                                  h->b_emb.d, h->h_res.as<float>(), 0, h->h_op.as<uint8_t>(), kc,
                                                  h->x0.as<float>(), h->xa.as<float>());
  else
    k_egnn_prepare<PREC_FP32_SIMT><<<(h->pl->M + PREP_NPB - 1) / PREP_NPB, HP, 0, st>>>(z, t, ctx, h->pl->d_node_mol.as<int>(), h->pl->d_node_off.as<int>(), h->pl->N, h->pl->M,
                                                       h->w_emb.d, h->b_emb.d, h->h_res.as<float>(), HP, nullptr, 0,
                                                       h->x0.as<float>(), h->xa.as<float>());
  KCHECK();
  bd_mark(h, BD_PREPARE, st);
  int rc = (h->precision == PREC_FP32_SIMT) ? egnn_forward_simt(h, st) : egnn_forward_tc(h, st);
  if (rc) return rc;
  // 9 blocks: blocks 0,2,4,6,8 write xb -> final coordinates are in xb
  k_egnn_readout<<<h->pl->B, 256, 0, st>>>(h->h_res.as<float>(), h->precision == PREC_FP32_SIMT ? HP : 0, h->xb.as<float>(), h->x0.as<float>(), h->pl->d_n_nodes.as<int>(),
                                       h->pl->d_node_off.as<int>(), h->pl->N, h->w_out.d, h->b_out.d, eps);
  KCHECK();
  bd_mark(h, BD_READOUT, st);
  return MLCG_OK;
}

/* One EGNN forward with a CUDA event after every launch: out_ms[c] = milliseconds spent in kernel class c
 * (0 prepare, 1 P/Q projections, 2 edge kernel GCL, 3 edge kernel equivariant, 4 split-target fix-ups, 5 node MLP 1,
 * 6 node MLP 2, 7 readout), out_ms[8] = whole forward, out_ms[9..16] = launches per class.  Synchronous. */
extern "C" int mlcg_egnn_forward_breakdown(mlcg_handle* h, const float* t, const float* z, const float* ctx, float* eps,
                                           double* out_ms, void* stream) {
  if (!h || !out_ms) return MLCG_E_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  h->bd_on = true;
  h->bd_ev.clear();
  int rc = mlcg_egnn_forward(h, t, z, ctx, eps, stream);
  h->bd_on = false;
  cudaError_t ce = cudaStreamSynchronize(st);
  for (int k = 0; k < 2 * BD_NCLASS + 1; ++k) out_ms[k] = 0.0;
  for (size_t i = 1; i < h->bd_ev.size(); ++i) {
    float ms = 0.f;
    cudaEventElapsedTime(&ms, h->bd_ev[i - 1].second, h->bd_ev[i].second);
    const int c = h->bd_ev[i].first;
    if (c >= 0 && c < BD_NCLASS) { out_ms[c] += ms; out_ms[BD_NCLASS + 1 + c] += 1.0; }
    out_ms[BD_NCLASS] += ms;
  }
  for (auto& e : h->bd_ev) cudaEventDestroy(e.second);
  h->bd_ev.clear();
  if (rc) return rc;
  CK(ce);
  return MLCG_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// diffusion-step kernels
// ---------------------------------------------------------------------------------------------------------------
static inline int warp_grid(int B) { return (B * 32 + 127) / 128; }

#define STEP_PROLOGUE(name)                                                                  \
  if (!h) return MLCG_E_ARG;                                                                 \
  if (!h->batch_set) FAIL(MLCG_E_STATE, name ": set the batch first");                       \
  cudaStream_t st = (cudaStream_t)stream;

extern "C" int mlcg_noise_init(mlcg_handle* h, float* z, const mlcg_noise* noise, void* stream) {
  STEP_PROLOGUE("noise_init");
  if (!z || !noise) FAIL(MLCG_E_ARG, "noise_init: null pointer");
  k_noise_init<<<warp_grid(h->pl->B), 128, 0, st>>>(z, h->pl->d_n_nodes.as<int>(), h->pl->B, h->pl->N, to_src(h, noise));
  KCHECK();
  return MLCG_OK;
}
extern "C" int mlcg_step(mlcg_handle* h, float* z, const float* eps, const mlcg_step_scalars* sc, const mlcg_noise* noise,
                         void* stream) {
  STEP_PROLOGUE("step");
  if (!z || !eps || !sc || !noise) FAIL(MLCG_E_ARG, "step: null pointer");
  k_step<<<warp_grid(h->pl->B), 128, 0, st>>>(z, eps, h->pl->d_n_nodes.as<int>(), h->pl->B, h->pl->N, sc->alpha_ts, sc->c_eps, sc->c_sigma,
                                          to_src(h, noise));
  KCHECK();
  return MLCG_OK;
}
extern "C" int mlcg_reinject(mlcg_handle* h, float* z, const float* z_known, const float* fixed_mask,
                             const mlcg_step_scalars* sc, const mlcg_noise* noise, void* stream) {
  STEP_PROLOGUE("reinject");
  if (!z || !z_known || !fixed_mask || !sc || !noise) FAIL(MLCG_E_ARG, "reinject: null pointer");
  k_reinject<<<warp_grid(h->pl->B), 128, 0, st>>>(z, z_known, fixed_mask, h->pl->d_n_nodes.as<int>(), h->pl->B, h->pl->N, sc->alpha_s,
                                              sc->sigma_s, sc->blend, to_src(h, noise));
  KCHECK();
  return MLCG_OK;
}
extern "C" int mlcg_forward_diffuse(mlcg_handle* h, float* z, const float* z_known, float alpha, float sigma,
                                    const mlcg_noise* noise, void* stream) {
  STEP_PROLOGUE("forward_diffuse");
  if (!z || !z_known || !noise) FAIL(MLCG_E_ARG, "forward_diffuse: null pointer");
  k_forward_diffuse<<<warp_grid(h->pl->B), 128, 0, st>>>(z, z_known, h->pl->d_n_nodes.as<int>(), h->pl->B, h->pl->N, alpha, sigma,
                                                     to_src(h, noise));
  KCHECK();
  return MLCG_OK;
}
extern "C" int mlcg_decode(mlcg_handle* h, const float* z0, const float* eps0, float sigma_0, float alpha_0, float sigma_x,
                           const mlcg_noise* noise, float* x, int32_t* atom_class, void* stream) {
  STEP_PROLOGUE("decode");
  if (!z0 || !eps0 || !noise || !x || !atom_class) FAIL(MLCG_E_ARG, "decode: null pointer");
  k_decode<<<warp_grid(h->pl->B), 128, 0, st>>>(z0, eps0, h->pl->d_n_nodes.as<int>(), h->pl->B, h->pl->N, sigma_0, alpha_0, sigma_x,
                                            to_src(h, noise), x, atom_class, h->nf_flag.as<int>());
  KCHECK();
  return MLCG_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// whole reverse loop
// ---------------------------------------------------------------------------------------------------------------
// The reverse loop of mlcg_sample with its noise draws numbered from `draw0` on (mlcg_sample: 0).
static int sample_loop(mlcg_handle* h, int mode, int T, const mlcg_step_scalars* steps, int resample_steps,
                       int diffusion_level, float merge_alpha, float merge_sigma, float sigma_0, float alpha_0, float sigma_x,
                       const float* ctx, const float* z_known, const float* fixed_mask, const float* noise_tape, uint64_t seed,
                       int64_t sample_offset, const int64_t* sample_ids, float* z, float* x_out, int32_t* atom_class_out,
                       float* trace_z, float* trace_eps, uint64_t draw0, void* stream) {
  STEP_PROLOGUE("sample");
  if (!h->egnn_loaded) FAIL(MLCG_E_STATE, "sample: load the EGNN weights first");
  if (mode < 0 || mode > 2 || T <= 0 || !steps || !ctx || !z || !x_out || !atom_class_out || resample_steps < 0)
    FAIL(MLCG_E_ARG, "sample: bad argument");
  if (mode != 0 && (!z_known || !fixed_mask)) FAIL(MLCG_E_ARG, "sample: inpaint / merge need z_known and fixed_mask");
  const size_t zsz = (size_t)h->pl->B * h->pl->N * ZC;
  float* eps = h->eps_dev.as<float>();
  float* tdev = h->t_dev.as<float>();
  uint64_t draw = draw0;
  long long fwd = 0;
  auto next_noise = [&]() {
    mlcg_noise n;
    n.raw = noise_tape ? noise_tape + (size_t)draw * zsz : nullptr;
    n.seed = seed;
    n.draw = draw;
    n.sample_offset = sample_offset;
    n.sample_ids = sample_ids;
    ++draw;
    return n;
  };
  auto network = [&](float tval) -> int {
    k_fill_f32<<<(h->pl->B + 127) / 128, 128, 0, st>>>(tdev, tval, h->pl->B);
    KCHECK();
    if (trace_z) CK(cudaMemcpyAsync(trace_z + (size_t)fwd * zsz, z, zsz * sizeof(float), cudaMemcpyDeviceToDevice, st));
    int rc = mlcg_egnn_forward(h, tdev, z, ctx, eps, stream);
    if (rc) return rc;
    if (trace_eps) CK(cudaMemcpyAsync(trace_eps + (size_t)fwd * zsz, eps, zsz * sizeof(float), cudaMemcpyDeviceToDevice, st));
    ++fwd;
    return MLCG_OK;
  };
  auto denoise = [&](int s) -> int {
    int rc = network(steps[s].t);
    if (rc) return rc;
    mlcg_noise n = next_noise();
    return mlcg_step(h, z, eps, &steps[s], &n, stream);
  };
  auto reinject = [&](int s) -> int {
    mlcg_noise n = next_noise();
    return mlcg_reinject(h, z, z_known, fixed_mask, &steps[s], &n, stream);
  };
  int rc;
  if (mode == 2) {
    mlcg_noise n = next_noise();
    if ((rc = mlcg_forward_diffuse(h, z, z_known, merge_alpha, merge_sigma, &n, stream))) return rc;
  } else {
    mlcg_noise n = next_noise();
    if ((rc = mlcg_noise_init(h, z, &n, stream))) return rc;
  }
  const int r_eff = (mode == 0) ? resample_steps : std::max(resample_steps, 1);
  for (int s = T - 1; s >= 0; --s) {
    if (mode == 2 && s > diffusion_level) continue;
    if (mode == 0) {
      for (int r = 0; r <= r_eff; ++r)
        if ((rc = denoise(s))) return rc;
    } else {
      for (int r = 0; r < r_eff; ++r) {
        if ((rc = denoise(s))) return rc;
        if ((rc = reinject(s))) return rc;
      }
      if (mode == 1 && (rc = denoise(s))) return rc;
    }
  }
  if ((rc = network(0.0f))) return rc;
  mlcg_noise n = next_noise();
  return mlcg_decode(h, z, eps, sigma_0, alpha_0, sigma_x, &n, x_out, atom_class_out, stream);
}

extern "C" int mlcg_sample(mlcg_handle* h, int mode, int T, const mlcg_step_scalars* steps, int resample_steps,
                           int diffusion_level, float merge_alpha, float merge_sigma, float sigma_0, float alpha_0,
                           float sigma_x, const float* ctx, const float* z_known, const float* fixed_mask,
                           const float* noise_tape, uint64_t seed, int64_t sample_offset, const int64_t* sample_ids, float* z,
                           float* x_out, int32_t* atom_class_out, float* trace_z, float* trace_eps, void* stream) {
  return sample_loop(h, mode, T, steps, resample_steps, diffusion_level, merge_alpha, merge_sigma, sigma_0, alpha_0, sigma_x,
                     ctx, z_known, fixed_mask, noise_tape, seed, sample_offset, sample_ids, z, x_out, atom_class_out, trace_z,
                     trace_eps, 0, stream);
}

// ---------------------------------------------------------------------------------------------------------------
// AdjMatSeer
// ---------------------------------------------------------------------------------------------------------------
extern "C" int mlcg_seer_inputs(mlcg_handle* h, const float* x, const int32_t* atom_class, int32_t* elements, float* dist,
                                float* adj, void* stream) {
  STEP_PROLOGUE("seer_inputs");
  if (!x || !atom_class || !elements || !dist || !adj) FAIL(MLCG_E_ARG, "seer_inputs: null pointer");
  k_seer_inputs<<<h->pl->B, 128, 0, st>>>(x, atom_class, h->pl->d_n_nodes.as<int>(), h->pl->N, elements, dist, adj);
  KCHECK();
  return MLCG_OK;
}

static int seer_chunk(mlcg_handle* h, const int32_t* elements, const float* dist, const float* adj, float* logits,
                      int8_t* bonds, int B, cudaStream_t st) {
  const int R = B * SEER_D;
  const int mt = (R + TILE_M - 1) / TILE_M;
  const size_t rpad = (size_t)mt * TILE_M;
  const bool simt = (h->precision == PREC_FP32_SIMT);
  const int mode = PREC_TF32;
  const int kcH = SEER_H / epc(mode), kcE = SEER_E / epc(mode);
  const int split3 = (!simt && seer_split3()) ? 1 : 0, ks = split3 ? 3 : 1;
  auto& m = h->seer_w;
  CK(h->s_ld.ensure((size_t)B * SEER_D * SEER_D * 4));
  CK(h->s_la.ensure((size_t)B * SEER_D * SEER_D * 4));
  CK(h->s_rowd.ensure(rpad * 4));
  CK(h->s_rowa.ensure(rpad * 4));
  CK(h->s_x64.ensure(rpad * SEER_E * 4));
  CK(h->s_x.ensure(rpad * SEER_H * 4));
  CK(h->s_emb.ensure(rpad * 4));
  CK(h->s_add.ensure(rpad * SEER_E * 4));
  CK(h->s_raw.ensure(rpad * 224 * 4));
  if (simt) CK(h->s_y_f32.ensure(rpad * SEER_H * 4));
  else CK(h->s_y_op.ensure((size_t)mt * ks * kcH * A_CHUNK_BYTES));
  k_lnorm<<<B, 64, 0, st>>>(dist, h->s_ld.as<float>(), h->s_rowd.as<float>());
  KCHECK();
  k_lnorm<<<B, 64, 0, st>>>(adj, h->s_la.as<float>(), h->s_rowa.as<float>());
  KCHECK();
  float* X = h->s_x.as<float>();
  auto conv = [&](SeerLayer& S, const float* L, const float* lrow, const float* xin, int C) -> int {
    // Y = L.X ; X <- relu(Y.W^T + rowsum(L) b)
    dim3 g(B, (C + 127) / 128);
    if (simt) {
      k_lmul<PREC_FP32_SIMT><<<g, 128, 0, st>>>(L, xin, C, h->s_y_f32.as<float>(), nullptr, 0);
      KCHECK();
      return simt_gemm(h, h->s_y_f32.as<float>(), C, S.w.d, S.k, S.b.d, X, SEER_H, R, SEER_H, S.k, SG_BIAS | SG_RELU, lrow, st);
    }
    const int kc = (C == SEER_E) ? kcE : kcH;
    k_lmul<PREC_TF32><<<g, 128, 0, st>>>(L, xin, C, nullptr, h->s_y_op.as<uint8_t>(), kc, split3);
    KCHECK();
    GemmArgs a{};
    a.a0 = h->s_y_op.as<uint8_t>(); a.a0_chunks = ks * kc; a.a0_per_tile = ks * kc; a.n_kc = ks * kc;
    a.w = S.w_op.as<uint8_t>(); a.bias = S.b_pad.as<float>(); a.m_rows = R;
    a.out_f32 = X; a.ldo = SEER_H; a.n_valid = SEER_H; a.rowscale = lrow; a.relu = 1;
    CK((launch_gemm<PREC_TF32, 256, EPI_F32>(a, mt, SEER_H / 256, st)));
    h->launches++;
    return MLCG_OK;
  };
  int rc;
  const int eg = (R * SEER_E + 255) / 256;
  k_seer_embed<<<eg, 256, 0, st>>>(elements, m["dm_nodes_embedding.weight"].d, nullptr, h->s_x64.as<float>(), R);
  KCHECK();
  if ((rc = conv(h->seer_gcn[0], h->s_ld.as<float>(), h->s_rowd.as<float>(), h->s_x64.as<float>(), SEER_E))) return rc;
  if ((rc = conv(h->seer_gcn[1], h->s_ld.as<float>(), h->s_rowd.as<float>(), X, SEER_H))) return rc;
  if ((rc = conv(h->seer_gcn[2], h->s_ld.as<float>(), h->s_rowd.as<float>(), X, SEER_H))) return rc;
  k_seer_bottleneck<<<(R * 32 + 127) / 128, 128, 0, st>>>(X, m["dm_resize.weight"].d, m["dm_resize.bias"].d,
                                                          h->s_emb.as<float>(), R);
  KCHECK();
  k_seer_coord_fc<<<B, 256, 0, st>>>(h->s_emb.as<float>(), m["nodes_coord_fc.weight"].d, m["nodes_coord_fc.bias"].d,
                                     h->s_add.as<float>(), B);
  KCHECK();
  k_seer_embed<<<eg, 256, 0, st>>>(elements, m["nodes_embedding.weight"].d, h->s_add.as<float>(), h->s_x64.as<float>(), R);
  KCHECK();
  if ((rc = conv(h->seer_gcn[3], h->s_la.as<float>(), h->s_rowa.as<float>(), h->s_x64.as<float>(), SEER_E))) return rc;
  for (int i = 4; i < 7; ++i)
    if ((rc = conv(h->seer_gcn[i], h->s_la.as<float>(), h->s_rowa.as<float>(), X, SEER_H))) return rc;
  // resize: plain Linear 2048 -> 210
  float* raw = h->s_raw.as<float>();
  if (simt) {
    if ((rc = simt_gemm(h, X, SEER_H, h->seer_resize.w.d, SEER_H, h->seer_resize.b.d, raw, 224, R, SEER_D * SEER_NB, SEER_H,
                        SG_BIAS, nullptr, st)))
      return rc;
  } else {
    const long long pieces = (long long)R * kcH * 8;
    k_rowmajor_to_op<PREC_TF32><<<(unsigned)((pieces + 255) / 256), 256, 0, st>>>(X, SEER_H, R, SEER_H, h->s_y_op.as<uint8_t>(), kcH,
                                                                                  split3);
    KCHECK();
    GemmArgs a{};
    a.a0 = h->s_y_op.as<uint8_t>(); a.a0_chunks = ks * kcH; a.a0_per_tile = ks * kcH; a.n_kc = ks * kcH;
    a.w = h->seer_resize.w_op.as<uint8_t>(); a.bias = h->seer_resize.b_pad.as<float>(); a.m_rows = R;
    a.out_f32 = raw; a.ldo = 224; a.n_valid = SEER_D * SEER_NB; a.rowscale = nullptr; a.relu = 0;
    CK((launch_gemm<PREC_TF32, 256, EPI_F32>(a, mt, 1, st)));
    h->launches++;
  }
  k_seer_symmetrise<<<B, 256, 0, st>>>(raw, 224, logits, bonds);
  KCHECK();
  return MLCG_OK;
}

extern "C" int mlcg_seer_forward(mlcg_handle* h, const int32_t* elements, const float* dist, const float* adj, float* logits,
                                 int8_t* bonds, int B, void* stream) {
  if (!h) return MLCG_E_ARG;
  if (!h->seer_loaded) FAIL(MLCG_E_STATE, "seer_forward: load the AdjMatSeer weights first");
  if (!elements || !dist || !adj || B <= 0 || (!logits && !bonds)) FAIL(MLCG_E_ARG, "seer_forward: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  const int chunk = 3072;
  for (int b0 = 0; b0 < B; b0 += chunk) {
    const int nb = std::min(chunk, B - b0);
    const size_t o2 = (size_t)b0 * SEER_D * SEER_D;
    int rc = seer_chunk(h, elements + (size_t)b0 * SEER_D, dist + o2, adj + o2, logits ? logits + o2 * SEER_NB : nullptr,
                        bonds ? bonds + o2 : nullptr, nb, st);
    if (rc) return rc;
  }
  return MLCG_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// end-to-end with host buffers
// ---------------------------------------------------------------------------------------------------------------
// GCN inputs + GCN on the decoded batch in g_x / g_cls (active plan) -> g_bonds.
static int seer_device(mlcg_handle* h, void* stream) {
  int rc = mlcg_seer_inputs(h, h->g_x.as<float>(), h->g_cls.as<int32_t>(), h->g_el.as<int32_t>(), h->g_dist.as<float>(),
                            h->g_adj.as<float>(), stream);
  if (rc) return rc;
  return mlcg_seer_forward(h, h->g_el.as<int32_t>(), h->g_dist.as<float>(), h->g_adj.as<float>(), nullptr,
                           h->g_bonds.as<int8_t>(), h->pl->B, stream);
}

// The device part of mlcg_generate: reverse loop + GCN inputs + GCN.  Pure kernel / async-copy sequence on `stream`
// (no allocation, no synchronisation once the workspaces exist), hence capturable into a CUDA graph.
static int generate_device(mlcg_handle* h, int T, const mlcg_step_scalars* steps, int resample_steps, float sigma_0,
                           float alpha_0, float sigma_x, uint64_t seed, int64_t sample_offset, void* stream) {
  int rc = mlcg_sample(h, 0, T, steps, resample_steps, 0, 0.f, 0.f, sigma_0, alpha_0, sigma_x, h->g_ctx.as<float>(), nullptr,
                       nullptr, nullptr, seed, sample_offset, h->g_ids.as<int64_t>(), h->g_z.as<float>(), h->g_x.as<float>(),
                       h->g_cls.as<int32_t>(), nullptr, nullptr, stream);
  if (rc) return rc;
  return seer_device(h, stream);
}

static inline long long fbits(float f) {
  int32_t i;
  memcpy(&i, &f, 4);
  return (long long)i;
}

// Host side shared by mlcg_generate and mlcg_generate_fragment.  `key` holds everything the device sequence bakes into
// kernel arguments.  A new key rebuilds the batch plan (mlcg_set_batch: plan 0 = n_nodes_host / N, plus plan 1 =
// plan1_n_nodes / plan1_N when given) and drops the captured graph.  Every call uploads the per-call inputs -- context,
// sample ids, {seed, sample_offset}, and whatever `upload(stream)` adds -- to handle-owned device buffers, then runs
// `device(stream)`: eagerly on the first call with a key, captured into a CUDA graph on the second, replayed from then on.
// The outputs are copied to x_out / atom_class_out / bonds_out (pinned host or device) and the stream is synchronised.
template <class Upload, class Device>
static int generate_graphed(mlcg_handle* h, const std::vector<long long>& key, const int32_t* n_nodes_host, int B, int N,
                            const int32_t* plan1_n_nodes, int plan1_N, const float* ctx_host, uint64_t seed,
                            int64_t sample_offset, const int64_t* sample_ids_host, float* x_out, int32_t* atom_class_out,
                            int8_t* bonds_out, void* stream, Upload upload, Device device) {
  CK(cudaSetDevice(h->device));  // the call may come from any host thread (pipeline.GenerationPipeline's feeder)
  cudaStream_t st = (cudaStream_t)stream;
  if (st == nullptr) {
    // the legacy NULL stream cannot be captured; the call is synchronous and takes host buffers, so run it on a
    // private stream
    if (h->own_stream == nullptr) CK(cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking));
    CK(cudaDeviceSynchronize());
    st = h->own_stream;
    stream = (void*)st;
  }
  const bool same = (key == h->gen_key);
  if (!same) {
    int rc = mlcg_set_batch(h, n_nodes_host, B, N);  // also drops any previously captured graph
    if (rc) return rc;
    // set_batch drained the device: plan 1 may be rewritten too (outside any capture)
    if (plan1_n_nodes && (rc = build_plan(h, h->plans[1], plan1_n_nodes, B, plan1_N))) return rc;
    h->gen_key = key;
  }
  h->gen_key_hits++;
  const size_t bn = (size_t)B * N, dd = (size_t)B * SEER_D * SEER_D;
  CK(h->g_ctx.ensure((size_t)B * 3 * 4));
  CK(h->g_z.ensure(bn * ZC * 4));
  CK(h->g_x.ensure(bn * 3 * 4));
  CK(h->g_cls.ensure(bn * 4));
  CK(h->g_el.ensure((size_t)B * SEER_D * 4));
  CK(h->g_dist.ensure(dd * 4));
  CK(h->g_adj.ensure(dd * 4));
  CK(h->g_bonds.ensure(dd));
  CK(h->noise_ctl.ensure(2 * sizeof(unsigned long long)));
  CK(h->g_ids.ensure((size_t)B * sizeof(int64_t)));
  // global sample ids (the RNG key): always read from this device buffer, so a captured graph replays with any ids
  h->ids_stage.resize((size_t)B);
  for (int b = 0; b < B; ++b) h->ids_stage[b] = sample_ids_host ? sample_ids_host[b] : sample_offset + b;
  static int graphs_enabled = -1;
  if (graphs_enabled < 0) {
    const char* e = getenv("MLCG_GRAPH");
    graphs_enabled = (e == nullptr) ? 1 : (atoi(e) != 0);
  }
  CK(cudaMemcpyAsync(h->g_ctx.p, ctx_host, (size_t)B * 3 * 4, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(h->g_ids.p, h->ids_stage.data(), (size_t)B * sizeof(int64_t), cudaMemcpyHostToDevice, st));
  const unsigned long long ctl[2] = {(unsigned long long)seed, (unsigned long long)sample_offset};
  CK(cudaMemcpyAsync(h->noise_ctl.p, ctl, sizeof(ctl), cudaMemcpyHostToDevice, st));
  int rc = upload(st);
  if (rc) return rc;
  h->use_noise_ctl = true;  // the noise kernels read {seed, sample_offset} from device memory (graph-replayable)
  if (graphs_enabled && h->gen_graph == nullptr && h->gen_key_hits >= 2) {
    // second call with this key: all workspaces exist and every kernel attribute has been set by the eager first call,
    // so the launch sequence can be captured
    cudaGraph_t graph = nullptr;
    const long long launches0 = h->launches;
    CK(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
    rc = device(stream);
    cudaError_t ce = cudaStreamEndCapture(st, &graph);
    if (rc == MLCG_OK && ce == cudaSuccess && graph != nullptr) {
      ce = cudaGraphInstantiate(&h->gen_graph, graph, 0);
      if (ce != cudaSuccess) h->gen_graph = nullptr;
    }
    if (graph) cudaGraphDestroy(graph);
    if (h->gen_graph != nullptr) h->graph_captures++;
    h->gen_graph_launches = h->launches - launches0;
    h->launches = launches0;  // nothing has run yet
    if (rc != MLCG_OK || h->gen_graph == nullptr) {
      cudaGetLastError();
      h->use_noise_ctl = false;
      if (rc == MLCG_OK) FAIL(MLCG_E_STATE, "generate: CUDA graph capture failed");
      return rc;
    }
  }
  if (h->gen_graph != nullptr) {
    CK(cudaGraphLaunch(h->gen_graph, st));
    h->launches += h->gen_graph_launches;
  } else {
    rc = device(stream);
  }
  h->use_noise_ctl = false;
  if (rc) return rc;
  // the outputs may be pinned host buffers or device buffers (multi-GPU driver: results stay on the device for the gather)
  CK(cudaMemcpyAsync(x_out, h->g_x.p, bn * 3 * 4, cudaMemcpyDefault, st));
  CK(cudaMemcpyAsync(atom_class_out, h->g_cls.p, bn * 4, cudaMemcpyDefault, st));
  CK(cudaMemcpyAsync(bonds_out, h->g_bonds.p, dd, cudaMemcpyDefault, st));
  CK(cudaStreamSynchronize(st));
  return MLCG_OK;
}

extern "C" int mlcg_generate(mlcg_handle* h, const int32_t* n_nodes_host, int B, int N, const float* ctx_host, int T,
                             const mlcg_step_scalars* steps, int resample_steps, float sigma_0, float alpha_0, float sigma_x,
                             uint64_t seed, int64_t sample_offset, const int64_t* sample_ids_host, float* x_host,
                             int32_t* atom_class_host, int8_t* bonds_host, void* stream) {
  if (!h) return MLCG_E_ARG;
  if (!h->egnn_loaded || !h->seer_loaded) FAIL(MLCG_E_STATE, "generate: load both weight sets first");
  if (!n_nodes_host || !ctx_host || !steps || !x_host || !atom_class_host || !bonds_host) FAIL(MLCG_E_ARG, "generate: null pointer");
  // Key of the captured graph: batch geometry, schedule and every scalar baked into kernel arguments.
  std::vector<long long> key;
  key.reserve((size_t)B + 8 * (size_t)T + 16);
  key.push_back(B); key.push_back(N); key.push_back(T); key.push_back(resample_steps); key.push_back(h->precision);
  key.push_back(fbits(sigma_0)); key.push_back(fbits(alpha_0)); key.push_back(fbits(sigma_x));
  for (int b = 0; b < B; ++b) key.push_back(n_nodes_host[b]);
  for (int s = 0; s < T; ++s) {
    key.push_back(fbits(steps[s].t)); key.push_back(fbits(steps[s].alpha_ts)); key.push_back(fbits(steps[s].c_eps));
    key.push_back(fbits(steps[s].c_sigma));
  }
  return generate_graphed(
      h, key, n_nodes_host, B, N, nullptr, 0, ctx_host, seed, sample_offset, sample_ids_host, x_host, atom_class_host,
      bonds_host, stream, [](cudaStream_t) { return (int)MLCG_OK; },
      [&](void* s) { return generate_device(h, T, steps, resample_steps, sigma_0, alpha_0, sigma_x, seed, sample_offset, s); });
}

// Draw numbering of the merge loop of inertial fragment matching.  It starts at 0 like the first loop's, so both loops
// draw the same normals per (sample, atom, draw) -- exactly what the eager composition
// (MLConformerGenerator.edm_sample_tensors: two mlcg_sample calls) does, which this path reproduces bit for bit.
static const uint64_t kMergeDrawBase = 0;

// The device part of mlcg_generate_fragment_jobs (see mlcg.h): the launch sequence of the eager composition, on plan 0
// (whole molecules) and -- mode 2 -- plan 1 (the atoms still to be generated, stride Ng).  The plan switches happen on the
// host between launches; each launch bakes in the pointers of its plan, so one captured graph holds both loops.
static int generate_fragment_device(mlcg_handle* h, int mode, int Ng, const IfmNorms& nrm, int T,
                                    const mlcg_step_scalars* steps, int resample_steps, int diffusion_level, float merge_alpha,
                                    float merge_sigma, float sigma_0, float alpha_0, float sigma_x, uint64_t seed,
                                    int64_t sample_offset, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  const int B = h->plans[0].B, N = h->plans[0].N;
  const int64_t* ids = h->g_ids.as<int64_t>();
  const int* job = h->f_job.as<int>();
  const FragJob* jobs = h->f_jobs.as<FragJob>();
  float* zk = h->f_zk.as<float>();
  float* fm = h->f_fm.as<float>();
  int rc;
  if (mode == 1) {
    // z_known / fixed_mask of EquivariantDiffusion.inpaint (prepare_fragment): the merge-input kernel with no generated atoms
    k_ifm_merge_inputs<<<B, 64, 0, st>>>(nullptr, nullptr, nullptr, nullptr, h->f_ffx.as<float>(), h->f_ffh.as<float>(), job,
                                         jobs, 0, N, zk, fm);
    KCHECK();
    rc = sample_loop(h, 1, T, steps, resample_steps, diffusion_level, 0.f, 0.f, sigma_0, alpha_0, sigma_x, h->g_ctx.as<float>(),
                     zk, fm, nullptr, seed, sample_offset, ids, h->g_z.as<float>(), h->g_x.as<float>(), h->g_cls.as<int32_t>(),
                     nullptr, nullptr, 0, stream);
    if (rc) return rc;
    return seer_device(h, stream);
  }
  // inertial fragment matching: per-sample context of the atoms still to be generated ...
  k_ifm_context<<<(B + 127) / 128, 128, 0, st>>>(h->plans[0].d_n_nodes.as<int>(), job, jobs, B, nrm, h->f_ctx.as<float>(),
                                                 h->f_shift.as<float>(), h->f_rot.as<float>(), h->f_ngen.as<int>());
  KCHECK();
  // ... generated on their own (plan 1) ...
  h->pl = &h->plans[1];
  rc = sample_loop(h, 0, T, steps, resample_steps, diffusion_level, 0.f, 0.f, sigma_0, alpha_0, sigma_x, h->f_ctx.as<float>(),
                   nullptr, nullptr, nullptr, seed, sample_offset, ids, h->g_z.as<float>(), h->f_xg.as<float>(),
                   h->f_clsg.as<int32_t>(), nullptr, nullptr, 0, stream);
  h->pl = &h->plans[0];
  if (rc) return rc;
  // ... moved back to the reference frame next to the fixed fragment, and merged with it (plan 0)
  k_ifm_merge_inputs<<<B, 64, 0, st>>>(h->f_xg.as<float>(), h->f_clsg.as<int32_t>(), h->f_shift.as<float>(), h->f_rot.as<float>(),
                                       h->f_ffx.as<float>(), h->f_ffh.as<float>(), job, jobs, Ng, N, zk, fm);
  KCHECK();
  rc = sample_loop(h, 2, T, steps, resample_steps, diffusion_level, merge_alpha, merge_sigma, sigma_0, alpha_0, sigma_x,
                   h->g_ctx.as<float>(), zk, fm, nullptr, seed, sample_offset, ids, h->g_z.as<float>(), h->g_x.as<float>(),
                   h->g_cls.as<int32_t>(), nullptr, nullptr, kMergeDrawBase, stream);
  if (rc) return rc;
  return seer_device(h, stream);
}

extern "C" int mlcg_generate_fragment_jobs(mlcg_handle* h, const mlcg_fragment_jobs* fj, const int32_t* n_nodes_host, int B,
                                           int N, const float* ctx_host, int T, const mlcg_step_scalars* steps,
                                           int resample_steps, float sigma_0, float alpha_0, float sigma_x, uint64_t seed,
                                           int64_t sample_offset, const int64_t* sample_ids_host, float* x_out,
                                           int32_t* atom_class_out, int8_t* bonds_out, void* stream) {
  if (!h) return MLCG_E_ARG;
  if (!h->egnn_loaded || !h->seer_loaded) FAIL(MLCG_E_ARG, "generate_fragment: load both weight sets first");
  if (!fj || !n_nodes_host || !ctx_host || !steps || !x_out || !atom_class_out || !bonds_out || !fj->job_of_sample_host ||
      !fj->n_ff_host || !fj->ff_x_host || !fj->ff_h_host)
    FAIL(MLCG_E_ARG, "generate_fragment: null pointer");
  const int mode = fj->mode, n_jobs = fj->n_jobs;
  if (mode != 1 && mode != 2) FAIL(MLCG_E_ARG, "generate_fragment: mode must be 1 (inpaint) or 2 (inertial fragment matching)");
  if (mode == 2 && (!fj->moi_gen_origin_host || !fj->ff_weighted_com_host || !fj->norm_mean_host || !fj->norm_mad_host))
    FAIL(MLCG_E_ARG, "generate_fragment: null pointer (inertial fragment matching needs the moment-of-inertia prologue)");
  if (B <= 0 || N <= 0 || N > EDGE_MAXN || T <= 0 || resample_steps < 0 || n_jobs < 1)
    FAIL(MLCG_E_ARG, "generate_fragment: need B > 0, 1 <= N <= 39, T > 0, resample_steps >= 0 and n_jobs >= 1");
  // the job table: each job's fragment rows in the packed ff_x / ff_h and its prologue
  std::vector<FragJob> jobs((size_t)n_jobs);
  int n_ff_total = 0;
  for (int j = 0; j < n_jobs; ++j) {
    const int n_ff = fj->n_ff_host[j];
    if (n_ff < 1) FAIL(MLCG_E_ARG, "generate_fragment: the fragment needs at least one atom (job " + std::to_string(j) + ")");
    if (N - n_ff < 1) FAIL(MLCG_E_ARG, "generate_fragment: the fragment must have fewer atoms than N (job " + std::to_string(j) + ")");
    FragJob& q = jobs[j];
    q.n_ff = n_ff;
    q.ff_off = n_ff_total;
    n_ff_total += n_ff;
    if (mode == 2) {
      memcpy(q.moi0, fj->moi_gen_origin_host + (size_t)j * 9, sizeof(q.moi0));
      memcpy(q.ffsum, fj->ff_weighted_com_host + (size_t)j * 3, sizeof(q.ffsum));
    }
  }
  // per sample: its job's fragment size, which must leave at least one atom to generate
  std::vector<int32_t> n_ff_of((size_t)B), n_gen;
  int min_n_ff = N;
  for (int b = 0; b < B; ++b) {
    const int j = fj->job_of_sample_host[b];
    if (j < 0 || j >= n_jobs) FAIL(MLCG_E_ARG, "generate_fragment: job index out of range (sample " + std::to_string(b) + ")");
    n_ff_of[b] = jobs[j].n_ff;
    if (n_ff_of[b] >= n_nodes_host[b])
      FAIL(MLCG_E_ARG, "generate_fragment: the fragment must have fewer atoms than every sample (sample " + std::to_string(b) + ")");
    min_n_ff = std::min(min_n_ff, (int)n_ff_of[b]);
  }
  // first IFM loop: the atoms still to be generated, padded to the longest of them
  const int Ng = N - min_n_ff;
  IfmNorms nrm{};
  if (mode == 2) {
    memcpy(nrm.mean, fj->norm_mean_host, sizeof(nrm.mean));
    memcpy(nrm.mad, fj->norm_mad_host, sizeof(nrm.mad));
    n_gen.resize(B);
    for (int b = 0; b < B; ++b) n_gen[b] = n_nodes_host[b] - n_ff_of[b];
  }
  // Key of the captured graph: the geometry and every scalar baked into kernel arguments.  It starts with -mode, so it
  // never equals a key of mlcg_generate (which starts with B).  The job count and the packed fragment length fix the sizes
  // of the buffers the graph reads.  The fragments, the job table, the job of every sample, the context, the ids and
  // {seed, sample_offset} are uploaded on every call, so a replay with other references or fragments of the same sizes
  // reuses the graph and never sees a previous call's inputs.
  std::vector<long long> key;
  key.reserve(2 * (size_t)B + 7 * (size_t)T + 32);
  key.push_back(-mode); key.push_back(B); key.push_back(N); key.push_back(T); key.push_back(resample_steps);
  key.push_back(h->precision); key.push_back(n_jobs); key.push_back(n_ff_total);
  key.push_back(fbits(sigma_0)); key.push_back(fbits(alpha_0)); key.push_back(fbits(sigma_x));
  if (mode == 2) {
    key.push_back(fj->diffusion_level); key.push_back(fbits(fj->merge_alpha)); key.push_back(fbits(fj->merge_sigma));
    for (int c = 0; c < 3; ++c) { key.push_back(fbits(nrm.mean[c])); key.push_back(fbits(nrm.mad[c])); }
  }
  for (int b = 0; b < B; ++b) key.push_back(n_nodes_host[b]);
  for (int b = 0; b < B; ++b) key.push_back(n_ff_of[b]);
  for (int s = 0; s < T; ++s) {
    const mlcg_step_scalars& c = steps[s];
    for (float v : {c.t, c.alpha_ts, c.c_eps, c.c_sigma, c.alpha_s, c.sigma_s, c.blend}) key.push_back(fbits(v));
  }
  const size_t bn = (size_t)B * N, bg = (size_t)B * Ng;
  auto upload = [&](cudaStream_t st) -> int {
    CK(h->f_ffx.ensure((size_t)n_ff_total * 3 * 4));
    CK(h->f_ffh.ensure((size_t)n_ff_total * 8 * 4));
    CK(h->f_jobs.ensure((size_t)n_jobs * sizeof(FragJob)));
    CK(h->f_job.ensure((size_t)B * 4));
    CK(h->f_zk.ensure(bn * ZC * 4));
    CK(h->f_fm.ensure(bn * 4));
    if (mode == 2) {
      CK(h->f_ctx.ensure((size_t)B * 3 * 4));
      CK(h->f_shift.ensure((size_t)B * 3 * 4));
      CK(h->f_rot.ensure((size_t)B * 9 * 4));
      CK(h->f_ngen.ensure((size_t)B * 4));
      CK(h->f_xg.ensure(bg * 3 * 4));
      CK(h->f_clsg.ensure(bg * 4));
    }
    CK(cudaMemcpyAsync(h->f_ffx.p, fj->ff_x_host, (size_t)n_ff_total * 3 * 4, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(h->f_ffh.p, fj->ff_h_host, (size_t)n_ff_total * 8 * 4, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(h->f_jobs.p, jobs.data(), (size_t)n_jobs * sizeof(FragJob), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(h->f_job.p, fj->job_of_sample_host, (size_t)B * 4, cudaMemcpyHostToDevice, st));
    return MLCG_OK;
  };
  const int diffusion_level = mode == 2 ? fj->diffusion_level : 0;
  const float merge_alpha = mode == 2 ? fj->merge_alpha : 0.f, merge_sigma = mode == 2 ? fj->merge_sigma : 0.f;
  return generate_graphed(h, key, n_nodes_host, B, N, mode == 2 ? n_gen.data() : nullptr, Ng, ctx_host, seed, sample_offset,
                          sample_ids_host, x_out, atom_class_out, bonds_out, stream, upload, [&](void* s) {
                            return generate_fragment_device(h, mode, Ng, nrm, T, steps, resample_steps, diffusion_level,
                                                            merge_alpha, merge_sigma, sigma_0, alpha_0, sigma_x, seed,
                                                            sample_offset, s);
                          });
}

// One fragment for every sample: the one-job case of mlcg_generate_fragment_jobs.
extern "C" int mlcg_generate_fragment(mlcg_handle* h, const mlcg_fragment* frag, const int32_t* n_nodes_host, int B, int N,
                                      const float* ctx_host, int T, const mlcg_step_scalars* steps, int resample_steps,
                                      float sigma_0, float alpha_0, float sigma_x, uint64_t seed, int64_t sample_offset,
                                      const int64_t* sample_ids_host, float* x_out, int32_t* atom_class_out, int8_t* bonds_out,
                                      void* stream) {
  if (!h) return MLCG_E_ARG;
  if (!frag) FAIL(MLCG_E_ARG, "generate_fragment: null pointer");
  std::vector<int32_t> job_of_sample((size_t)std::max(B, 1), 0);  // never empty: B <= 0 fails the B check
  mlcg_fragment_jobs fj{};
  fj.mode = frag->mode;
  fj.n_jobs = 1;
  fj.job_of_sample_host = job_of_sample.data();
  fj.n_ff_host = &frag->n_ff;
  fj.ff_x_host = frag->ff_x_host;
  fj.ff_h_host = frag->ff_h_host;
  fj.diffusion_level = frag->diffusion_level;
  fj.merge_alpha = frag->merge_alpha;
  fj.merge_sigma = frag->merge_sigma;
  fj.moi_gen_origin_host = frag->moi_gen_origin_host;
  fj.ff_weighted_com_host = frag->ff_weighted_com_host;
  fj.norm_mean_host = frag->norm_mean_host;
  fj.norm_mad_host = frag->norm_mad_host;
  return mlcg_generate_fragment_jobs(h, &fj, n_nodes_host, B, N, ctx_host, T, steps, resample_steps, sigma_0, alpha_0,
                                     sigma_x, seed, sample_offset, sample_ids_host, x_out, atom_class_out, bonds_out, stream);
}

// ---------------------------------------------------------------------------------------------------------------
// measurement / test hooks
// ---------------------------------------------------------------------------------------------------------------
extern "C" float mlcg_time_edge_kernel(mlcg_handle* h, int layer, int iters, void* stream) {
  if (!h || !h->egnn_loaded || !h->batch_set || h->precision == PREC_FP32_SIMT || layer < 0 || layer >= 27 || iters <= 0)
    return -1.f;
  cudaStream_t st = (cudaStream_t)stream;
  const LayerW& L = h->layers[layer];
  EdgeArgs ea = edge_args(h, L, h->xa.as<float>(), h->xb.as<float>());
  const int grid_e = edge_grid(h);
  cudaEvent_t e0, e1;
  if (cudaEventCreate(&e0) != cudaSuccess || cudaEventCreate(&e1) != cudaSuccess) return -1.f;
  if (launch_edge_mode(h->precision, L.equiv, ea, grid_e, st) != cudaSuccess) return -1.f;  // warm-up
  cudaEventRecord(e0, st);
  for (int i = 0; i < iters; ++i) {
    if (launch_edge_mode(h->precision, L.equiv, ea, grid_e, st) != cudaSuccess) return -1.f;
    h->launches++;
  }
  cudaEventRecord(e1, st);
  if (launch_edge_fixup(h, h->precision, L.equiv, ea, st) != cudaSuccess) return -1.f;  // clears the split-target buffers
  if (cudaEventSynchronize(e1) != cudaSuccess || cudaStreamSynchronize(st) != cudaSuccess) return -1.f;
  float ms = 0.f;
  cudaEventElapsedTime(&ms, e0, e1);
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  return ms / iters;
}

// Diagnostics: per-phase cycle counters of the fused edge kernel, averaged over CTAs and tiles.
// out[0..5] = cycles per tile: row-info + P/Q wait, A generation, MMA tail, pass 1, pass 2, A-ring back-pressure.
extern "C" int mlcg_edge_phase_profile(mlcg_handle* h, int layer, double* out, void* stream) {
  if (!h || !out) return MLCG_E_ARG;
  if (!h->egnn_loaded || !h->batch_set || h->precision == PREC_FP32_SIMT || layer < 0 || layer >= 27)
    FAIL(MLCG_E_STATE, "edge_phase_profile: needs a tensor-core precision, weights and a batch");
  cudaStream_t st = (cudaStream_t)stream;
  const LayerW& L = h->layers[layer];
  const int grid_e = edge_grid(h);
  DevBuf buf;
  CK(buf.ensure((size_t)grid_e * 16 * sizeof(long long)));
  CK(cudaMemsetAsync(buf.p, 0, (size_t)grid_e * 16 * sizeof(long long), st));
  EdgeArgs ea = edge_args(h, L, h->xa.as<float>(), h->xb.as<float>());
  ea.prof = buf.as<long long>();
  CK(launch_edge_mode(h->precision, L.equiv, ea, grid_e, st, true));
  h->launches++;
  CK(launch_edge_fixup(h, h->precision, L.equiv, ea, st));
  std::vector<long long> host((size_t)grid_e * 16);
  CK(cudaMemcpyAsync(host.data(), buf.p, host.size() * sizeof(long long), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  buf.release();
  double acc[16] = {0};
  for (int b = 0; b < grid_e; ++b)
    for (int k = 0; k < 16; ++k) acc[k] += (double)host[(size_t)b * 16 + k];
  const double tiles = acc[6] > 0 ? acc[6] : 1.0;
  for (int k = 0; k < 16; ++k) out[k] = (k == 6) ? acc[k] : acc[k] / tiles;
  return MLCG_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// Gaussian shape similarity (reference cheminformatics/shape_similarity.py)
// ---------------------------------------------------------------------------------------------------------------
static double shape_alpha(double amplitude, double atom_radius) {  // get_alpha, shape_similarity.py:322-329
  const double pi = 3.14159265358979323846;
  const double lam = 4.0 * pi / 3.0 / amplitude;
  return pi / pow(lam, 2.0 / 3.0) / (atom_radius * atom_radius);
}

extern "C" int mlcg_shape_moments(mlcg_handle* h, const float* coords, const int32_t* n_nodes, int B, int N, float amplitude,
                                  float atom_radius, int n_terms, float* out, void* stream) {
  if (!h) return MLCG_E_ARG;
  if (!coords || !n_nodes || !out || B <= 0 || N <= 0 || N > SHAPE_MAX_ATOMS || n_terms < 1 || n_terms > SHAPE_MAX_TERMS ||
      !(amplitude > 0.f) || !(atom_radius > 0.f))
    FAIL(MLCG_E_ARG, "shape_moments: need B > 0, 1 <= N <= 64, 1 <= n_terms <= 6");
  CK(cudaSetDevice(h->device));
  const double pi = 3.14159265358979323846, alpha = shape_alpha(amplitude, atom_radius);
  ShapeConsts k{};
  k.amplitude = amplitude;
  k.alpha = (float)alpha;
  k.threshold = 2.0f * amplitude;  // neighbour_threshold default, shape_similarity.py:23
  k.n_terms = n_terms;
  for (int o = 1; o <= SHAPE_MAX_TERMS; ++o) {
    k.amp_k[o] = (float)pow((double)amplitude, (double)o);
    k.vol_k[o] = (float)pow(pi / (o * alpha), 1.5);
    k.inv2ka[o] = (float)(1.0 / (2.0 * o * alpha));
  }
  k_shape_moments<<<B, 128, 0, (cudaStream_t)stream>>>(coords, n_nodes, N, k, out);
  KCHECK();
  h->launches++;
  return MLCG_OK;
}

extern "C" int mlcg_shape_tanimoto(mlcg_handle* h, const float* ref_pts, int n_ref, const float* coords, const int32_t* n_nodes,
                                   int B, int N, const float* frames, const float* orient, int n_orient, const float* axes,
                                   int G, float amplitude, float atom_radius, float* workspace, float* scores, float* aligned,
                                   void* stream) {
  if (!h) return MLCG_E_ARG;
  if (!ref_pts || !coords || !n_nodes || !frames || !orient || !axes || !workspace || !scores || B <= 0 || N <= 0 ||
      N > SHAPE_MAX_ATOMS || n_ref <= 0 || n_ref > SHAPE_MAX_ATOMS || n_orient <= 0 || n_orient > 65535 || G <= 1 ||
      G > SHAPE_MAX_GRID)
    FAIL(MLCG_E_ARG, "shape_tanimoto: need 1 <= N, n_ref <= 64, 2 <= G <= 48, n_orient >= 1");
  CK(cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)stream;
  const float alpha = (float)shape_alpha(amplitude, atom_radius);
  k_shape_grid<true><<<dim3(1, 1), 256, 0, st>>>(ref_pts, nullptr, n_ref, n_ref, nullptr, nullptr, 1, axes, G, amplitude, alpha,
                                                 workspace, nullptr, nullptr);
  KCHECK();
  k_shape_grid<false><<<dim3(B, n_orient), 256, 0, st>>>(coords, n_nodes, 0, N, frames, orient, n_orient, axes, G, amplitude,
                                                         alpha, workspace, scores, aligned);
  KCHECK();
  h->launches += 2;
  return MLCG_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// inertial fragment matching between the two reverse loops (reference utils/mol_utils.py:373-550)
// ---------------------------------------------------------------------------------------------------------------
extern "C" int mlcg_ifm_context(mlcg_handle* h, const float* moi_gen_origin_host, const float* ff_weighted_com_host, int n_ff,
                                const float* norm_mean_host, const float* norm_mad_host, const int32_t* n_nodes, int B,
                                float* ctx_out, float* shift_out, float* rot_out, int32_t* n_gen_out, void* stream) {
  if (!h) return MLCG_E_ARG;
  if (!moi_gen_origin_host || !ff_weighted_com_host || !norm_mean_host || !norm_mad_host || !n_nodes || !ctx_out || !shift_out ||
      !rot_out || !n_gen_out || B <= 0 || n_ff <= 0)
    FAIL(MLCG_E_ARG, "ifm_context: bad argument");
  FragJob q{};
  memcpy(q.moi0, moi_gen_origin_host, sizeof(q.moi0));
  memcpy(q.ffsum, ff_weighted_com_host, sizeof(q.ffsum));
  q.n_ff = n_ff;
  IfmNorms nrm{};
  memcpy(nrm.mean, norm_mean_host, sizeof(nrm.mean));
  memcpy(nrm.mad, norm_mad_host, sizeof(nrm.mad));
  cudaStream_t st = (cudaStream_t)stream;
  CK(h->hook_job.ensure(sizeof(FragJob)));
  CK(cudaMemcpyAsync(h->hook_job.p, &q, sizeof(q), cudaMemcpyHostToDevice, st));
  k_ifm_context<<<(B + 127) / 128, 128, 0, st>>>(n_nodes, nullptr, h->hook_job.as<FragJob>(), B, nrm, ctx_out, shift_out,
                                                 rot_out, n_gen_out);
  KCHECK();
  return MLCG_OK;
}

extern "C" int mlcg_ifm_merge_inputs(mlcg_handle* h, const float* x_gen, const int32_t* cls_gen, const float* shift,
                                     const float* rot, const float* ff_x, const float* ff_h, int n_ff, int B, int Ng, int N,
                                     float* z_known, float* fixed_mask, void* stream) {
  if (!h) return MLCG_E_ARG;
  if (!x_gen || !cls_gen || !shift || !rot || !ff_x || !ff_h || !z_known || !fixed_mask || B <= 0 || n_ff <= 0 || Ng <= 0 ||
      N < n_ff || N > 64)
    FAIL(MLCG_E_ARG, "ifm_merge_inputs: bad argument");
  FragJob q{};
  q.n_ff = n_ff;
  cudaStream_t st = (cudaStream_t)stream;
  CK(h->hook_job.ensure(sizeof(FragJob)));
  CK(cudaMemcpyAsync(h->hook_job.p, &q, sizeof(q), cudaMemcpyHostToDevice, st));
  k_ifm_merge_inputs<<<B, 64, 0, st>>>(x_gen, cls_gen, shift, rot, ff_x, ff_h, nullptr, h->hook_job.as<FragJob>(), Ng, N, z_known,
                                       fixed_mask);
  KCHECK();
  return MLCG_OK;
}

extern "C" int mlcg_gemm_phase_profile(mlcg_handle* h, int which, double* out, void* stream) {
  if (!h || !out) return MLCG_E_ARG;
  if (!h->egnn_loaded || !h->batch_set || h->precision == PREC_FP32_SIMT || which < 0 || which > 2)
    FAIL(MLCG_E_STATE, "gemm_phase_profile: needs a tensor-core precision, weights, a batch and which in 0..2");
  cudaStream_t st = (cudaStream_t)stream;
  const int mode = h->precision, kc = h->kc448();
  const LayerW& L = h->layers[0];
  const int grid = std::min(h->pl->n_mtiles * (which == 0 ? 2 : 1), h->num_sms);
  DevBuf buf;
  CK(buf.ensure((size_t)grid * 8 * sizeof(long long)));
  CK(cudaMemsetAsync(buf.p, 0, (size_t)grid * 8 * sizeof(long long), st));
  GemmArgs a{};
  a.prof = buf.as<long long>();
  a.m_rows = h->pl->M;
  a.out_scale = (which == 0) ? act_scale(mode) : op_scale(mode);
  cudaEvent_t e0, e1;
  CK(cudaEventCreate(&e0));
  CK(cudaEventCreate(&e1));
  CK(cudaEventRecord(e0, st));
  if (which == 0) {
    a.a0 = h->h_op.as<uint8_t>(); a.a0_chunks = kc; a.a0_per_tile = kc; a.n_kc = kc;
    a.w = L.w1ab_op.as<uint8_t>(); a.bias = L.bias_pq.as<float>();
    a.out_f32 = h->pq.as<float>(); a.ldo = 2 * HP; a.n_valid = 2 * HP;
    if (mode == PREC_FP16) CK((launch_gemm<PREC_FP16, HP, EPI_BF16>(a, h->pl->n_mtiles, 2, st)));
    else if (mode == PREC_BF16) CK((launch_gemm<PREC_BF16, HP, EPI_BF16>(a, h->pl->n_mtiles, 2, st)));
    else CK((launch_gemm<PREC_TF32, HP, EPI_F32>(a, h->pl->n_mtiles, 2, st)));
  } else if (which == 1) {
    a.a0 = h->h_op.as<uint8_t>(); a.a0_chunks = kc; a.a0_per_tile = kc;
    a.a1 = h->agg_op.as<uint8_t>(); a.a1_per_tile = kc; a.n_kc = 2 * kc;
    a.w = L.w3_op.as<uint8_t>(); a.bias = L.b3p.as<float>();
    a.out_op = h->t_op.as<uint8_t>(); a.out_op_chunks = kc;
    CK((launch_gemm_mode<HP, EPI_SILU_OP>(mode, a, h->pl->n_mtiles, 1, st)));
  } else {
    a.a0 = h->t_op.as<uint8_t>(); a.a0_chunks = kc; a.a0_per_tile = kc; a.n_kc = kc;
    a.w = L.w4_op.as<uint8_t>(); a.bias = L.b4p.as<float>();
    a.out_op = h->h_op.as<uint8_t>(); a.out_op_chunks = kc; a.resid = h->h_res.as<float>(); a.ldr = 0;
    CK((launch_gemm_mode<HP, EPI_RESID_OP>(mode, a, h->pl->n_mtiles, 1, st)));
  }
  CK(cudaEventRecord(e1, st));
  h->launches++;
  std::vector<long long> host((size_t)grid * 8);
  CK(cudaMemcpyAsync(host.data(), buf.p, host.size() * sizeof(long long), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  float ms = 0.f;
  cudaEventElapsedTime(&ms, e0, e1);
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  buf.release();
  for (int k = 0; k < 8; ++k) out[k] = 0.0;
  for (int b = 0; b < grid; ++b)
    for (int k = 0; k < 7; ++k) out[k] += (double)host[(size_t)b * 8 + k] / grid;
  out[7] = ms;
  return MLCG_OK;
}

extern "C" int mlcg_test_gemm(mlcg_handle* h, int mode, int bn, const float* a, const float* w, const float* bias, float* c,
                              int M, int N, int K, void* stream) {
  if (!h) return MLCG_E_ARG;
  if ((mode != PREC_TF32 && mode != PREC_BF16 && mode != PREC_FP16) || (bn != 448 && bn != 256) || !a || !w || !bias || !c || M <= 0 || N <= 0 || K <= 0)
    FAIL(MLCG_E_ARG, "test_gemm: bad argument");
  if (N % 4 != 0) FAIL(MLCG_E_ARG, "test_gemm: N must be a multiple of 4");
  cudaStream_t st = (cudaStream_t)stream;
  const int kc = (K + epc(mode) - 1) / epc(mode);
  const int mt = (M + TILE_M - 1) / TILE_M, nt = (N + bn - 1) / bn;
  CK(h->tg_a.ensure((size_t)mt * kc * A_CHUNK_BYTES));
  CK(h->tg_w.ensure((size_t)nt * kc * bn * CHUNK_BYTES));
  CK(h->tg_b.ensure((size_t)nt * bn * 4));
  CK(cudaMemsetAsync(h->tg_b.p, 0, (size_t)nt * bn * 4, st));
  CK(cudaMemcpyAsync(h->tg_b.p, bias, (size_t)N * 4, cudaMemcpyDeviceToDevice, st));
  const long long pieces = (long long)M * kc * 8;
  if (mode == PREC_FP16) k_rowmajor_to_op<PREC_FP16><<<(unsigned)((pieces + 255) / 256), 256, 0, st>>>(a, K, M, K, h->tg_a.as<uint8_t>(), kc);
  else if (mode == PREC_BF16) k_rowmajor_to_op<PREC_BF16><<<(unsigned)((pieces + 255) / 256), 256, 0, st>>>(a, K, M, K, h->tg_a.as<uint8_t>(), kc);
  else k_rowmajor_to_op<PREC_TF32><<<(unsigned)((pieces + 255) / 256), 256, 0, st>>>(a, K, M, K, h->tg_a.as<uint8_t>(), kc);
  KCHECK();
  PackArgs pa{};
  pa.src = w; pa.ld = K; pa.n_real = N; pa.bn = bn; pa.n_kc = kc; pa.seg_len = kc * epc(mode); pa.kreal0 = K;
  pa.bias = nullptr; pa.bias_k = -1; pa.dst = h->tg_w.as<uint8_t>();
  CK(launch_pack(mode, pa, nt, st));
  h->launches++;
  GemmArgs g{};
  g.a0 = h->tg_a.as<uint8_t>(); g.a0_chunks = kc; g.a0_per_tile = kc; g.n_kc = kc;
  g.w = h->tg_w.as<uint8_t>(); g.bias = h->tg_b.as<float>(); g.m_rows = M;
  g.out_f32 = c; g.ldo = N; g.n_valid = N; g.rowscale = nullptr; g.relu = 0;
  if (bn == 448) CK((launch_gemm_mode<448, EPI_F32>(mode, g, mt, nt, st)));
  else CK((launch_gemm_mode<256, EPI_F32>(mode, g, mt, nt, st)));
  h->launches++;
  return MLCG_OK;
}
