// Library plumbing: error string, model geometry, workspace sizing.
#include "common.cuh"
#include "mlp_fp32.cuh"
#include "mlp_tc.cuh"
#include "../../include/knerf_debug.h"

#include <atomic>

namespace knerf {

static std::atomic<uint64_t> g_launches{0};
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

char* last_error_buffer() {
  static thread_local char buf[512] = {0};
  return buf;
}

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(last_error_buffer(), 512, fmt, ap);
  va_end(ap);
  return code;
}

// keras_nerf/model/nerf/mlp.py:11-27,33-46: widths of every Dense layer, in Keras variable order
int build_model(const knerf_config* cfg, Model* m) {
  KN_CHECK_ARG(cfg != nullptr, "null config");
  KN_CHECK_ARG(cfg->n_layers >= 1 && cfg->n_layers <= kMaxLayers - 4, "n_layers=%d out of range", cfg->n_layers);
  KN_CHECK_ARG(cfg->dense_units >= 2 && cfg->dense_units % 2 == 0, "dense_units=%d must be even", cfg->dense_units);
  KN_CHECK_ARG(cfg->skip_layer >= 1, "skip_layer=%d", cfg->skip_layer);
  m->cfg = *cfg;
  m->dx = cfg->dx > 0 ? cfg->dx : 3 + 6 * cfg->pos_emb_xyz;
  m->dd = cfg->dd > 0 ? cfg->dd : 3 + 6 * cfg->pos_emb_dir;
  m->U = cfg->dense_units;
  m->n_layers = cfg->n_layers;
  m->n_dense = cfg->n_layers + 4;
  int64_t off = 0;
  int kh = 0, kx = m->dx;
  auto add = [&](int idx, int k_h, int k_x, int fan_out) {
    LayerDesc& L = m->L[idx];
    L.k_h = k_h; L.k_x = k_x; L.fan_in = k_h + k_x; L.fan_out = fan_out;
    L.w_off = off; off += (int64_t)L.fan_in * fan_out;
    L.b_off = off; off += fan_out;
  };
  for (int i = 0; i < m->n_layers; ++i) {
    add(i, kh, kx, m->U);
    kh = m->U;
    kx = (i % cfg->skip_layer == 0 && i > 0) ? m->dx : 0;   // mlp.py:36-38, concat order [h, x]
  }
  m->head_skip = kx > 0;
  const int n = m->n_layers;
  add(n, kh, kx, 1);                 // sigma
  add(n + 1, kh, kx, m->U);          // features
  add(n + 2, m->U, m->dd, m->U / 2); // rgb_features: [features, dir]
  add(n + 3, m->U / 2, 0, 3);        // rgb
  m->n_params = off;
  return KNERF_OK;
}

// The fused bf16 chain kernels run ONE fixed program: eight 256-wide ReLU layers, the encoding concatenated in front of
// chain layer 5, then the heads.  A model fits when it can be embedded in that program exactly:
//  * encodings that are prefixes of PE_10 / PE_4 (unused columns get zero weights);
//  * dense_units <= 256: the operands are zero-padded to 256 columns (relu(0) = 0 stays 0, its gradients are not flushed);
//  * up to eight layers with at most one layer that takes the skip concat (and not the heads): its layers
//    keep their order, the concat layer sits at chain layer 5, and the remaining chain layers are IDENTITY layers
//    (kernel I, bias 0).  An identity layer behind a ReLU is exact, in fp32 and in bf16 alike: its input h >= 0 is
//    already rounded, relu(I h) = h has the same bits, and backwards (dH [h > 0]) [h > 0] = dH [h > 0].
// chain_map[c] = the model layer at chain layer c, -1 = identity.
bool tc_chain_map(const Model& m, int chain_map[8]) {
  if (!(m.U >= 2 && m.U <= 256 && m.U % 2 == 0 && m.n_layers >= 1 && m.n_layers <= 8 && !m.head_skip && m.cfg.pos_emb_xyz >= 0 &&
        m.cfg.pos_emb_xyz <= 10 && m.cfg.pos_emb_dir >= 0 && m.cfg.pos_emb_dir <= 4 &&
        m.dx == 3 + 6 * m.cfg.pos_emb_xyz && m.dd == 3 + 6 * m.cfg.pos_emb_dir))
    return false;
  int s = -1;                                   // the layer that takes [h, x]
  for (int i = 1; i < m.n_layers; ++i)
    if (m.L[i].k_x > 0) {
      if (s >= 0) return false;
      s = i;
    }
  for (int c = 0; c < 8; ++c) chain_map[c] = -1;
  if (s < 0) {
    for (int c = 0; c < m.n_layers; ++c) chain_map[c] = c;
    return true;
  }
  if (s > 5 || m.n_layers - 1 - s > 2) return false;
  for (int c = 0; c < s; ++c) chain_map[c] = c;
  for (int i = s; i < m.n_layers; ++i) chain_map[5 + (i - s)] = i;
  return true;
}
bool is_flagship(const Model& m) {
  int map[8];
  return tc_chain_map(m, map);
}

}  // namespace knerf

using namespace knerf;

extern "C" int knerf_abi_version(void) { return KNERF_ABI_VERSION; }
extern "C" uint64_t knerf_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }
extern "C" const char* knerf_last_error(void) { return last_error_buffer(); }

extern "C" int knerf_device_supports_bf16(void) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 0;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, dev) != cudaSuccess) return 0;
  return (prop.major == 10 && tc_path_compiled()) ? 1 : 0;
}

extern "C" int knerf_debug_tc_timing(unsigned long long* host_out, int n) { return tc_debug_timing(host_out, n); }
extern "C" int knerf_debug_wgrad_timing(unsigned long long* host_out, int n) { return tc_debug_wgrad_timing(host_out, n); }

extern "C" int64_t knerf_param_count(const knerf_config* cfg) {
  Model m;
  if (build_model(cfg, &m) != KNERF_OK) return -1;
  return m.n_params;
}

extern "C" int knerf_layer_table(const knerf_config* cfg, int max_layers, int64_t* kernel_off, int64_t* bias_off,
                                 int32_t* fan_in, int32_t* fan_out) {
  Model m;
  KN_TRY(build_model(cfg, &m));
  KN_CHECK_ARG(max_layers >= m.n_dense && kernel_off && bias_off && fan_in && fan_out,
               "knerf_layer_table: need room for %d layers", m.n_dense);
  for (int i = 0; i < m.n_dense; ++i) {
    kernel_off[i] = m.L[i].w_off; bias_off[i] = m.L[i].b_off;
    fan_in[i] = m.L[i].fan_in; fan_out[i] = m.L[i].fan_out;
  }
  return m.n_dense;
}

extern "C" int64_t knerf_workspace_bytes(const knerf_config* cfg, int64_t rows, int precision, int training) {
  Model m;
  if (build_model(cfg, &m) != KNERF_OK || rows < 0) return -1;
  int64_t mlp = 0;
  const bool rec8 = (precision & KNERF_REC_FP8) != 0;
  precision &= KNERF_PRECISION_MASK;
  if (precision == KNERF_FP32 || precision == KNERF_FP32_TC)
    mlp = (int64_t)make_fp32_plan(m, rows, training != 0, precision == KNERF_FP32_TC).total;
  else if (precision == KNERF_BF16) mlp = tc_workspace_bytes(m, rows, training != 0, rec8);
  else return -1;
  if (mlp < 0) return -1;
  // chunk-level scratch of knerf_render_chunk / knerf_train_chunk: rgbsigma + d_pre (16 B/row each),
  // t_sorted + weights (4 B/row each), per-ray image / sqerr (<= 16 B/row), alignment slack
  return mlp + rows * 64 + 8192;
}
