// extern "C" surface of librr_sm100 (include/rr_sm100.h).  No C++ exception crosses it.
#include <stdarg.h>
#include <stdlib.h>

#include "rr_common.cuh"

namespace rr {
thread_local char g_err[512] = "";
std::atomic<int64_t> g_launches{0};
std::atomic<int> g_gemm_mode{0};
std::atomic<int> g_bwd_bf16{1};
std::atomic<int> g_fwd_bf16{0};
std::atomic<int> g_deterministic{0};
ProfState g_prof;
std::mutex g_prof_mutex;

static Switches g_switches;
static std::atomic<bool> g_switches_loaded{false};
static std::mutex g_switches_mutex;
static int env_int(const char* name, int dflt) {
  const char* e = getenv(name);
  return (e && *e) ? atoi(e) : dflt;
}
void reload_switches() {
  std::lock_guard<std::mutex> lock(g_switches_mutex);
  Switches w;
  w.mp_v1 = env_int("RR_MP_V1", 0);
  g_switches = w;
  g_switches_loaded.store(true);
}
const Switches& switches() {
  if (!g_switches_loaded.load()) reload_switches();
  return g_switches;
}
int det_scratch(DetScratch* d, void* given, long long given_bytes, long long need, cudaStream_t s) {
  if (given) {
    if (given_bytes < need) return fail(RR_ERR_WORKSPACE, "deterministic mode: workspace has %lld bytes of scratch, needs %lld", given_bytes, need);
    d->p = given;
    return RR_OK;
  }
  if (need <= 0) return RR_OK;
  RR_CUDA(cudaMallocAsync(&d->p, static_cast<size_t>(need), s));
  d->s = s;
  d->owned = true;
  return RR_OK;
}

void prof_push(int cls, cudaEvent_t a, cudaEvent_t b) {
  std::lock_guard<std::mutex> lock(g_prof_mutex);
  ProfState& p = g_prof;
  if (p.n == p.cap) {
    const int cap = p.cap ? p.cap * 2 : 4096;
    ProfState::Rec* r = static_cast<ProfState::Rec*>(realloc(p.recs, cap * sizeof(ProfState::Rec)));
    if (!r) return;
    p.recs = r;
    p.cap = cap;
  }
  p.recs[p.n++] = ProfState::Rec{cls, a, b};
}

}  // namespace rr

#define S(stream) static_cast<cudaStream_t>(stream)

extern "C" {

int rr_version(void) { return RR_ABI_VERSION; }
const char* rr_last_error(void) { return rr::g_err; }

int rr_device_check(int device) {
  cudaDeviceProp prop;
  RR_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) return rr::fail(RR_ERR_ARCH, "device %d is sm_%d%d; librr_sm100 contains sm_100a code only", device, prop.major, prop.minor);
  return RR_OK;
}

int rr_padded(int width) { return rr::padded(width); }

int rr_graph_assemble(const rr_mol_store* store, int n_mols, const int32_t* mol_ids, const int32_t* a_start, const int32_t* b_start,
                      const int32_t* mol_W, const int32_t* mol_pad_bond, const int32_t* mol_pad_atom, int n_segments, const int32_t* seg_pad_atom,
                      const int32_t* seg_pad_bond, const int32_t* seg_W, const rr_graph* out, void* stream) {
  return rr::graph_assemble(store, n_mols, mol_ids, a_start, b_start, mol_W, mol_pad_bond, mol_pad_atom, n_segments, seg_pad_atom, seg_pad_bond,
                            seg_W, out, S(stream));
}
int rr_bond_message_fwd(const rr_graph* g, const float* m, float* pre, int hp, int relu_src, void* stream) {
  return rr::bond_message_fwd(g, m, pre, hp, relu_src, S(stream));
}
int rr_bond_message_bwd(const rr_graph* g, const float* dpre, float* dm, int hp, void* stream) {
  return rr::bond_message_bwd(g, dpre, dm, hp, S(stream));
}
int rr_neighbor_sum_fwd(const rr_graph* g, int which, const float* src, float* out, int ld, int relu_src, void* stream) {
  RR_REQUIRE(which == 0 || which == 1, "which must be 0 (a2b) or 1 (a2a)");
  return rr::neighbor_sum_fwd(g, which, src, out, ld, relu_src, S(stream));
}
int rr_neighbor_sum_bwd(const rr_graph* g, int which, const float* dout, float* dsrc, int ld, void* stream) {
  RR_REQUIRE(which == 0 || which == 1, "which must be 0 (a2b) or 1 (a2a)");
  return rr::neighbor_sum_bwd(g, which, dout, dsrc, ld, S(stream));
}
int rr_bond_message_bwd_act(const rr_graph* g, const float* dpre, float* dm, int hp, const float* y, float scale, int y_is_preact, float* acc, int acc_mode,
                            int skip_out, void* stream) {
  return rr::bond_message_bwd_act(g, dpre, dm, hp, y, scale, y_is_preact, acc, acc_mode, skip_out, S(stream));
}
int rr_neighbor_sum_bwd_act(const rr_graph* g, int which, const float* dout, float* dsrc, int ld, const float* y, float scale, int y_is_preact, float* acc,
                            int acc_mode, int skip_out, void* stream) {
  RR_REQUIRE(which == 0 || which == 1, "which must be 0 (a2b) or 1 (a2a)");
  return rr::neighbor_sum_bwd_act(g, which, dout, dsrc, ld, y, scale, y_is_preact, acc, acc_mode, skip_out, S(stream));
}
int rr_readout_fwd(const rr_graph* g, const float* hid, int hp, int hidden, const float* add_features, int n_add, float* vec, int vp,
                   float dropout, uint64_t seed, uint64_t stream_id, void* stream) {
  return rr::readout_fwd(g, hid, hp, hidden, add_features, n_add, vec, vp, dropout, seed, stream_id, S(stream));
}
int rr_readout_bwd(const rr_graph* g, const float* dvec, int vp, const float* vec, const float* hid, float* dz, int hp, float dropout, void* stream) {
  return rr::readout_bwd(g, dvec, vp, vec, hid, dz, hp, dropout, dropout, S(stream));
}
int rr_linear_fwd(int M, int n, const float* X1, int ldx1, const float* W1, int k1, const float* X2, int ldx2, const float* W2, int k2,
                  const float* bias, const float* residual, int ldr, float* Y, int ldy, int flags, float dropout, uint64_t seed,
                  uint64_t stream_id, void* stream) {
  return rr::linear_fwd(M, n, X1, ldx1, W1, k1, X2, ldx2, W2, k2, bias, residual, ldr, Y, ldy, flags, dropout, seed, stream_id, S(stream));
}
int rr_linear_dgrad(int M, int n, int k, const float* dZ, int lddz, const float* W, int ldw, float* dX, int lddx, int accumulate, void* stream) {
  return rr::simt_dgrad(M, n, k, dZ, lddz, W, ldw, dX, lddx, accumulate, S(stream));
}
int64_t rr_linear_dgrad_tc_scratch_bytes(int n, int k) { return rr::tc_dgrad_scratch_bytes(n, k); }
int rr_linear_dgrad_tc(int M, int n, int k, const float* dZ, int lddz, const float* W, int ldw, float* dX, int lddx, int accumulate, void* scratch,
                       int64_t scratch_bytes, void* stream) {
  return rr::linear_dgrad_tc(M, n, k, dZ, lddz, W, ldw, dX, lddx, accumulate, scratch, scratch_bytes, S(stream));
}
int rr_linear_wgrad(int M, int n, int k, const float* dZ, int lddz, const float* X, int ldx, float* dW, int lddw, float* dbias, void* stream) {
  return rr::linear_wgrad(M, n, k, dZ, lddz, X, ldx, dW, lddw, dbias, S(stream));
}
int rr_relu_bwd(int64_t rows, int ld, const float* dy, const float* y, float scale, int y_is_preact, float* dz, float* acc, int acc_mode, void* stream) {
  return rr::relu_bwd(rows, ld, dy, y, scale, y_is_preact, dz, acc, acc_mode, S(stream));
}
int rr_sub(int64_t n, const float* a, const float* b, float* out, void* stream) { return rr::sub(n, a, b, out, S(stream)); }

int rr_loss_fwdbwd(int kind, int N, int G, const float* scores, const float* targets, const int32_t* seg_off, float norm, float sigma,
                   float* loss, float* dscore, void* stream) {
  return rr::loss_fwdbwd(kind, N, G, scores, targets, seg_off, norm, sigma, loss, dscore, S(stream));
}
int rr_loss_fwdbwd_ex(int kind, int N, int G, const float* scores, const float* targets, const int32_t* seg_off, int max_group, float norm,
                      float sigma, float* loss, float* dscore, void* stream) {
  return rr::loss_fwdbwd(kind, N, G, scores, targets, seg_off, norm, sigma, loss, dscore, S(stream), max_group);
}
int rr_loss_max_group(void) { return rr::loss_max_group(); }
int rr_rank_metrics(int N, int G, const float* scores, int score_ld, const double* targets, const int32_t* seg_off, int max_group, double ratio,
                    double* out, void* stream) {
  return rr::rank_metrics(N, G, scores, score_ld, targets, seg_off, max_group, ratio, out, S(stream));
}
int rr_rank_predict(int N, int G, int T, const float* scores, int64_t sample_stride, int score_ld, const int32_t* seg_off, int max_group,
                    float* out, void* stream) {
  return rr::rank_predict(N, G, T, scores, sample_stride, score_ld, seg_off, max_group, out, S(stream));
}

int64_t rr_model_workspace_bytes_ex(const rr_model_cfg_ex* cfg, const rr_graph* r, const rr_graph* p) {
  if (!cfg || !r || !p) {
    rr::fail(RR_ERR_INVALID, "rr_model_workspace_bytes: NULL argument");
    return -1;
  }
  return rr::model_workspace_bytes(cfg, r, p);
}
int64_t rr_model_buffer_offset_ex(const rr_model_cfg_ex* cfg, const rr_graph* r, const rr_graph* p, const char* name) {
  if (!cfg || !r || !p || !name) {
    rr::fail(RR_ERR_INVALID, "rr_model_buffer_offset: NULL argument");
    return -1;
  }
  return rr::model_buffer_offset(cfg, r, p, name);
}
int rr_model_forward_ex(const rr_model_cfg_ex* cfg, const rr_params* w, const rr_graph* r, const rr_graph* p, const float* add_features,
                        float* scores, void* ws, int64_t ws_bytes, void* stream) {
  return rr::model_forward(cfg, w, r, p, add_features, scores, ws, ws_bytes, S(stream));
}
int rr_model_backward_ex(const rr_model_cfg_ex* cfg, const rr_params* w, const rr_graph* r, const rr_graph* p, const float* dscores,
                         rr_params* grads, void* ws, int64_t ws_bytes, void* stream) {
  return rr::model_backward(cfg, w, r, p, dscores, grads, ws, ws_bytes, S(stream));
}
// ABI 3: every sub-module has cfg->hidden and cfg->dropout (a NULL cfg stays NULL for the _ex entry point to report)
static const rr_model_cfg_ex* tied(const rr_model_cfg* cfg, rr_model_cfg_ex* ex) {
  if (!cfg) return nullptr;
  *ex = rr_model_cfg_ex{*cfg, cfg->hidden, cfg->hidden, cfg->dropout, cfg->dropout};
  return ex;
}
int64_t rr_model_workspace_bytes(const rr_model_cfg* cfg, const rr_graph* r, const rr_graph* p) {
  rr_model_cfg_ex ex;
  return rr_model_workspace_bytes_ex(tied(cfg, &ex), r, p);
}
int64_t rr_model_buffer_offset(const rr_model_cfg* cfg, const rr_graph* r, const rr_graph* p, const char* name) {
  rr_model_cfg_ex ex;
  return rr_model_buffer_offset_ex(tied(cfg, &ex), r, p, name);
}
int rr_model_forward(const rr_model_cfg* cfg, const rr_params* w, const rr_graph* r, const rr_graph* p, const float* add_features,
                     float* scores, void* ws, int64_t ws_bytes, void* stream) {
  rr_model_cfg_ex ex;
  return rr_model_forward_ex(tied(cfg, &ex), w, r, p, add_features, scores, ws, ws_bytes, stream);
}
int rr_model_backward(const rr_model_cfg* cfg, const rr_params* w, const rr_graph* r, const rr_graph* p, const float* dscores,
                      rr_params* grads, void* ws, int64_t ws_bytes, void* stream) {
  rr_model_cfg_ex ex;
  return rr_model_backward_ex(tied(cfg, &ex), w, r, p, dscores, grads, ws, ws_bytes, stream);
}
int rr_set_gemm_mode(int mode) {
  RR_REQUIRE(mode >= 0 && mode <= 3, "gemm mode must be 0 (fp32 SIMT), 1 (tcgen05 3xTF32) or the debug masks 2 (forward only) / 3 (dgrad only)");
  rr::g_gemm_mode.store(mode);
  return RR_OK;
}
int rr_get_gemm_mode(void) { return rr::g_gemm_mode.load(); }
int rr_set_backward_bf16(int on) {
  rr::g_bwd_bf16.store(on ? 1 : 0);
  return RR_OK;
}
int rr_get_backward_bf16(void) { return rr::g_bwd_bf16.load(); }
int rr_set_forward_bf16(int on) {
  rr::g_fwd_bf16.store(on ? 1 : 0);
  return RR_OK;
}
int rr_get_forward_bf16(void) { return rr::g_fwd_bf16.load(); }
int rr_set_deterministic(int on) {
  RR_REQUIRE(on == 0 || on == 1, "rr_set_deterministic: on must be 0 or 1 (got %d)", on);
  rr::g_deterministic.store(on);
  return RR_OK;
}
int rr_get_deterministic(void) { return rr::g_deterministic.load(); }
int rr_profile_begin(void) {
  std::lock_guard<std::mutex> lock(rr::g_prof_mutex);
  rr::g_prof.enabled = true;
  rr::g_prof.n = 0;
  return RR_OK;
}
int rr_profile_end(double* ms_by_class, int64_t* launches_by_class, int n_classes) {
  std::lock_guard<std::mutex> lock(rr::g_prof_mutex);
  rr::ProfState& p = rr::g_prof;
  p.enabled = false;
  RR_REQUIRE(ms_by_class && launches_by_class && n_classes >= rr::KC_COUNT, "rr_profile_end: need %d classes", rr::KC_COUNT);
  for (int i = 0; i < n_classes; ++i) {
    ms_by_class[i] = 0.0;
    launches_by_class[i] = 0;
  }
  int status = RR_OK;
  for (int i = 0; i < p.n; ++i) {
    float ms = 0.f;
    if (cudaEventSynchronize(p.recs[i].b) != cudaSuccess || cudaEventElapsedTime(&ms, p.recs[i].a, p.recs[i].b) != cudaSuccess)
      status = rr::fail(RR_ERR_CUDA, "rr_profile_end: event %d not complete", i);
    ms_by_class[p.recs[i].cls] += ms;
    launches_by_class[p.recs[i].cls] += 1;
    cudaEventDestroy(p.recs[i].a);
    cudaEventDestroy(p.recs[i].b);
  }
  p.n = 0;
  return status;
}
int rr_profile_classes(void) { return rr::KC_COUNT; }
void rr_reload_switches(void) { rr::reload_switches(); }
int64_t rr_launch_count(void) { return rr::g_launches.load(); }
void rr_launch_count_reset(void) { rr::g_launches.store(0); }

}  // extern "C"
