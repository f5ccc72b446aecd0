// C ABI of libdposer_b200: error plumbing, score-network handle, engine dispatch for
// forward / sampler / prior loss, metrics.  See include/dposer_b200.h for the contract.
#include <algorithm>
#include <cstring>
#include <vector>

#include "score.h"
#include "train.h"

namespace dpb {

static thread_local std::string g_last_error;
void set_error(const std::string& msg) { g_last_error = msg; }
int fail(int code, const std::string& msg) {
  g_last_error = msg;
  return code;
}

// sampler.cu launchers
// sampler.cu launchers; `dp` = the handle's padded pose width (64 or 128)
int launch_em_update(float*, const float*, const float*, const float*, const float*, const float*, int, uint64_t,
                     uint32_t, float*, float*, int64_t, int, int dp, cudaStream_t);
int launch_impute(float*, const float*, const float*, const float*, const float*, uint64_t, uint32_t, int64_t, int dp,
                  cudaStream_t);
int launch_scale_out(const float*, const float*, float, float*, int64_t, int dp, cudaStream_t);
int launch_perturb(const float*, const float*, uint64_t, uint32_t, float, float, float*, int64_t, int dp, cudaStream_t);
int launch_prior_loss(const float*, const float*, const float*, float, float, float, float, float, float*, float*,
                      float*, int64_t, int dp, cudaStream_t);

static int pick_engine(const dpb_score* h, int flags, int64_t B, bool uniform_t) {
  int e = flags & DPB_ENGINE_MASK;
  if (e == DPB_ENGINE_AUTO) e = (h->tc_ready && uniform_t && B >= 64) ? DPB_ENGINE_TC : DPB_ENGINE_FP32;
  return e;
}

}  // namespace dpb

using namespace dpb;

extern "C" int dpb_version(void) { return DPB_VERSION; }
extern "C" const char* dpb_last_error(void) { return g_last_error.c_str(); }

extern "C" int dpb_device_info(int device, int* sm_count, int* cc_major, int* cc_minor) {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n <= 0) return fail(DPB_ECUDA, std::string("no CUDA device: ") + cudaGetErrorString(e));
  if (device < 0 || device >= n) return fail(DPB_EINVAL, "dpb_device_info: device index out of range");
  cudaDeviceProp p;
  DPB_CUDA_CHECK(cudaGetDeviceProperties(&p, device));
  if (sm_count) *sm_count = p.multiProcessorCount;
  if (cc_major) *cc_major = p.major;
  if (cc_minor) *cc_minor = p.minor;
  return DPB_OK;
}

// ------------------------------------------------------------------ score handle
static int up_f32(float** dst, const float* src, size_t n) {
  DPB_CUDA_CHECK(cudaMalloc((void**)dst, n * sizeof(float)));
  DPB_CUDA_CHECK(cudaMemcpy(*dst, src, n * sizeof(float), cudaMemcpyHostToDevice));
  return DPB_OK;
}

extern "C" int dpb_score_create_dim(dpb_score_t** out, const dpb_score_weights* w, int pose_dim, int device) {
  if (pose_dim != DPB_POSE_DIM && pose_dim != DPB_POSE_DIM_ROT6D)
    return fail(DPB_EUNSUPPORTED, "dpb_score_create_dim: pose_dim must be 63 (axis-angle) or 126 (rot6d)");
  if (!out || !w) return fail(DPB_EINVAL, "dpb_score_create_dim: null argument");
  const void* req[] = {w->pre_w, w->pre_b, w->pre_t_w, w->pre_t_b, w->pre_gn_w, w->pre_gn_b, w->temb_w, w->temb_b,
                       w->post_w, w->post_b, w->emb_freqs};
  for (const void* p : req) DPB_REQUIRE(p, "dpb_score_create_dim: missing weight pointer");
  for (int i = 0; i < 4; ++i)
    DPB_REQUIRE(w->blk_w[i] && w->blk_b[i] && w->blk_t_w[i] && w->blk_t_b[i] && w->blk_gn_w[i] && w->blk_gn_b[i],
                "dpb_score_create_dim: missing block weight pointer");
  int sm = 0, maj = 0, mnr = 0;
  int rc = dpb_device_info(device, &sm, &maj, &mnr);
  if (rc != DPB_OK) return rc;
  if (maj != 10) return fail(DPB_ECUDA, "dpb_score_create_dim: device is not sm_100 (B200) class");
  DeviceGuard guard(device);
  dpb_score* h = new dpb_score();
  h->device = device;
  h->sm_count = sm;
  h->pose_dim = pose_dim;
  h->pose_dp = pose_dim == D126 ? DP128 : DP;
  const int hd = h->pose_dim, hdp = h->pose_dp;
  // padded fp32 copies
  std::vector<float> prew((size_t)H * hdp, 0.f), postw((size_t)hdp * H, 0.f), postb(hdp, 0.f);
  for (int o = 0; o < H; ++o) std::memcpy(&prew[(size_t)o * hdp], w->pre_w + (size_t)o * hd, hd * sizeof(float));
  std::memcpy(postw.data(), w->post_w, (size_t)hd * H * sizeof(float));
  std::memcpy(postb.data(), w->post_b, hd * sizeof(float));
  const float* lin_b[5] = {w->pre_b, w->blk_b[0], w->blk_b[1], w->blk_b[2], w->blk_b[3]};
  const float* t_w[5] = {w->pre_t_w, w->blk_t_w[0], w->blk_t_w[1], w->blk_t_w[2], w->blk_t_w[3]};
  const float* t_b[5] = {w->pre_t_b, w->blk_t_b[0], w->blk_t_b[1], w->blk_t_b[2], w->blk_t_b[3]};
  const float* gn_w[5] = {w->pre_gn_w, w->blk_gn_w[0], w->blk_gn_w[1], w->blk_gn_w[2], w->blk_gn_w[3]};
  const float* gn_b[5] = {w->pre_gn_b, w->blk_gn_b[0], w->blk_gn_b[1], w->blk_gn_b[2], w->blk_gn_b[3]};
  rc = up_f32(&h->pre_w, prew.data(), prew.size());
  if (rc == DPB_OK) rc = up_f32(&h->post_w, postw.data(), postw.size());
  if (rc == DPB_OK) rc = up_f32(&h->post_b, postb.data(), postb.size());
  if (rc == DPB_OK) rc = up_f32(&h->temb_w, w->temb_w, (size_t)E * E);
  if (rc == DPB_OK) rc = up_f32(&h->temb_b, w->temb_b, E);
  if (rc == DPB_OK) rc = up_f32(&h->emb_freqs, w->emb_freqs, E / 2);
  for (int i = 0; i < 4 && rc == DPB_OK; ++i) rc = up_f32(&h->blk_w[i], w->blk_w[i], (size_t)H * H);
  std::vector<float> gnp((size_t)NL * 2 * H);
  for (int l = 0; l < NL && rc == DPB_OK; ++l) {
    rc = up_f32(&h->lin_b[l], lin_b[l], H);
    if (rc == DPB_OK) rc = up_f32(&h->t_w[l], t_w[l], (size_t)H * E);
    if (rc == DPB_OK) rc = up_f32(&h->t_b[l], t_b[l], H);
    if (rc == DPB_OK) rc = up_f32(&h->gn_w[l], gn_w[l], H);
    if (rc == DPB_OK) rc = up_f32(&h->gn_b[l], gn_b[l], H);
    std::memcpy(&gnp[(size_t)(l * 2) * H], gn_w[l], H * sizeof(float));
    std::memcpy(&gnp[(size_t)(l * 2 + 1) * H], gn_b[l], H * sizeof(float));
  }
  if (rc == DPB_OK) rc = up_f32(&h->gn_packed, gnp.data(), gnp.size());
  if (rc == DPB_OK) rc = tc_prepare(h, w);
  if (rc != DPB_OK) {
    dpb_score_destroy(h);
    return rc;
  }
  *out = h;
  return DPB_OK;
}

extern "C" int dpb_score_pose_dim(dpb_score_t* h) {
  if (!h) return fail(DPB_EINVAL, "dpb_score_pose_dim: null handle");
  return h->pose_dim;
}

extern "C" int dpb_score_destroy(dpb_score_t* h) {
  if (!h) return DPB_OK;
  DeviceGuard guard(h->device);
  tc_release(h);
  score_jvp_tc_release(h);
  std::vector<void*> ptrs = {h->pre_w, h->post_w, h->post_b, h->temb_w, h->temb_b, h->emb_freqs, h->gn_packed};
  for (int i = 0; i < 4; ++i) ptrs.push_back(h->blk_w[i]);
  for (int l = 0; l < NL; ++l) {
    ptrs.push_back(h->lin_b[l]); ptrs.push_back(h->t_w[l]); ptrs.push_back(h->t_b[l]);
    ptrs.push_back(h->gn_w[l]); ptrs.push_back(h->gn_b[l]);
  }
  for (void* p : ptrs) if (p) cudaFree(p);
  delete h;
  return DPB_OK;
}

extern "C" int dpb_score_time_table(dpb_score_t* h, const float* labels, int n, float* table, void* stream) {
  if (!h || !labels || !table || n < 0) return fail(DPB_EINVAL, "dpb_score_time_table: bad argument");
  DeviceGuard guard(h->device);
  return simt_time_table(h, labels, n, table, (cudaStream_t)stream);
}

extern "C" size_t dpb_score_workspace_bytes(dpb_score_t* h, int64_t B, int flags) {
  (void)flags;
  if (!h || B <= 0) return 0;
  // fp32 engine buffers + raw [B,DP] + perturbed x [B,D]; the tcgen05 engine owns its scratch
  return simt_forward_ws_bytes(B, h->pose_dp) + align_up((size_t)B * h->pose_dp * 4, 256) + align_up((size_t)B * h->pose_dim * 4, 256) +
         1024;
}

namespace {
struct ScoreWs {
  float* raw;
  float* xt;
  void* rest;
  size_t rest_bytes;
};
bool carve_score_ws(const dpb_score* h, int64_t B, void* ws, size_t ws_bytes, ScoreWs* o) {
  if (!ws) return false;
  WsCarver c(ws, ws_bytes);
  o->raw = c.take<float>((size_t)B * h->pose_dp);
  o->xt = c.take<float>((size_t)B * h->pose_dim);
  c.off = align_up(c.off, 256);
  if (!c.ok()) return false;
  o->rest = c.base + c.off;
  o->rest_bytes = ws_bytes - c.off;
  return o->rest_bytes >= simt_forward_ws_bytes(B, h->pose_dp);
}
}  // namespace

extern "C" int dpb_score_forward(dpb_score_t* h, const float* x, const float* table, const int32_t* t_index,
                                 const float* row_scale, float scale, float* out, int64_t B, int flags, void* ws,
                                 size_t ws_bytes, void* stream) {
  if (!h) return fail(DPB_EINVAL, "dpb_score_forward: null handle");
  DeviceGuard guard(h->device);
  DPB_REQUIRE(x && table && out, "dpb_score_forward: x, table and out are required");
  if (B <= 0) return DPB_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const int engine = pick_engine(h, flags, B, t_index == nullptr);
  if (engine == DPB_ENGINE_TC) {
    if (!h->tc_ready) return fail(DPB_EUNSUPPORTED, "dpb_score_forward: tcgen05 engine unavailable");
    if (t_index) return fail(DPB_EUNSUPPORTED, "dpb_score_forward: tcgen05 engine needs batch-uniform t");
    TcJob j{};
    j.mode = 0; j.B = B; j.x_in = x; j.table = table; j.n_steps = 1;
    j.row_scale = row_scale; j.scale = scale; j.out = out;
    return tc_launch(h, j, st);
  }
  ScoreWs w;
  if (!carve_score_ws(h, B, ws, ws_bytes, &w)) return fail(DPB_ENOMEM, "dpb_score_forward: workspace too small");
  int rc = simt_forward_raw(h, x, table, t_index, w.raw, B, w.rest, w.rest_bytes, st);
  if (rc != DPB_OK) return rc;
  return launch_scale_out(w.raw, row_scale, scale, out, B, h->pose_dp, st);
}

// Predictor-corrector sampling with the Langevin corrector (sampling.py:456-461 with :282-302), all steps from one host
// call: per step  score -> batch norms -> corrector update -> (one fused predictor step incl. imputation).  The corrector
// needs batch-global norms between its score evaluation and its update, so a step is five launches, issued here without
// returning to the caller (the Python loop of round 1 was bound by its per-step host work at small batches).
extern "C" size_t dpb_sampler_pc_workspace_bytes(dpb_score_t* h, int64_t B) {
  if (!h || B <= 0) return 0;
  return dpb_score_workspace_bytes(h, B, 0) + 2 * align_up((size_t)B * h->pose_dim * 4, 256) + 256 + 1024;
}

extern "C" int dpb_sampler_run_pc(dpb_score_t* h, float* x_io, const dpb_step_tables* tbl, const float* score_scale,
                                  const float* lang_alpha, float snr, const float* obs, const float* mask,
                                  const float* noise, uint64_t seed, uint64_t step_offset, float* traj, float* x_mean,
                                  int64_t B, int flags, void* ws, size_t ws_bytes, void* stream) {
  if (!h || !tbl) return fail(DPB_EINVAL, "dpb_sampler_run_pc: null handle or tables");
  DeviceGuard guard(h->device);
  DPB_REQUIRE(x_io && tbl->coef && tbl->time_table && score_scale && lang_alpha && x_mean,
              "dpb_sampler_run_pc: x_io, tables, score_scale, lang_alpha and x_mean are required");
  if (B <= 0 || tbl->n_steps <= 0) return DPB_OK;
  if (ws == nullptr || ws_bytes < dpb_sampler_pc_workspace_bytes(h, B))
    return fail(DPB_ENOMEM, "dpb_sampler_run_pc: workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  const bool impute = (flags & DPB_SAMPLER_IMPUTE) != 0, given = (flags & DPB_SAMPLER_NOISE_GIVEN) != 0;
  if (given) DPB_REQUIRE(noise, "dpb_sampler_run_pc: DPB_SAMPLER_NOISE_GIVEN without a noise tensor");
  const int noise_k = impute ? 3 : 1;
  if (pick_engine(h, flags, B, true) == DPB_ENGINE_TC && tc_pc_possible(h, B, tbl->n_steps)) {
    // ONE persistent kernel for all steps: the corrector's batch norms cross the grid through a counter barrier
    // (score_tc.cu, pc mode).  Columns 5 / 6 of the coefficient table take the per-step score scale and alpha.
    float* coef = const_cast<float*>(tbl->coef);
    DPB_CUDA_CHECK(cudaMemcpy2DAsync(coef + 5, DPB_COEF_STRIDE * sizeof(float), score_scale, sizeof(float), sizeof(float),
                                     tbl->n_steps, cudaMemcpyHostToDevice, st));
    DPB_CUDA_CHECK(cudaMemcpy2DAsync(coef + 6, DPB_COEF_STRIDE * sizeof(float), lang_alpha, sizeof(float), sizeof(float),
                                     tbl->n_steps, cudaMemcpyHostToDevice, st));
    TcJob j{};
    j.mode = 1; j.B = B; j.x_io = x_io; j.table = tbl->time_table; j.coef = tbl->coef; j.n_steps = tbl->n_steps;
    j.obs = obs; j.mask = mask; j.noise = given ? noise : nullptr; j.noise_k = noise_k;
    j.seed = seed; j.step_offset = step_offset; j.traj = traj; j.x_mean = x_mean; j.impute = impute ? 1 : 0;
    j.pc = 1; j.snr = snr;
    return tc_launch(h, j, st);
  }
  WsCarver c(ws, ws_bytes);
  float* grad = c.take<float>((size_t)B * h->pose_dim);
  float* z = c.take<float>((size_t)B * h->pose_dim);
  float* sums = c.take<float>(2);
  c.off = align_up(c.off, 256);
  void* rest = static_cast<uint8_t*>(ws) + c.off;
  const size_t rest_bytes = ws_bytes - c.off;
  const int kp = noise_k;                              // predictor planes per step; the Langevin draw comes first
  const size_t plane = (size_t)B * h->pose_dim;
  for (int i = 0; i < tbl->n_steps; ++i) {
    const float* table_i = tbl->time_table + (size_t)i * NL * H;
    int rc = dpb_score_forward(h, x_io, table_i, nullptr, nullptr, score_scale[i], grad, B, flags & DPB_ENGINE_MASK, rest,
                               rest_bytes, stream);
    if (rc != DPB_OK) return rc;
    const float* zi = z;
    if (given) zi = noise + (size_t)i * (kp + 1) * plane;
    else if ((rc = dpb_normal_fill_dim(z, B, seed, step_offset + (uint64_t)i, 4, h->pose_dim, stream)) != DPB_OK) return rc;
    DPB_CUDA_CHECK(cudaMemsetAsync(sums, 0, 2 * sizeof(float), st));
    if ((rc = dpb_langevin_norms_dim(grad, zi, sums, B, h->pose_dim, stream)) != DPB_OK) return rc;
    if ((rc = dpb_langevin_update_dim(x_io, nullptr, grad, zi, sums, snr, lang_alpha[i], B, h->pose_dim, stream)) != DPB_OK)
      return rc;
    dpb_step_tables one{};
    one.n_steps = 1;
    one.coef = tbl->coef + (size_t)i * DPB_COEF_STRIDE;
    one.time_table = table_i;
    rc = dpb_sampler_run(h, x_io, &one, obs, mask, given ? noise + ((size_t)i * (kp + 1) + 1) * plane : nullptr, seed,
                         step_offset + (uint64_t)i, traj ? traj + (size_t)i * plane : nullptr, x_mean, B, flags, rest,
                         rest_bytes, stream);
    if (rc != DPB_OK) return rc;
  }
  return DPB_OK;
}

extern "C" size_t dpb_score_jvp_workspace_bytes(dpb_score_t* h, int64_t B) {
  if (!h || B <= 0) return 0;
  const int dp = h->pose_dp;
  const size_t simt = simt_forward_ws_bytes(2 * B, dp), tc = score_jvp_tc_ws_bytes(B, dp);
  return (simt > tc ? simt : tc) + align_up((size_t)2 * B * dp * 4, 256) + 1024;
}

extern "C" int dpb_score_jvp(dpb_score_t* h, const float* x, const float* v, const float* table, const int32_t* t_index,
                             const float* row_scale, float scale, float* out, float* jv, int64_t B, void* ws,
                             size_t ws_bytes, void* stream) {
  if (!h) return fail(DPB_EINVAL, "dpb_score_jvp: null handle");
  DeviceGuard guard(h->device);
  DPB_REQUIRE(x && v && table && out && jv, "dpb_score_jvp: x, v, table, out and jv are required");
  if (B <= 0) return DPB_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const int dp = h->pose_dp;
  WsCarver c(ws, ws_bytes);
  float* raw = c.take<float>((size_t)2 * B * dp);
  if (!c.ok() || ws == nullptr || ws_bytes < dpb_score_jvp_workspace_bytes(h, B))
    return fail(DPB_ENOMEM, "dpb_score_jvp: workspace too small");
  void* rest = static_cast<uint8_t*>(ws) + c.off;
  // batch-uniform time (the likelihood's case): every contraction on tcgen05; per-row tables keep the fp32 SGEMM path
  int rc = !t_index ? score_jvp_tc_raw(h, x, v, table, raw, B, rest, ws_bytes - c.off, st)
                    : simt_forward_jvp_raw(h, x, v, table, t_index, raw, B, rest, ws_bytes - c.off, st);
  if (rc != DPB_OK) return rc;
  rc = launch_scale_out(raw, row_scale, scale, out, B, dp, st);
  if (rc != DPB_OK) return rc;
  return launch_scale_out(raw + (size_t)B * dp, row_scale, scale, jv, B, dp, st);   // the scaling is linear: same factor
}

extern "C" int dpb_sampler_run(dpb_score_t* h, float* x_io, const dpb_step_tables* tbl, const float* obs,
                               const float* mask, const float* noise, uint64_t seed, uint64_t step_offset,
                               float* traj, float* x_mean, int64_t B, int flags, void* ws, size_t ws_bytes,
                               void* stream) {
  if (!h || !tbl) return fail(DPB_EINVAL, "dpb_sampler_run: null handle or tables");
  DeviceGuard guard(h->device);
  DPB_REQUIRE(x_io && tbl->coef && tbl->time_table && tbl->n_steps >= 0, "dpb_sampler_run: bad tables / x_io");
  const int impute = (flags & DPB_SAMPLER_IMPUTE) ? 1 : 0;
  const bool given = (flags & DPB_SAMPLER_NOISE_GIVEN) != 0;
  if (impute) DPB_REQUIRE(obs && mask, "dpb_sampler_run: completion needs observation and mask");
  if (given) DPB_REQUIRE(noise, "dpb_sampler_run: DPB_SAMPLER_NOISE_GIVEN without a noise tensor");
  if (B <= 0 || tbl->n_steps == 0) return DPB_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const int noise_k = impute ? 3 : 1;
  const int engine = pick_engine(h, flags, B, true);
  if (engine == DPB_ENGINE_TC) {
    if (!h->tc_ready) return fail(DPB_EUNSUPPORTED, "dpb_sampler_run: tcgen05 engine unavailable");
    TcJob j{};
    j.mode = 1; j.B = B; j.x_io = x_io; j.table = tbl->time_table; j.coef = tbl->coef; j.n_steps = tbl->n_steps;
    j.obs = obs; j.mask = mask; j.noise = given ? noise : nullptr; j.noise_k = noise_k;
    j.seed = seed; j.step_offset = step_offset; j.traj = traj; j.x_mean = x_mean; j.impute = impute;
    return tc_launch(h, j, st);
  }
  ScoreWs w;
  if (!carve_score_ws(h, B, ws, ws_bytes, &w)) return fail(DPB_ENOMEM, "dpb_sampler_run: workspace too small");
  const size_t plane = (size_t)B * h->pose_dim;
  for (int i = 0; i < tbl->n_steps; ++i) {
    const float* coef = tbl->coef + (size_t)i * DPB_COEF_STRIDE;
    const float* nz = given ? noise + (size_t)i * noise_k * plane : nullptr;
    const uint32_t step = (uint32_t)(step_offset + (uint64_t)i);
    int rc = DPB_OK;
    if (impute) rc = launch_impute(x_io, coef, obs, mask, nz, seed, step, B, h->pose_dp, st);
    if (rc == DPB_OK)
      rc = simt_forward_raw(h, x_io, tbl->time_table + (size_t)i * NL * H, nullptr, w.raw, B, w.rest, w.rest_bytes, st);
    if (rc == DPB_OK)
      rc = launch_em_update(x_io, w.raw, coef, obs, mask, nz, noise_k, seed, step,
                            traj ? traj + (size_t)i * plane : nullptr, x_mean, B, impute, h->pose_dp, st);
    if (rc != DPB_OK) return rc;
  }
  return DPB_OK;
}

extern "C" int dpb_prior_loss(dpb_score_t* h, const float* x0, const float* table, float alpha, float sd,
                              float inv_sigma_std, int weighted, float divisor, const float* z, uint64_t seed,
                              uint64_t step, float* loss_out, float* grad_out, float* row_loss, int64_t B, int flags,
                              void* ws, size_t ws_bytes, void* stream) {
  if (!h) return fail(DPB_EINVAL, "dpb_prior_loss: null handle");
  DeviceGuard guard(h->device);
  DPB_REQUIRE(x0 && table && loss_out, "dpb_prior_loss: x0, table and loss_out are required");
  DPB_REQUIRE(divisor > 0.f && alpha > 0.f, "dpb_prior_loss: divisor and alpha must be positive");
  if (B <= 0) return DPB_OK;
  cudaStream_t st = (cudaStream_t)stream;
  // SNR = alpha / sqrt(std^2) (run/completion.py:108); w = 0.5 sqrt(1+SNR) or 0.5
  const float wgt = weighted ? 0.5f * sqrtf(1.0f + alpha / sqrtf(sd * sd)) : 0.5f;
  const int engine = pick_engine(h, flags, B, true);
  if (engine == DPB_ENGINE_TC) {
    if (!h->tc_ready) return fail(DPB_EUNSUPPORTED, "dpb_prior_loss: tcgen05 engine unavailable");
    TcJob j{};
    j.mode = 2; j.B = B; j.x_in = x0; j.table = table; j.n_steps = 1;
    j.alpha = alpha; j.std = sd; j.inv_sigma_std = inv_sigma_std; j.divisor = divisor; j.weighted = weighted;
    j.z = z; j.seed = seed; j.step_offset = step; j.loss_out = loss_out; j.grad_out = grad_out; j.row_loss = row_loss;
    j.scale = wgt;
    DPB_CUDA_CHECK(cudaMemsetAsync(loss_out, 0, sizeof(float), st));
    return tc_launch(h, j, st);
  }
  ScoreWs w;
  if (!carve_score_ws(h, B, ws, ws_bytes, &w)) return fail(DPB_ENOMEM, "dpb_prior_loss: workspace too small");
  int rc = launch_perturb(x0, z, seed, (uint32_t)step, alpha, sd, w.xt, B, h->pose_dp, st);
  if (rc == DPB_OK) rc = simt_forward_raw(h, w.xt, table, nullptr, w.raw, B, w.rest, w.rest_bytes, st);
  if (rc == DPB_OK)
    rc = launch_prior_loss(x0, w.xt, w.raw, alpha, sd, inv_sigma_std, wgt, 1.0f / divisor, loss_out, grad_out,
                           row_loss, B, h->pose_dp, st);
  return rc;
}
