// rd_dreamer.cuh -- host-side orchestration of the on-device Dreamer agent (SURVEY.md §8-f2).
//
// One agent step = RacingDreamer.action [REF ros_agent/models/dreamer/racing_dreamer.py:62-82] for every env:
//   img1 -> GRU cell -> obs1 (concat([deter, embed])) -> obs2 + posterior sample -> actor h0..h3 -> hout + mode()
// = k_embed_lidar, five launches of k_dense, one of k_dense_chain (the actor trunk; with RD_DREAMER_HEAD=1 and up to
// 33 x 128 envs also hout, which is the fifth k_dense launch otherwise) and k_actor_mode (rd_gemm.cuh);
// activations live in a handful of [envs][width] float32 arrays that stay in
// L2 between launches, the recurrent state in two ping-pong "latent" arrays whose rows are
//   [ stoch (30) | previous action (2) | deter (200) ]          (232 floats, 928 bytes)
// so that img1's input concat([stoch, action]), the GRU's state, obs1's concat([deter, ...]) and the actor's
// concat([stoch, deter]) are all plain TMA views of one row (the actor's weight rows for the two action slots are
// zero).  The prior head (img2/img3) only feeds a sample that obs_step's caller discards and is not evaluated.
#pragma once
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "rd_gemm.cuh"

// Actor trunk (400-wide Dense layers) in float32-grade mode: output columns per CTA, ring stages, epilogue groups.
// 128-wide tiles make 4 N tiles instead of 7: 128 CTAs, one per SM (two 64-wide CTAs on half the SMs share the SM's L2
// ingress), which also leaves room for three 64 KB stages and four epilogue groups.  Measured: 64/2/2 0.190 ms,
// 128/2/2 0.191, 128/2/4 0.188, 128/3/4 0.181 ms per agent step.
#ifndef DR_ACT_BN
#define DR_ACT_BN 128
#define DR_ACT_STAGES 3
#define DR_ACT_EW 4
#endif

// epilogue warp groups of the launches that have an SM to themselves (GRU cell, obs1, obs2 + posterior)
#ifndef DR_EW_WIDE
#define DR_EW_WIDE 4
#endif

struct DreamerPolicy {
  bool ready = false;
  int n = 0, deter = 0, hidden = 0, embed = 0, units = 0, layers = 0, ldf = 0;
  float raw_init_std = 0.f, min_std = 0.f, mean_scale = 0.f, bn_eps = 0.f;
  int n_samples = 0;
  bool lidar_normalised = false;
  bool x3 = true;        // three-pass hi/lo TF32 products (float32-grade) instead of one TF32 pass
  std::vector<float*> owned;   // every device allocation of this policy
  // an MMA operand: device array(s) of TF32-representable values ([1] = remainder part, x3 mode) and their TMA views
  struct Operand { float* p[2] = {nullptr, nullptr}; CUtensorMap m[2]; };
  // weights (transposed: [out][in]) and biases
  Operand w_img1, w_gruk, w_grur, w_obs1, w_obs2, w_act[8];
  float *b_img1 = nullptr, *b_gru = nullptr, *b_obs1 = nullptr, *b_obs2 = nullptr, *bn = nullptr;
  float* b_act[8] = {};
  // activations.  feat[p]: latent rows; sa/det/all are views of the same rows (img1 input, deter, actor input)
  Operand feat[2], v_sa[2], v_det[2], x1, hobs, hid[2], lidar;
  float* head_raw = nullptr;   // [n][4] hout pre-activations
  // k_dense_chain (the actor trunk in one launch): per-row-block layer counters and the values they have reached
  bool chain = true;           // RD_DREAMER_CHAIN=0: one k_dense launch per actor layer instead
  bool head_fused = false;     // RD_DREAMER_HEAD=1: hout inside the last k_dense_chain launch (cluster launches of <= 33 row
                               // blocks).  Opt-in: 4 % faster, tests / memcheck / synccheck green, but racecheck flags the
                               // remote stores ("block might not have entered yet"), see profiles/r5b_dreamer_chain.txt
  bool chain_cluster = true;   // the N tiles of a row block are launched as a thread-block cluster (RD_DREAMER_CLUSTER=0: plain grid)
  bool tma_out = true;         // RD_DREAMER_TMA_OUT=0: Dense / GRU epilogues store from registers (see gm_stage_f4)
  unsigned* chain_flags = nullptr;
  unsigned chain_count[GM_CHAIN_MAX] = {};
  int sm_count = 148;
  int cur = 0;           // feat[cur] holds the latest latent
  uint32_t step = 0;     // agent steps taken (Philox counter)
  // training-mode exploration [REF dreamer/dreamer.py, Dreamer._exploration]: amount * 0.5^(env_steps / decay) (decay > 0),
  // at least min_amount (min_amount > 0); env_steps = Dreamer's step counter, + n_envs * action_repeat per training step
  double expl_amount = 0.3, expl_decay = 0.0, expl_min = 0.0;
  int64_t env_steps = 0;
  float* stage = nullptr;      // device copy of host-pointer weights for dreamer_set_weights (sized at init)
  std::string err;
};

static inline float dr_tf32(float x) {   // cvt.rna.tf32.f32 on the host (finite values)
  uint32_t u;
  std::memcpy(&u, &x, 4);
  u = (u + 0x1000u) & ~0x1fffu;
  std::memcpy(&x, &u, 4);
  return x;
}

static inline void dreamer_free(DreamerPolicy& d) {
  for (float* p : d.owned) cudaFree(p);
  d.owned.clear();
  d.bn = nullptr;
  d.stage = nullptr;
  d.ready = false;
}

// The policy's weight layout: each checkpoint array, where it goes and how.  Matrices ([in][out] Keras kernels) become
// K-major TF32 operands (dr_upload_t: pitch ld, the K slots from k_from on shifted by k_shift); vectors (op == null)
// are copied as they are to *vec.  Both dreamer_init and dreamer_set_weights walk this one list.
struct DrPart { const float* src; DreamerPolicy::Operand* op; float** vec; int in, out, ld, k_from, k_shift; };
static inline int dr_parts(DreamerPolicy& d, const rd_dreamer_weights* w, DrPart* p) {
  const int H = d.hidden, D = d.deter, E = d.embed, U = d.units, L = d.layers, NO = 1 << 30;
  int k = 0;
  auto mat = [&](const float* src, DreamerPolicy::Operand& op, int in, int out, int ld, int k_from, int k_shift) {
    p[k++] = DrPart{src, &op, nullptr, in, out, ld, k_from, k_shift};
  };
  auto vec = [&](const float* src, float*& dst, int count) { p[k++] = DrPart{src, nullptr, &dst, 1, count, 0, NO, 0}; };
  mat(w->img1_w, d.w_img1, GM_STOCH + 2, H, 32, NO, 0);
  vec(w->img1_b, d.b_img1, H);
  mat(w->gru_kernel, d.w_gruk, H, 3 * D, H, NO, 0);
  mat(w->gru_recurrent, d.w_grur, D, 3 * D, D, NO, 0);
  vec(w->gru_bias, d.b_gru, 6 * D);
  mat(w->obs1_w, d.w_obs1, D + E, H, D + E, NO, 0);
  vec(w->obs1_b, d.b_obs1, H);
  mat(w->obs2_w, d.w_obs2, H, 2 * GM_STOCH, H, NO, 0);
  vec(w->obs2_b, d.b_obs2, 2 * GM_STOCH);
  // actor h0: rows [stoch | deter] -> K slots [0, 30) and [32, 32 + deter); the two action slots get zero weights
  mat(w->actor_w[0], d.w_act[0], GM_STOCH + D, U, d.ldf, GM_STOCH, 2);
  vec(w->actor_b[0], d.b_act[0], U);
  for (int i = 1; i < L; ++i) {
    mat(w->actor_w[i], d.w_act[i], U, U, U, NO, 0);
    vec(w->actor_b[i], d.b_act[i], U);
  }
  mat(w->actor_w[L], d.w_act[L], U, 4, U, NO, 0);
  vec(w->actor_b[L], d.b_act[L], 4);
  if (w->bn) vec(w->bn, d.bn, 16);
  return k;
}
#define DR_MAX_PARTS (9 + 2 * 8 + 1)

// [in][out] host matrix -> device [out][ld] (K-major), element (o, kmap(i)) = scale_i * W[i][o], split into its TF32
// rounding (op.p[0]) and, in x3 mode, the TF32 rounding of the remainder (op.p[1])
static inline cudaError_t dr_upload_t(DreamerPolicy& d, DreamerPolicy::Operand& op, const float* w, int in, int out, int ld,
                                      int k_shift_from, int k_shift, const std::vector<float>* col_scale = nullptr) {
  std::vector<float> hi((size_t)out * ld, 0.f), lo((size_t)out * ld, 0.f);
  for (int i = 0; i < in; ++i) {
    const int k = i >= k_shift_from ? i + k_shift : i;
    const float sc = col_scale ? (*col_scale)[i] : 1.f;
    for (int o = 0; o < out; ++o) {
      const float x = w[(size_t)i * out + o] * sc, h = dr_tf32(x);
      hi[(size_t)o * ld + k] = h;
      lo[(size_t)o * ld + k] = dr_tf32(x - h);
    }
  }
  for (int part = 0; part < (d.x3 ? 2 : 1); ++part) {
    cudaError_t e = cudaMalloc(&op.p[part], hi.size() * sizeof(float));
    if (e != cudaSuccess) return e;
    d.owned.push_back(op.p[part]);
    e = cudaMemcpy(op.p[part], (part ? lo : hi).data(), hi.size() * sizeof(float), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) return e;
  }
  return cudaSuccess;
}
static inline cudaError_t dr_upload(DreamerPolicy& d, float** dst, const float* v, size_t count) {
  cudaError_t e = cudaMalloc(dst, count * sizeof(float));
  if (e != cudaSuccess) return e;
  d.owned.push_back(*dst);
  return cudaMemcpy(*dst, v, count * sizeof(float), cudaMemcpyHostToDevice);
}
// zero-initialised activation array(s) [rows][ld]
static inline cudaError_t dr_alloc(DreamerPolicy& d, DreamerPolicy::Operand& op, size_t rows, size_t ld) {
  for (int part = 0; part < (d.x3 ? 2 : 1); ++part) {
    cudaError_t e = cudaMalloc(&op.p[part], rows * ld * sizeof(float));
    if (e != cudaSuccess) return e;
    d.owned.push_back(op.p[part]);
    e = cudaMemset(op.p[part], 0, rows * ld * sizeof(float));
    if (e != cudaSuccess) return e;
  }
  return cudaSuccess;
}
// TMA views of both parts: columns [col0, col0 + inner) of rows of pitch ld
static inline bool dr_view(const DreamerPolicy& d, DreamerPolicy::Operand& view, const DreamerPolicy::Operand& base, size_t col0,
                           uint64_t inner, uint64_t rows, uint64_t ld, uint32_t box_rows) {
  for (int part = 0; part < (d.x3 ? 2 : 1); ++part) {
    view.p[part] = base.p[part] + col0;
    if (!gm_make_map(&view.m[part], view.p[part], inner, rows, ld, box_rows)) return false;
  }
  return true;
}

#define DR_TRY(expr)                                                                            \
  do {                                                                                          \
    cudaError_t e_ = (expr);                                                                    \
    if (e_ != cudaSuccess) { cudaGetLastError(); d.err = std::string(#expr) + ": " + cudaGetErrorString(e_); return RD_ERR_CUDA; } \
  } while (0)
#define DR_MAP(expr)                                                                            \
  do {                                                                                          \
    if (!(expr)) { d.err = "cuTensorMapEncodeTiled failed: " #expr; return RD_ERR_CUDA; }       \
  } while (0)

// lidar_normalised: the env already emits r/15 - 0.5 (RD_OBS_LIDAR_NORM), so k_embed_lidar only splits the values
static inline int dreamer_init(DreamerPolicy& d, int n, int n_beams, bool lidar_normalised, const rd_dreamer_weights* w) {
  if (!w) { d.err = "null weights"; return RD_ERR_INVALID; }
  if (w->stoch != GM_STOCH || w->deter <= 0 || w->deter % 4 || w->hidden <= 0 || w->hidden % 4 || w->embed != n_beams ||
      n_beams % 4 || w->actor_units <= 0 || w->actor_units % 4 || w->actor_layers < 1 || w->actor_layers > 7 ||
      w->n_samples < 1 || !(w->mean_scale > 0.f)) {
    d.err = "unsupported Dreamer architecture (need stoch 30, deter/hidden/units/embed multiples of 4, embed == n_beams, 1..7 actor layers)";
    return RD_ERR_INVALID;
  }
  const float* need[] = {w->gru_kernel, w->gru_recurrent, w->gru_bias, w->img1_w, w->img1_b, w->obs1_w, w->obs1_b, w->obs2_w, w->obs2_b};
  for (const float* p : need)
    if (!p) { d.err = "null weight pointer"; return RD_ERR_INVALID; }
  for (int i = 0; i <= w->actor_layers; ++i)
    if (!w->actor_w[i] || !w->actor_b[i]) { d.err = "null actor weight pointer"; return RD_ERR_INVALID; }
  if (!gm_get_encoder()) { d.err = "cuTensorMapEncodeTiled is not available from this driver"; return RD_ERR_CUDA; }
  if (w->precision != RD_PRECISION_TF32X3 && w->precision != RD_PRECISION_TF32) { d.err = "bad precision"; return RD_ERR_INVALID; }
  dreamer_free(d);
  d.x3 = w->precision == RD_PRECISION_TF32X3;
  d.lidar_normalised = lidar_normalised;
  d.n = n; d.deter = w->deter; d.hidden = w->hidden; d.embed = w->embed; d.units = w->actor_units; d.layers = w->actor_layers;
  d.ldf = 32 + d.deter;
  d.raw_init_std = (float)std::log(std::exp((double)w->init_std) - 1.0);   // [REF models.py:321]
  d.min_std = w->min_std; d.mean_scale = w->mean_scale; d.bn_eps = w->bn_eps; d.n_samples = w->n_samples;
  const int H = d.hidden, D = d.deter, E = d.embed, U = d.units;
  DrPart parts[DR_MAX_PARTS];
  const int n_parts = dr_parts(d, w, parts);
  size_t stage_floats = 0;
  for (int k = 0; k < n_parts; ++k) {
    const DrPart& p = parts[k];
    if (p.op) DR_TRY(dr_upload_t(d, *p.op, p.src, p.in, p.out, p.ld, p.k_from, p.k_shift));
    else DR_TRY(dr_upload(d, p.vec, p.src, (size_t)p.out));
    stage_floats += (size_t)p.in * p.out;
  }
  DR_TRY(cudaMalloc(&d.stage, stage_floats * sizeof(float)));
  d.owned.push_back(d.stage);
  const size_t N = (size_t)n;
  for (int p = 0; p < 2; ++p) {
    DR_TRY(dr_alloc(d, d.feat[p], N, d.ldf));
    DR_TRY(dr_alloc(d, d.hid[p], N, U));
  }
  DR_TRY(cudaMalloc(&d.head_raw, N * 4 * sizeof(float)));
  d.owned.push_back(d.head_raw);
  {
    const size_t row_blocks = (N + GM_BM - 1) / GM_BM;
    DR_TRY(cudaMalloc(&d.chain_flags, GM_CHAIN_MAX * row_blocks * sizeof(unsigned)));
    d.owned.push_back(reinterpret_cast<float*>(d.chain_flags));
    DR_TRY(cudaMemset(d.chain_flags, 0, GM_CHAIN_MAX * row_blocks * sizeof(unsigned)));
    for (unsigned& c : d.chain_count) c = 0;
    int dev = 0;
    DR_TRY(cudaGetDevice(&dev));
    DR_TRY(cudaDeviceGetAttribute(&d.sm_count, cudaDevAttrMultiProcessorCount, dev));
    d.chain = true;
    if (const char* ev = std::getenv("RD_DREAMER_CHAIN")) d.chain = std::atoi(ev) != 0;
    d.head_fused = false;
    if (const char* ev = std::getenv("RD_DREAMER_HEAD")) d.head_fused = std::atoi(ev) != 0;
    d.chain_cluster = true;
    if (const char* ev = std::getenv("RD_DREAMER_CLUSTER")) d.chain_cluster = std::atoi(ev) != 0;
    d.tma_out = true;
    if (const char* ev = std::getenv("RD_DREAMER_TMA_OUT")) d.tma_out = std::atoi(ev) != 0;
  }
  DR_TRY(dr_alloc(d, d.x1, N, H));
  DR_TRY(dr_alloc(d, d.hobs, N, H));
  DR_TRY(dr_alloc(d, d.lidar, N, E));   // the embedded scans (k_embed_lidar)
  for (int p = 0; p < 2; ++p) {
    DR_MAP(dr_view(d, d.v_sa[p], d.feat[p], 0, 32, N, d.ldf, GM_BM));
    DR_MAP(dr_view(d, d.v_det[p], d.feat[p], 32, D, N, d.ldf, GM_BM));
    DR_MAP(dr_view(d, d.feat[p], d.feat[p], 0, d.ldf, N, d.ldf, GM_BM));
    DR_MAP(dr_view(d, d.hid[p], d.hid[p], 0, U, N, U, GM_BM));
  }
  DR_MAP(dr_view(d, d.x1, d.x1, 0, H, N, H, GM_BM));
  DR_MAP(dr_view(d, d.hobs, d.hobs, 0, H, N, H, GM_BM));
  DR_MAP(dr_view(d, d.lidar, d.lidar, 0, E, N, E, GM_BM));
  DR_MAP(dr_view(d, d.w_img1, d.w_img1, 0, 32, H, 32, GM_BN));
  DR_MAP(dr_view(d, d.w_gruk, d.w_gruk, 0, H, 3 * D, H, GM_BN));
  DR_MAP(dr_view(d, d.w_grur, d.w_grur, 0, D, 3 * D, D, GM_BN));
  DR_MAP(dr_view(d, d.w_obs1, d.w_obs1, 0, D + E, H, D + E, GM_BN));
  DR_MAP(dr_view(d, d.w_obs2, d.w_obs2, 0, H, 2 * GM_STOCH, H, GM_BN));
  DR_MAP(dr_view(d, d.w_act[0], d.w_act[0], 0, d.ldf, U, d.ldf, d.x3 ? DR_ACT_BN : GM_BN));
  for (int i = 1; i < d.layers; ++i) DR_MAP(dr_view(d, d.w_act[i], d.w_act[i], 0, U, U, U, d.x3 ? DR_ACT_BN : GM_BN));
  DR_MAP(dr_view(d, d.w_act[d.layers], d.w_act[d.layers], 0, U, 4, U, GM_BN));
  d.cur = 0;
  d.step = 0;
  d.env_steps = 0;
  d.ready = true;
  return RD_OK;
}

// the exploration amount of the next training step, rounded once to float32
static inline float dreamer_expl_amount(const DreamerPolicy& d) {
  double a = d.expl_amount;
  if (d.expl_decay > 0.0) a *= std::pow(0.5, (double)d.env_steps / d.expl_decay);
  if (d.expl_min > 0.0) a = std::max(d.expl_min, a);
  return (float)a;
}

// New values for every weight of an initialised policy, packed on the device on `s` into the buffers it already owns
// (no allocation; the tensor maps stay valid) bit for bit as dreamer_init packs them.  Latent state, Philox step and
// env_steps are kept.  w holds device pointers (on_device) or host pointers, which are first copied to d.stage.  The
// architecture, precision and head scalars must be the init's; otherwise RD_ERR_INVALID and nothing changes.
static inline int dreamer_set_weights(DreamerPolicy& d, const rd_dreamer_weights* w, bool on_device, cudaStream_t s) {
  if (!w) { d.err = "null weights"; return RD_ERR_INVALID; }
  const float raw_init_std = (float)std::log(std::exp((double)w->init_std) - 1.0);
  if (w->stoch != GM_STOCH || w->deter != d.deter || w->hidden != d.hidden || w->embed != d.embed ||
      w->actor_units != d.units || w->actor_layers != d.layers || (w->bn != nullptr) != (d.bn != nullptr) ||
      (w->precision != RD_PRECISION_TF32X3 && w->precision != RD_PRECISION_TF32) ||
      (w->precision == RD_PRECISION_TF32X3) != d.x3 || w->n_samples != d.n_samples || raw_init_std != d.raw_init_std ||
      w->min_std != d.min_std || w->mean_scale != d.mean_scale || w->bn_eps != d.bn_eps) {
    d.err = "the weights' architecture, precision or head scalars differ from the ones the policy was initialised with";
    return RD_ERR_INVALID;
  }
  DrPart parts[DR_MAX_PARTS];
  const int n_parts = dr_parts(d, w, parts);
  int dev = 0;
  DR_TRY(cudaGetDevice(&dev));
  for (int k = 0; k < n_parts; ++k) {
    if (!parts[k].src) { d.err = "null weight pointer"; return RD_ERR_INVALID; }
    cudaPointerAttributes at{};
    DR_TRY(cudaPointerGetAttributes(&at, parts[k].src));
    const bool device_ptr = at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged;
    if (on_device && (!device_ptr || at.device != dev)) { d.err = "on_device: a weight pointer is not memory of the policy's device"; return RD_ERR_INVALID; }
    if (!on_device && at.type == cudaMemoryTypeDevice) { d.err = "a device pointer was passed with on_device = 0"; return RD_ERR_INVALID; }
  }
  PackArgs a{};
  a.n_jobs = n_parts;
  size_t off = 0;
  for (int k = 0; k < n_parts; ++k) {
    const DrPart& p = parts[k];
    const size_t count = (size_t)p.in * p.out;
    const float* src = p.src;
    if (!on_device) {
      DR_TRY(cudaMemcpyAsync(d.stage + off, p.src, count * sizeof(float), cudaMemcpyHostToDevice, s));
      src = d.stage + off;
    }
    PackJob& J = a.job[k];
    J.src = src;
    J.hi = p.op ? p.op->p[0] : *p.vec;
    J.lo = p.op ? p.op->p[1] : nullptr;
    J.in = p.in; J.out = p.out; J.ld = p.ld; J.k_from = p.k_from; J.k_shift = p.k_shift; J.raw = p.op ? 0 : 1;
    J.begin = (long long)off;
    off += count;
  }
  a.total = (long long)off;
  const unsigned grid = (unsigned)std::min<size_t>((off + 255) / 256, (size_t)d.sm_count * 8);
  k_pack_weights<<<grid, 256, 0, s>>>(a);
  DR_TRY(cudaGetLastError());
  return RD_OK;
}

// One layer's launch description: up to two (A source, W, K range) terms.  dr_build expands them into phases:
// in x3 mode first the lo*hi and hi*lo passes of every term (into the "small" accumulator group), then the hi*hi pass
// cut into K groups of at most ~6 blocks, one accumulator group each (see "truncation" in rd_gemm.cuh).
// Accumulator slot = group * gates + gate; `gate[t][i]` maps slab i of term t to its gate (Dense layers: one gate).
struct DrTerm { const DreamerPolicy::Operand* a; const DreamerPolicy::Operand* w; int k_elems; int w_k0; };
static inline void dr_build(const DreamerPolicy& d, GemmMaps& maps, GemmArgs& g, const DrTerm* terms, int n_terms, int nb,
                            const int* w_row0, const int (*gate)[3], int gates, int slots) {
  g.n_phases = 0;
  int small_group = 0;   // the accumulator group of the cross products (set below, before the first add)
  auto add = [&](int t, int a_part, int w_part, int kb0, int kbs, int group) {
    GemmPhase& p = g.ph[g.n_phases++];
    p = GemmPhase{};
    p.a_map = 2 * t + a_part;   // maps.a / maps.w slots: term t -> hi at 2t, lo at 2t + 1
    p.w_map = 2 * t + w_part;
    p.a_map_lo = 2 * t + 1;     // X3 kernels: the lo parts ride in the same K block (k_dense<..., X3 = true>)
    p.w_map_lo = 2 * t + 1;
    p.k_blocks = kbs;
    p.a_k0 = kb0 * GM_BK;
    p.w_k0 = terms[t].w_k0 + kb0 * GM_BK;
    p.nb = nb;
    for (int i = 0; i < nb; ++i) {
      p.w_row0[i] = w_row0 ? w_row0[i] : 0;
      p.acc[i] = group * gates + (gate ? gate[t][i] : 0);
      p.acc_small[i] = small_group * gates + (gate ? gate[t][i] : 0);
    }
  };
  int total = 0;
  for (int t = 0; t < n_terms; ++t) {
    maps.a[2 * t] = terms[t].a->m[0];
    maps.w[2 * t] = terms[t].w->m[0];
    if (d.x3) { maps.a[2 * t + 1] = terms[t].a->m[1]; maps.w[2 * t + 1] = terms[t].w->m[1]; }
    total += (terms[t].k_elems + GM_BK - 1) / GM_BK;
  }
  const int max_groups = slots / gates - (d.x3 ? 1 : 0);
  const int groups = std::max(1, std::min(max_groups, (total + 5) / 6));
  small_group = groups;
  // x3: no separate lo*hi / hi*lo passes -- every hi*hi K block below carries the lo tiles and feeds all three products
  // hi*hi: walk the concatenated K blocks, group boundaries every total/groups blocks
  int done = 0;
  for (int t = 0; t < n_terms; ++t) {
    const int kbs = (terms[t].k_elems + GM_BK - 1) / GM_BK;
    int kb = 0;
    while (kb < kbs) {
      const int grp = std::min(groups - 1, (int)(((long long)(done + kb) * groups) / total));
      const int grp_end = (int)(((long long)(grp + 1) * total + groups - 1) / groups) - done;   // first block of the next group
      const int stop = grp == groups - 1 ? kbs : std::min(kbs, std::max(kb + 1, grp_end));
      add(t, 0, 0, kb, stop - kb, grp);
      kb = stop;
    }
    done += kbs;
  }
  g.n_acc = groups + (d.x3 ? 1 : 0);
}

// Enqueues one agent step for all envs on `s`; returns the number of kernels launched in *launched.
// train: null = evaluation mode (SampleDist.mode(), eps_actor [N][n_samples][2]); else the training head k_actor_train
// with exploration amount train->amount (eps_actor = the sample's draws [N][2], train->eps_expl the exploration's).
struct DrTrain { const float* eps_expl; float amount; };
static inline int dreamer_step(DreamerPolicy& d, const float* lidar, float* actions, int noise, const float* eps_stoch,
                               const float* eps_actor, float* debug, uint64_t seed, uint32_t gid0, cudaStream_t s, int* launched,
                               const DrTrain* train = nullptr) {
  *launched = 0;
  const int cur = d.cur, nxt = cur ^ 1;
  const int H = d.hidden, D = d.deter, U = d.units;
  {   // 0. embed = _preprocess_lidar(scan), split for the tensor-core passes
    const size_t count4 = (size_t)d.n * d.embed / 4;
    const unsigned grid = (unsigned)std::min<size_t>((count4 + 255) / 256, 148 * 8);
    k_embed_lidar<<<grid, 256, 0, s>>>(reinterpret_cast<const float4*>(lidar), reinterpret_cast<float4*>(d.lidar.p[0]),
                                       reinterpret_cast<float4*>(d.lidar.p[1]), count4, d.lidar_normalised ? 0 : 1);
    DR_TRY(cudaGetLastError());
    ++*launched;
  }
  GemmMaps maps;
  // 1. img1: x1 = elu(concat([stoch, action]) @ W + b) [REF models.py:78-80]
  {
    GemmArgs g{};
    g.M = d.n; g.N = H;
    const DrTerm t[1] = {{&d.v_sa[cur], &d.w_img1, 32, 0}};
    dr_build(d, maps, g, t, 1, 1, nullptr, nullptr, 1, 4);
    g.step = d.step; g.bias = d.b_img1; g.out = d.x1.p[0]; g.out_lo = d.x1.p[1]; g.ldo = H; g.act = 1;
    g.tma_out = d.tma_out; maps.o[0] = d.x1.m[0]; maps.o[1] = d.x1.m[1];
    if (d.x3) DR_TRY((gm_launch<EPI_DENSE, 1, 4, 2, true, DR_EW_WIDE>(maps, g, s)));
    else DR_TRY((gm_launch<EPI_DENSE, 1, 4, 4>(maps, g, s)));
    ++*launched;
  }
  // 2. GRU cell [REF models.py:81-82]: z and r accumulate both products, the candidate keeps its halves apart
  {
    GemmArgs g{};
    g.M = d.n; g.N = D;
    const DrTerm t[2] = {{&d.x1, &d.w_gruk, H, 0}, {&d.v_det[cur], &d.w_grur, D, 0}};
    const int rows[3] = {0, D, 2 * D};
    const int gate[2][3] = {{0, 1, 2}, {0, 1, 3}};
    dr_build(d, maps, g, t, 2, 3, rows, gate, 4, d.x3 ? 8 : 4);   // one main group (every gate slot must be fed), one small
    g.step = d.step; g.bias = d.b_gru; g.out = d.v_det[nxt].p[0]; g.out_lo = d.v_det[nxt].p[1]; g.ldo = d.ldf;
    g.hold = d.v_det[cur].p[0]; g.hold_lo = d.v_det[cur].p[1]; g.ldh = d.ldf;
    g.tma_out = d.tma_out; maps.o[0] = d.v_det[nxt].m[0]; maps.o[1] = d.v_det[nxt].m[1];
    if (d.x3) DR_TRY((gm_launch<EPI_GRU, 3, 8, 2, true, DR_EW_WIDE>(maps, g, s)));
    else DR_TRY((gm_launch<EPI_GRU, 3, 8, 4>(maps, g, s)));
    ++*launched;
  }
  // 3. obs1 = elu(concat([deter, embed]) @ W + b) [REF models.py:66-67]: two K ranges over one weight matrix
  {
    GemmArgs g{};
    g.M = d.n; g.N = H;
    const DrTerm t[2] = {{&d.v_det[nxt], &d.w_obs1, D, 0}, {&d.lidar, &d.w_obs1, d.embed, D}};
    dr_build(d, maps, g, t, 2, 1, nullptr, nullptr, 1, 8);
    g.step = d.step; g.bias = d.b_obs1; g.out = d.hobs.p[0]; g.out_lo = d.hobs.p[1]; g.ldo = H; g.act = 1;
    g.tma_out = d.tma_out; maps.o[0] = d.hobs.m[0]; maps.o[1] = d.hobs.m[1];
    if (d.x3) DR_TRY((gm_launch<EPI_DENSE, 1, 8, 4, true, DR_EW_WIDE>(maps, g, s)));
    else DR_TRY((gm_launch<EPI_DENSE, 1, 8, 8>(maps, g, s)));
    ++*launched;
  }
  // 4. obs2 + posterior sample [REF models.py:68-72]
  {
    GemmArgs g{};
    g.M = d.n; g.N = 2 * GM_STOCH;
    const DrTerm t[1] = {{&d.hobs, &d.w_obs2, H, 0}};
    dr_build(d, maps, g, t, 1, 1, nullptr, nullptr, 1, 4);
    g.bias = d.b_obs2; g.feat = d.feat[nxt].p[0]; g.feat_lo = d.feat[nxt].p[1]; g.ldf = d.ldf;
    g.noise = noise; g.eps = eps_stoch; g.ld_eps = GM_STOCH;
    g.key0 = (uint32_t)seed; g.key1 = (uint32_t)(seed >> 32) ^ RD_STREAM_STOCH; g.step = d.step; g.gid0 = gid0;
    g.dbg = debug;
    if (d.x3) DR_TRY((gm_launch<EPI_STOCH, 1, 4, 4, true, DR_EW_WIDE>(maps, g, s)));
    else DR_TRY((gm_launch<EPI_STOCH, 1, 4, 4>(maps, g, s)));
    ++*launched;
  }
  // 5. actor trunk [REF models.py:321-322]: float32-grade mode runs up to GM_CHAIN_MAX layers per launch (k_dense_chain)
  const bool chain = d.x3 && d.chain;
  bool head_fused = false;   // hout computed by the last chain launch (k_dense_chain's fused head)
  for (int i0 = 0; chain && i0 < d.layers; i0 += GM_CHAIN_MAX) {
    ChainMaps cm;
    ChainArgs c{};
    c.M = d.n; c.N = U; c.ldo = U; c.n_layers = std::min(GM_CHAIN_MAX, d.layers - i0);
    c.row_blocks = (d.n + GM_BM - 1) / GM_BM;
    c.flags = d.chain_flags;
    const unsigned nt = (unsigned)((U + DR_ACT_BN - 1) / DR_ACT_BN) * DR_ACT_EW;   // counter increments per row block and layer
    for (int j = 0; j < c.n_layers; ++j) {
      const int i = i0 + j;
      const DreamerPolicy::Operand& a = i == 0 ? d.feat[nxt] : d.hid[(i - 1) & 1];
      GemmArgs g{};   // the K blocks and accumulator groups of the per-layer launch (bitwise the same sums)
      const DrTerm t[1] = {{&a, &d.w_act[i], i == 0 ? d.ldf : U, 0}};
      dr_build(d, maps, g, t, 1, 1, nullptr, nullptr, 1, 4);
      ChainLayer& L = c.L[j];
      L.n_groups = g.n_acc - 1;
      L.kb_total = 0;
      for (int p = 0; p < g.n_phases; ++p) { L.grp_blocks[g.ph[p].acc[0]] = g.ph[p].k_blocks; L.kb_total += g.ph[p].k_blocks; }
      L.bias = d.b_act[i]; L.out = d.hid[i & 1].p[0]; L.out_lo = d.hid[i & 1].p[1];
      if (j + 1 < c.n_layers) { d.chain_count[j] += nt; L.target = d.chain_count[j]; }
      cm.a[j][0] = a.m[0]; cm.a[j][1] = a.m[1];
      cm.w[j][0] = d.w_act[i].m[0]; cm.w[j][1] = d.w_act[i].m[1];
      if (j + 1 == c.n_layers) { cm.o_last[0] = d.hid[i & 1].m[0]; cm.o_last[1] = d.hid[i & 1].m[1]; }
    }
    if (d.head_fused && i0 + c.n_layers == d.layers) {
      c.head = 1; c.head_bias = d.b_act[d.layers]; c.head_out = d.head_raw;
      cm.wh[0] = d.w_act[d.layers].m[0]; cm.wh[1] = d.w_act[d.layers].m[1];
    }
    DR_TRY((gm_launch_chain<DR_ACT_STAGES, DR_ACT_EW, DR_ACT_BN>(cm, c, d.sm_count, d.chain_cluster, s, &head_fused)));
    ++*launched;
  }
  for (int i = 0; !chain && i < d.layers; ++i) {
    GemmArgs g{};
    g.M = d.n; g.N = U;
    const DrTerm t[1] = {{i == 0 ? &d.feat[nxt] : &d.hid[(i - 1) & 1], &d.w_act[i], i == 0 ? d.ldf : U, 0}};
    dr_build(d, maps, g, t, 1, 1, nullptr, nullptr, 1, 4);
    g.bias = d.b_act[i]; g.out = d.hid[i & 1].p[0]; g.out_lo = d.hid[i & 1].p[1]; g.ldo = U; g.act = 1;
    g.tma_out = d.tma_out; maps.o[0] = d.hid[i & 1].m[0]; maps.o[1] = d.hid[i & 1].m[1];
    if (d.x3) DR_TRY((gm_launch<EPI_DENSE, 1, 4, DR_ACT_STAGES, true, DR_ACT_EW, DR_ACT_BN>(maps, g, s)));
    else DR_TRY((gm_launch<EPI_DENSE, 1, 4, 4>(maps, g, s)));
    ++*launched;
  }
  // 6. hout + distribution head + SampleDist.mode() [REF models.py:323-346; tools.py:70-73]
  {
    GemmArgs g{};
    g.M = d.n; g.N = 4;
    const DrTerm t[1] = {{&d.hid[(d.layers - 1) & 1], &d.w_act[d.layers], U, 0}};
    dr_build(d, maps, g, t, 1, 1, nullptr, nullptr, 1, 4);
    g.bias = d.b_act[d.layers]; g.actions = actions; g.feat = d.feat[nxt].p[0]; g.feat_lo = d.feat[nxt].p[1]; g.ldf = d.ldf;
    g.noise = noise; g.eps = eps_actor; g.ld_eps = 2 * d.n_samples;
    g.key0 = (uint32_t)seed; g.key1 = (uint32_t)(seed >> 32) ^ RD_STREAM_ACTOR; g.step = d.step; g.gid0 = gid0;
    g.bn = d.bn; g.raw_init_std = d.raw_init_std; g.min_std = d.min_std; g.mean_scale = d.mean_scale; g.bn_eps = d.bn_eps;
    g.n_samples = d.n_samples;
    g.dbg = debug ? debug + (size_t)d.n * 2 * GM_STOCH : nullptr;
    g.out = d.head_raw;
    if (!head_fused) {
      if (d.x3) DR_TRY((gm_launch<EPI_ACTOR, 1, 4, 4, true>(maps, g, s)));
      else DR_TRY((gm_launch<EPI_ACTOR, 1, 4, 4>(maps, g, s)));
      ++*launched;
    }
    {
      cudaLaunchConfig_t cfg = {};
      cfg.gridDim = dim3((unsigned)((d.n + 7) / 8));
      cfg.blockDim = dim3(256);
      cfg.stream = s;
      cudaLaunchAttribute attrs[1];
      attrs[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;   // griddepcontrol.wait in k_actor_mode / k_actor_train
      attrs[0].val.programmaticStreamSerializationAllowed = 1;
      cfg.attrs = attrs;
      cfg.numAttrs = 1;
      if (train) {
        cfg.gridDim = dim3((unsigned)((d.n + 255) / 256));   // one thread per env
        g.ld_eps = 2;
        g.key1 = (uint32_t)(seed >> 32) ^ RD_STREAM_TRAIN;
        DR_TRY(cudaLaunchKernelEx(&cfg, k_actor_train, g, train->eps_expl, train->amount));
      } else {
        DR_TRY(cudaLaunchKernelEx(&cfg, k_actor_mode, g));
      }
    }
    ++*launched;
  }
  d.cur = nxt;
  d.step++;
  return RD_OK;
}

// latent rows <-> the reference's `state` tuple (stoch, deter, action); dir 0 = read, 1 = write
static inline int dreamer_state_io(DreamerPolicy& d, float* stoch, float* deter, float* action, int dir, cudaStream_t s) {
  DreamerPolicy::Operand& f = d.feat[d.cur];
  struct { float* ext; int col0, width; } parts[3] = {{stoch, 0, GM_STOCH}, {action, GM_STOCH, 2}, {deter, 32, d.deter}};
  for (auto& p : parts) {
    if (!p.ext) continue;
    const size_t total = (size_t)d.n * p.width;
    k_latent_copy<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(f.p[0], f.p[1], d.ldf, p.col0, p.width, p.ext, d.n, dir);
    DR_TRY(cudaGetLastError());
  }
  return RD_OK;
}
