// rd_dreamer.cuh -- host-side orchestration of the on-device Dreamer agent (SURVEY.md §8-f2).
//
// One agent step = RacingDreamer.action [REF ros_agent/models/dreamer/racing_dreamer.py:62-82] for every env:
//   img1 -> GRU cell -> obs1 (concat([deter, embed])) -> obs2 + posterior sample -> actor h0..h3 -> hout + mode()
// = k_embed_lidar, five launches of k_dense (the fifth is hout), one of k_dense_chain per four layers of the actor trunk
// and k_actor_mode (rd_gemm.cuh); activations live in a handful of [envs][width] float32 arrays that stay in L2 between
// launches, the recurrent state in two ping-pong "latent" arrays whose rows are
//   [ stoch (30) | previous action (2) | deter (200) ]          (232 floats, 928 bytes)
// so that img1's input concat([stoch, action]), the GRU's state, obs1's concat([deter, ...]) and the actor's
// concat([stoch, deter]) are all plain TMA views of one row (the actor's weight rows for the two action slots are
// zero).  The prior head (img2/img3) only feeds a sample that obs_step's caller discards and is not evaluated.
// Several agents (rd_policy_dreamer_init_agents) share these launches: the rows are ordered by agent (GmAgents in
// rd_gemm.cuh), agent a's envs in ascending id order from row start[a] = the previous agent's end rounded up to GM_BM,
// and every weight array holds the agents' values one after the other.  One agent on every env is the case start = {0},
// rows = envs.  Only the embed (k_embed_lidar, k_conv1), the posterior's draws and debug rows (EPI_STOCH), the head
// (k_actor_mode / k_actor_train), the latent copies and the reset zeroing map between rows and envs.
#pragma once
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <string>
#include <vector>

#include "rd_gemm.cuh"

// Actor trunk (400-wide Dense layers) in float32-grade mode: output columns per CTA, ring stages, epilogue groups.
// 128-wide tiles make 4 N tiles instead of 7: 128 CTAs, one per SM (two 64-wide CTAs on half the SMs share the SM's L2
// ingress), which also leaves room for three 64 KB stages and four epilogue groups.  Measured: 64/2/2 0.190 ms,
// 128/2/2 0.191, 128/2/4 0.188, 128/3/4 0.181 ms per agent step.
#define DR_ACT_BN 128
#define DR_ACT_STAGES 3
#define DR_ACT_EW 4

// epilogue warp groups of the launches that have an SM to themselves (GRU cell, obs1, obs2 + posterior)
#define DR_EW_WIDE 4

struct DreamerPolicy {
  bool ready = false;
  int n_agents = 1;
  int rows = 0;                // internal rows: envs, plus the padding that starts every agent on a GM_BM boundary
  int n_of[GM_MAX_AGENTS] = {};   // envs per agent
  GmAgents ag{};
  int* env_of_row = nullptr;   // [rows] env of each row, -1 = padding; both maps null when rows = envs in order
  int* row_of_env = nullptr;   // [n]
  unsigned bn_mask = 0;        // bit a: agent a's actor head has BN ('normalized')
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
  // ConvEncoder agent (depth > 0; 0 = lidar agent): conv1's raw kernel [16][depth] and the biases, conv2..conv4's packed
  // kernels (k_pack_conv), the activations ping-ponging through enc_a (conv1, conv3) and enc_b (conv2) -- conv4 writes
  // `lidar`, the embed obs1 reads -- and per layer l = conv2..conv4 the 5-D input view and the 2-D output view
  int depth = 0;
  float* w_conv1 = nullptr;
  float* b_conv[4] = {};
  Operand w_conv[3], enc_a, enc_b, conv_in[3], conv_out[3];
  float* head_raw = nullptr;   // [n][4] hout pre-activations
  // k_dense_chain (the actor trunk in one launch): per-row-block layer counters and the values they have reached
  bool chain = true;           // RD_DREAMER_CHAIN=0: one k_dense launch per actor layer instead
  unsigned* chain_flags = nullptr;
  unsigned chain_count[GM_CHAIN_MAX] = {};
  int sm_count = 148;
  int cur = 0;           // feat[cur] holds the latest latent
  uint32_t step = 0;     // agent steps taken (Philox counter)
  // training-mode exploration per agent [REF dreamer/dreamer.py, Dreamer._exploration]: amount * 0.5^(env_steps / decay)
  // (decay > 0), at least min_amount (min_amount > 0); env_steps = Dreamer's step counter, + (the agent's envs) x
  // action_repeat per training step
  rd_dreamer_exploration expl[GM_MAX_AGENTS];
  DreamerPolicy() { for (auto& x : expl) x = rd_dreamer_exploration{0.3, 0.0, 0.0, 0}; }
  float* stage = nullptr;      // device copy of host-pointer weights for dr_pack (sized at init)
  std::string err;
};

static inline void dreamer_free(DreamerPolicy& d) {
  for (float* p : d.owned) cudaFree(p);
  d.owned.clear();
  d.bn = nullptr;
  d.stage = nullptr;
  d.env_of_row = d.row_of_env = nullptr;
  d.ready = false;
}

// The policy's weight layout: each checkpoint array, where it goes and how.  Matrices ([in][out] Keras kernels) become
// K-major TF32 operands [out][ld] (k_pack_weights: the K slots from k_from on shifted by k_shift, the slots skipped stay
// as init's zero fill left them); vectors (op == null) are copied as they are to *vec.  Sizes are w's, which the callers
// have checked (init) or held to the policy's (set_weights).  Init allocates what this list names for every agent
// (n_agents x out rows / values), dr_pack fills one agent's slice.
struct DrPart { const float* src; DreamerPolicy::Operand* op; float** vec; int in, out, ld, k_from, k_shift; };
static inline int dr_parts(DreamerPolicy& d, const rd_dreamer_weights* w, const rd_dreamer_conv_encoder* enc, DrPart* p) {
  const int H = w->hidden, D = w->deter, E = w->embed, U = w->actor_units, L = w->actor_layers, NO = 1 << 30;
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
  mat(w->actor_w[0], d.w_act[0], GM_STOCH + D, U, 32 + D, GM_STOCH, 2);
  vec(w->actor_b[0], d.b_act[0], U);
  for (int i = 1; i < L; ++i) {
    mat(w->actor_w[i], d.w_act[i], U, U, U, NO, 0);
    vec(w->actor_b[i], d.b_act[i], U);
  }
  mat(w->actor_w[L], d.w_act[L], U, 4, U, NO, 0);
  vec(w->actor_b[L], d.b_act[L], 4);
  if (w->bn) vec(w->bn, d.bn, 16);
  if (enc) {   // conv1 runs on CUDA cores from its Keras kernel as it is; conv2..conv4's kernels: dr_pack_conv
    vec(enc->w[0], d.w_conv1, 16 * enc->depth);
    for (int l = 0; l < 4; ++l) vec(enc->b[l], d.b_conv[l], enc->depth << l);
  }
  return k;
}
#define DR_MAX_PARTS (9 + 2 * 8 + 1 + 5)
static_assert(DR_MAX_PARTS <= GM_PACK_MAX, "dr_pack packs the whole table in one k_pack_weights launch");
static_assert(GM_MAX_AGENTS == RD_MAX_DREAMER_AGENTS, "one agent limit");

// Cin of conv layer l = 1..3 (conv2..conv4) of a depth-d encoder; Cout = 2 Cin
static inline int dr_conv_cin(int depth, int l) { return depth << (l - 1); }
// packs conv2..conv4's kernels (device pointers src[l - 1]) into agent `agent`'s slice of the policy's operands on `s`
static inline cudaError_t dr_pack_conv(DreamerPolicy& d, const float* const* src, int agent, cudaStream_t s) {
  for (int l = 1; l < 4; ++l) {
    const int cin = dr_conv_cin(d.depth, l), total = 16 * cin * 2 * cin;
    const DreamerPolicy::Operand& op = d.w_conv[l - 1];
    k_pack_conv<<<(unsigned)std::min((total + 255) / 256, d.sm_count * 8), 256, 0, s>>>(
        src[l - 1], op.p[0] + (size_t)agent * total, op.p[1] ? op.p[1] + (size_t)agent * total : nullptr, cin, 2 * cin);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
  }
  return cudaSuccess;
}

// zero-initialised operand array(s) [rows][ld].  In single-pass mode p[1] is null -- the packer and the epilogues test it
// -- also where the operand held a freed remainder array of an earlier tf32x3 agent (dr_view likewise).
// P: DreamerPolicy or MlpPolicy (rd_mlp.cuh), which read their x3 / owned / ag members the same way (dr_view, dr_build too).
template <class P>
static inline cudaError_t dr_alloc(P& d, DreamerPolicy::Operand& op, size_t rows, size_t ld) {
  op.p[1] = nullptr;
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
template <class P>
static inline bool dr_view(const P& d, DreamerPolicy::Operand& view, const DreamerPolicy::Operand& base, size_t col0,
                           uint64_t inner, uint64_t rows, uint64_t ld, uint32_t box_rows) {
  for (int part = 0; part < (d.x3 ? 2 : 1); ++part) {
    view.p[part] = base.p[part] + col0;
    if (!gm_make_map(&view.m[part], view.p[part], inner, rows, ld, box_rows)) return false;
  }
  if (!d.x3) view.p[1] = nullptr;
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

// Every source array of w and enc (dr_parts' and conv2..conv4's kernels) is non-null and, with on_device, memory of the
// current device, else not device memory.  Reads w's architecture: run it after that is checked.
static inline int dr_check_sources(DreamerPolicy& d, const rd_dreamer_weights* w, const rd_dreamer_conv_encoder* enc,
                                   bool on_device) {
  DrPart parts[DR_MAX_PARTS];
  const int n_parts = dr_parts(d, w, enc, parts);
  const float* srcs[DR_MAX_PARTS + 3];
  int n_src = 0;
  for (int k = 0; k < n_parts; ++k) srcs[n_src++] = parts[k].src;
  for (int l = 1; enc && l < 4; ++l) srcs[n_src++] = enc->w[l];
  int dev = 0;
  DR_TRY(cudaGetDevice(&dev));
  for (int k = 0; k < n_src; ++k) {
    if (!srcs[k]) { d.err = "null weight pointer"; return RD_ERR_INVALID; }
    cudaPointerAttributes at{};
    DR_TRY(cudaPointerGetAttributes(&at, srcs[k]));
    const bool device_ptr = at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged;
    if (on_device && (!device_ptr || at.device != dev)) { d.err = "on_device: a weight pointer is not memory of the policy's device"; return RD_ERR_INVALID; }
    if (!on_device && at.type == cudaMemoryTypeDevice) { d.err = "a weight pointer is device memory where host memory is expected (init, or on_device = 0)"; return RD_ERR_INVALID; }
  }
  return RD_OK;
}

// Packs w and enc (checked by dr_check_sources) into agent `agent`'s slice of the buffers init allocated, on `s`: host
// sources (!on_device) are first copied to d.stage, then one k_pack_weights launch packs the dr_parts table and
// dr_pack_conv conv2..conv4.
static inline int dr_pack(DreamerPolicy& d, const rd_dreamer_weights* w, const rd_dreamer_conv_encoder* enc, int agent,
                          bool on_device, cudaStream_t s) {
  DrPart parts[DR_MAX_PARTS];
  const int n_parts = dr_parts(d, w, enc, parts);
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
    const size_t slice = (size_t)agent * p.out * (p.op ? p.ld : 1);
    J.src = src;
    J.hi = (p.op ? p.op->p[0] : *p.vec) + slice;
    J.lo = (p.op && p.op->p[1]) ? p.op->p[1] + slice : nullptr;
    J.in = p.in; J.out = p.out; J.ld = p.ld; J.k_from = p.k_from; J.k_shift = p.k_shift; J.raw = p.op ? 0 : 1;
    J.begin = (long long)off;
    off += count;
  }
  a.total = (long long)off;
  const unsigned grid = (unsigned)std::min<size_t>((off + 255) / 256, (size_t)d.sm_count * 8);
  k_pack_weights<false><<<grid, 256, 0, s>>>(a);
  DR_TRY(cudaGetLastError());
  if (enc) {
    const float* src[3];
    for (int l = 1; l < 4; ++l) {
      const size_t count = (size_t)32 * dr_conv_cin(d.depth, l) * dr_conv_cin(d.depth, l);
      src[l - 1] = enc->w[l];
      if (!on_device) {
        DR_TRY(cudaMemcpyAsync(d.stage + off, enc->w[l], count * sizeof(float), cudaMemcpyHostToDevice, s));
        src[l - 1] = d.stage + off;
      }
      off += count;
    }
    DR_TRY(dr_pack_conv(d, src, agent, s));
  }
  return RD_OK;
}

// Every check of one agent's weights (w, enc) that init makes before it touches the policy.
static inline int dr_check_arch(DreamerPolicy& d, int n_beams, const rd_dreamer_weights* w, const rd_dreamer_conv_encoder* enc) {
  if (!w) { d.err = "null weights"; return RD_ERR_INVALID; }
  if (enc) {
    if (enc->depth != 32) { d.err = "unsupported ConvEncoder depth " + std::to_string(enc->depth) + " (need 32)"; return RD_ERR_INVALID; }
    if (w->embed != 32 * enc->depth) { d.err = "a ConvEncoder agent's embed must be 32 * depth"; return RD_ERR_INVALID; }
  }
  if (w->stoch != GM_STOCH || w->deter <= 0 || w->deter % 4 || w->hidden <= 0 || w->hidden % 4 ||
      (!enc && w->embed != n_beams) || w->embed % 4 || w->actor_units <= 0 || w->actor_units % 4 || w->actor_layers < 1 || w->actor_layers > 7 ||
      w->n_samples < 1 || !(w->mean_scale > 0.f)) {
    d.err = "unsupported Dreamer architecture (need stoch 30, deter/hidden/units/embed multiples of 4, embed == n_beams (lidar agent), 1..7 actor layers)";
    return RD_ERR_INVALID;
  }
  if (w->precision != RD_PRECISION_TF32X3 && w->precision != RD_PRECISION_TF32) { d.err = "bad precision"; return RD_ERR_INVALID; }
  return RD_OK;
}

// Agents of one policy share every size and scalar of the weights (their values differ); BN presence may differ.
static inline bool dr_same_arch(const rd_dreamer_weights* a, const rd_dreamer_weights* b) {
  return a->stoch == b->stoch && a->deter == b->deter && a->hidden == b->hidden && a->embed == b->embed &&
         a->actor_units == b->actor_units && a->actor_layers == b->actor_layers && a->precision == b->precision &&
         a->n_samples == b->n_samples && a->init_std == b->init_std && a->min_std == b->min_std &&
         a->mean_scale == b->mean_scale && a->bn_eps == b->bn_eps;
}

// lidar_normalised: the env already emits r/15 - 0.5 (RD_OBS_LIDAR_NORM), so k_embed_lidar only splits the values
// G agents: w[G] and, for ConvEncoder agents (embed = 32 depth) instead of lidar ones (embed = n_beams), enc[G];
// agent_of_env [n] host values in [0, G) (null: every env is agent 0's), every agent owning at least one env.
static inline int dreamer_init(DreamerPolicy& d, int n, int n_beams, bool lidar_normalised, int G, const rd_dreamer_weights* w,
                               const rd_dreamer_conv_encoder* enc = nullptr, const int32_t* agent_of_env = nullptr) {
  if (G < 1 || G > GM_MAX_AGENTS) { d.err = "n_agents must be 1.." + std::to_string(GM_MAX_AGENTS); return RD_ERR_INVALID; }
  if (!w) { d.err = "null weights"; return RD_ERR_INVALID; }
  int with_bn = -1;   // an agent with a BN head, if any: its table names every array init allocates
  for (int a = 0; a < G; ++a) {
    if (int rc = dr_check_arch(d, n_beams, w + a, enc ? enc + a : nullptr)) {
      if (G > 1) d.err = "agent " + std::to_string(a) + ": " + d.err;
      return rc;
    }
    if (!dr_same_arch(w, w + a) || (enc && enc[a].depth != enc[0].depth)) {
      d.err = "agent " + std::to_string(a) + ": every agent needs the architecture, precision, sample count and head scalars of agent 0";
      return RD_ERR_INVALID;
    }
    if (w[a].bn && with_bn < 0) with_bn = a;
  }
  std::vector<int> n_of(G, 0);
  for (int e = 0; agent_of_env && e < n; ++e) {
    if (agent_of_env[e] < 0 || agent_of_env[e] >= G) { d.err = "agent_of_env[" + std::to_string(e) + "] is not in [0, n_agents)"; return RD_ERR_INVALID; }
    ++n_of[agent_of_env[e]];
  }
  if (!agent_of_env) n_of[0] = n;
  for (int a = 0; a < G; ++a)
    if (n_of[a] == 0) { d.err = "agent " + std::to_string(a) + " drives no env"; return RD_ERR_INVALID; }
  if (!gm_get_encoder()) { d.err = "cuTensorMapEncodeTiled is not available from this driver"; return RD_ERR_CUDA; }
  for (int a = 0; a < G; ++a)   // all checks before dreamer_free: a rejected init changes nothing
    if (int rc = dr_check_sources(d, w + a, enc ? enc + a : nullptr, false)) return rc;
  dreamer_free(d);
  // the row layout: agent a's envs in ascending order from start[a], starts rounded up to GM_BM
  d.n_agents = G;
  d.ag = GmAgents{};   // start 0 past the last agent: no such agent
  for (int a = 0; a < GM_MAX_AGENTS; ++a) d.n_of[a] = a < G ? n_of[a] : 0;
  int rows = 0;
  for (int a = 0; a < G; ++a) {
    d.ag.start[a] = rows = (rows + GM_BM - 1) / GM_BM * GM_BM;
    rows += n_of[a];
  }
  d.rows = rows;
  std::vector<int> env_of_row(rows, -1), row_of_env(n);
  {
    std::vector<int> next(d.ag.start, d.ag.start + G);
    for (int e = 0; e < n; ++e) {
      const int r = next[agent_of_env ? agent_of_env[e] : 0]++;
      env_of_row[r] = e;
      row_of_env[e] = r;
    }
  }
  bool identity = rows == n;
  for (int e = 0; identity && e < n; ++e) identity = row_of_env[e] == e;
  if (!identity) {
    int* maps[2] = {nullptr, nullptr};
    DR_TRY(cudaMalloc(&maps[0], (size_t)rows * sizeof(int)));
    d.owned.push_back(reinterpret_cast<float*>(maps[0]));
    DR_TRY(cudaMalloc(&maps[1], (size_t)n * sizeof(int)));
    d.owned.push_back(reinterpret_cast<float*>(maps[1]));
    DR_TRY(cudaMemcpy(maps[0], env_of_row.data(), (size_t)rows * sizeof(int), cudaMemcpyHostToDevice));
    DR_TRY(cudaMemcpy(maps[1], row_of_env.data(), (size_t)n * sizeof(int), cudaMemcpyHostToDevice));
    d.env_of_row = maps[0];
    d.row_of_env = maps[1];
  }
  d.bn_mask = 0;
  for (int a = 0; a < G; ++a) d.bn_mask |= w[a].bn ? 1u << a : 0u;
  d.x3 = w->precision == RD_PRECISION_TF32X3;
  d.lidar_normalised = lidar_normalised;
  d.n = n; d.deter = w->deter; d.hidden = w->hidden; d.embed = w->embed; d.units = w->actor_units; d.layers = w->actor_layers;
  d.depth = enc ? enc->depth : 0;
  d.ldf = 32 + d.deter;
  d.raw_init_std = (float)std::log(std::exp((double)w->init_std) - 1.0);   // [REF models.py:321]
  d.min_std = w->min_std; d.mean_scale = w->mean_scale; d.bn_eps = w->bn_eps; d.n_samples = w->n_samples;
  const int H = d.hidden, D = d.deter, E = d.embed, U = d.units;
  int dev = 0;
  DR_TRY(cudaGetDevice(&dev));
  DR_TRY(cudaDeviceGetAttribute(&d.sm_count, cudaDevAttrMultiProcessorCount, dev));
  // the weights' buffers, G slices each (matrices zero-filled: the K slots k_pack_weights skips stay zero; BN zero-filled
  // for the agents without one), and the stage that holds a copy of one agent's host sources, the table's arrays and
  // then conv2..conv4's kernels
  DrPart parts[DR_MAX_PARTS];
  const int n_parts = dr_parts(d, w + std::max(with_bn, 0), enc, parts);
  size_t stage_floats = 0;
  for (int k = 0; k < n_parts; ++k) {
    const DrPart& p = parts[k];
    if (p.op) {
      DR_TRY(dr_alloc(d, *p.op, (size_t)G * p.out, (size_t)p.ld));
    } else {
      DR_TRY(cudaMalloc(p.vec, (size_t)G * p.out * sizeof(float)));
      d.owned.push_back(*p.vec);
      DR_TRY(cudaMemset(*p.vec, 0, (size_t)G * p.out * sizeof(float)));
    }
    stage_floats += (size_t)p.in * p.out;
  }
  for (int l = 1; d.depth && l < 4; ++l) {
    const int cin = dr_conv_cin(d.depth, l);
    DR_TRY(dr_alloc(d, d.w_conv[l - 1], (size_t)G * 2 * cin, (size_t)16 * cin));
    stage_floats += (size_t)32 * cin * cin;
  }
  DR_TRY(cudaMalloc(&d.stage, stage_floats * sizeof(float)));
  d.owned.push_back(d.stage);
  for (int a = 0; a < G; ++a)
    if (int rc = dr_pack(d, w + a, enc ? enc + a : nullptr, a, false, 0)) return rc;
  DR_TRY(cudaDeviceSynchronize());
  const size_t N = (size_t)rows;
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
    d.chain = true;
    if (const char* ev = std::getenv("RD_DREAMER_CHAIN")) d.chain = std::atoi(ev) != 0;
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
  if (d.depth) {   // encoder activations: conv1 / conv3 outputs in enc_a, conv2's in enc_b (see dreamer_encode)
    const int c = d.depth;
    DR_TRY(dr_alloc(d, d.enc_a, N * 32 * 32, c));
    DR_TRY(dr_alloc(d, d.enc_b, N * 16 * 16, 2 * c));
    const DreamerPolicy::Operand* in[3] = {&d.enc_a, &d.enc_b, &d.enc_a};
    const DreamerPolicy::Operand* out[3] = {&d.enc_b, &d.enc_a, &d.lidar};
    const int g_in[3] = {32, 16, 8}, g_out[3] = {16, 8, 2};
    for (int l = 0; l < 3; ++l) {
      const int cin = dr_conv_cin(c, l + 1);
      for (int part = 0; part < (d.x3 ? 2 : 1); ++part) {
        d.conv_in[l].p[part] = in[l]->p[part];
        DR_MAP(gm_make_map_conv(&d.conv_in[l].m[part], in[l]->p[part], cin, g_in[l], N, g_out[l]));
      }
      DR_MAP(dr_view(d, d.conv_out[l], *out[l], 0, 2 * cin, N * g_out[l] * g_out[l], 2 * cin, GM_BM));
      DR_MAP(dr_view(d, d.w_conv[l], d.w_conv[l], 0, 16 * cin, G * 2 * cin, 16 * cin, GM_BN));
    }
  }
  // the weight views span every agent's rows (the producer adds agent x out to the row coordinate); the masked columns of
  // an agent's last N tile read the next agent's rows, which no stored column uses
  DR_MAP(dr_view(d, d.w_img1, d.w_img1, 0, 32, G * H, 32, GM_BN));
  DR_MAP(dr_view(d, d.w_gruk, d.w_gruk, 0, H, G * 3 * D, H, GM_BN));
  DR_MAP(dr_view(d, d.w_grur, d.w_grur, 0, D, G * 3 * D, D, GM_BN));
  DR_MAP(dr_view(d, d.w_obs1, d.w_obs1, 0, D + E, G * H, D + E, GM_BN));
  DR_MAP(dr_view(d, d.w_obs2, d.w_obs2, 0, H, G * 2 * GM_STOCH, H, GM_BN));
  DR_MAP(dr_view(d, d.w_act[0], d.w_act[0], 0, d.ldf, G * U, d.ldf, d.x3 ? DR_ACT_BN : GM_BN));
  for (int i = 1; i < d.layers; ++i) DR_MAP(dr_view(d, d.w_act[i], d.w_act[i], 0, U, G * U, U, d.x3 ? DR_ACT_BN : GM_BN));
  DR_MAP(dr_view(d, d.w_act[d.layers], d.w_act[d.layers], 0, U, G * 4, U, GM_BN));
  d.cur = 0;
  d.step = 0;
  for (auto& x : d.expl) x.env_steps = 0;
  d.ready = true;
  return RD_OK;
}

// the exploration amount of agent `agent`'s next training step, rounded once to float32
static inline float dreamer_expl_amount(const DreamerPolicy& d, int agent) {
  const rd_dreamer_exploration& x = d.expl[agent];
  double a = x.amount;
  if (x.decay > 0.0) a *= std::pow(0.5, (double)x.env_steps / x.decay);
  if (x.min_amount > 0.0) a = std::max(x.min_amount, a);
  return (float)a;
}

// New values for every weight of agent `agent` of an initialised policy, packed on `s` by init's packer (dr_pack) into
// that agent's slice of the buffers the policy already owns (no allocation; the tensor maps stay valid).  Latent state,
// Philox step, env_steps and the other agents' weights are kept.  w holds device pointers (on_device) or host pointers,
// which are first copied to d.stage.  The architecture, the agent's BN presence, precision and head scalars must be the
// init's; otherwise RD_ERR_INVALID and nothing changes.
static inline int dreamer_set_weights(DreamerPolicy& d, int agent, const rd_dreamer_weights* w, const rd_dreamer_conv_encoder* enc,
                                      bool on_device, cudaStream_t s) {
  if (!w) { d.err = "null weights"; return RD_ERR_INVALID; }
  if (agent < 0 || agent >= d.n_agents) { d.err = "agent " + std::to_string(agent) + " is not in [0, n_agents)"; return RD_ERR_INVALID; }
  if ((enc != nullptr) != (d.depth > 0) || (enc && enc->depth != d.depth)) {
    d.err = "the encoder (present, depth) differs from the one the policy was initialised with";
    return RD_ERR_INVALID;
  }
  const float raw_init_std = (float)std::log(std::exp((double)w->init_std) - 1.0);
  if (w->stoch != GM_STOCH || w->deter != d.deter || w->hidden != d.hidden || w->embed != d.embed ||
      w->actor_units != d.units || w->actor_layers != d.layers || (w->bn != nullptr) != (((d.bn_mask >> agent) & 1u) != 0) ||
      (w->precision != RD_PRECISION_TF32X3 && w->precision != RD_PRECISION_TF32) ||
      (w->precision == RD_PRECISION_TF32X3) != d.x3 || w->n_samples != d.n_samples || raw_init_std != d.raw_init_std ||
      w->min_std != d.min_std || w->mean_scale != d.mean_scale || w->bn_eps != d.bn_eps) {
    d.err = "the weights' architecture, precision or head scalars differ from the ones the policy was initialised with";
    return RD_ERR_INVALID;
  }
  if (int rc = dr_check_sources(d, w, enc, on_device)) return rc;
  return dr_pack(d, w, enc, agent, on_device, s);
}

// One layer's launch description: up to two (A source, W, K range) terms.  dr_build expands them into phases:
// in x3 mode first the lo*hi and hi*lo passes of every term (into the "small" accumulator group), then the hi*hi pass
// cut into K groups of at most ~6 blocks, one accumulator group each (see "truncation" in rd_gemm.cuh).
// Accumulator slot = group * gates + gate; `gate[t][i]` maps slab i of term t to its gate (Dense layers: one gate).
struct DrTerm { const DreamerPolicy::Operand* a; const DreamerPolicy::Operand* w; int k_elems; int w_k0; };
template <class P>
static inline void dr_build(const P& d, GemmMaps& maps, GemmArgs& g, const DrTerm* terms, int n_terms, int nb,
                            const int* w_row0, const int (*gate)[3], int gates, int slots) {
  g.n_phases = 0;
  g.ag = d.ag;
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
struct DrTrain { const float* eps_expl; GmAmounts amount; };   // amount.a[agent]
// ConvEncoder [UPSTREAM-RECALL: danijar Dreamer models.py ConvEncoder] of u8 images [n][64][64] -> d.lidar, the embed
// operand obs1 reads ([n][32 depth], (y, x, c) order, TF32 hi + lo).  conv1 on CUDA cores (k_conv1) into enc_a's 32 x 32
// grid; conv2 (16 x 16 grid, 14 x 14 valid) -> enc_b, conv3 (8 x 8 grid, 6 x 6 valid) -> enc_a, conv4 (2 x 2, all valid)
// -> d.lidar as k_dense implicit GEMMs (gm_conv_a).  The padded grids' extra outputs are finite (they read zeros or other
// finite outputs) and no valid output reads them.
template <int G>
static inline cudaError_t dr_conv_launch(const DreamerPolicy& d, const GemmMaps& maps, const GemmArgs& g, cudaStream_t s) {
  if (d.x3) return gm_launch<EPI_DENSE, 1, 8, 4, true, DR_EW_WIDE, GM_BN, G>(maps, g, s);
  return gm_launch<EPI_DENSE, 1, 8, 8, false, GM_EPI_GROUPS, GM_BN, G>(maps, g, s);
}
static inline int dreamer_encode(DreamerPolicy& d, const uint8_t* occ, cudaStream_t s, int* launched) {
  k_conv1<<<(unsigned)d.rows * 32, 256, 0, s>>>(occ, d.w_conv1, d.b_conv[0], reinterpret_cast<float4*>(d.enc_a.p[0]),
                                                reinterpret_cast<float4*>(d.enc_a.p[1]), d.env_of_row, d.ag);
  DR_TRY(cudaGetLastError());
  ++*launched;
  GemmMaps maps;
  const int g_out[3] = {16, 8, 2};
  for (int l = 0; l < 3; ++l) {
    const int cin = dr_conv_cin(d.depth, l + 1);
    GemmArgs g{};
    g.M = d.rows * g_out[l] * g_out[l]; g.N = 2 * cin;
    const DrTerm t[1] = {{&d.conv_in[l], &d.w_conv[l], 16 * cin, 0}};
    dr_build(d, maps, g, t, 1, 1, nullptr, nullptr, 1, 8);
    g.step = d.step; g.bias = d.b_conv[l + 1]; g.out = d.conv_out[l].p[0]; g.out_lo = d.conv_out[l].p[1]; g.ldo = 2 * cin;
    maps.o[0] = d.conv_out[l].m[0]; maps.o[1] = d.conv_out[l].m[1];
    if (l == 0) DR_TRY(dr_conv_launch<16>(d, maps, g, s));
    else if (l == 1) DR_TRY(dr_conv_launch<8>(d, maps, g, s));
    else DR_TRY(dr_conv_launch<2>(d, maps, g, s));
    ++*launched;
  }
  return RD_OK;
}

// obs: the lidar scans (f32 [n][n_beams]) or, for a ConvEncoder agent, the occupancy images (u8 [n][64][64])
static inline int dreamer_step(DreamerPolicy& d, const void* obs, float* actions, int noise, const float* eps_stoch,
                               const float* eps_actor, float* debug, uint64_t seed, uint32_t gid0, cudaStream_t s, int* launched,
                               const DrTrain* train = nullptr) {
  *launched = 0;
  const int cur = d.cur, nxt = cur ^ 1;
  const int H = d.hidden, D = d.deter, U = d.units;
  if (d.depth) {   // 0. embed = ConvEncoder(image)
    const int rc = dreamer_encode(d, static_cast<const uint8_t*>(obs), s, launched);
    if (rc) return rc;
  } else {   // 0. embed = _preprocess_lidar(scan), split for the tensor-core passes
    const float* lidar = static_cast<const float*>(obs);
    const size_t count4 = (size_t)d.rows * d.embed / 4;
    const unsigned grid = (unsigned)std::min<size_t>((count4 + 255) / 256, 148 * 8);
    k_embed_lidar<<<grid, 256, 0, s>>>(reinterpret_cast<const float4*>(lidar), reinterpret_cast<float4*>(d.lidar.p[0]),
                                       reinterpret_cast<float4*>(d.lidar.p[1]), count4, d.lidar_normalised ? 0 : 1,
                                       d.env_of_row, d.embed / 4);
    DR_TRY(cudaGetLastError());
    ++*launched;
  }
  GemmMaps maps;
  // 1. img1: x1 = elu(concat([stoch, action]) @ W + b) [REF models.py:78-80]
  {
    GemmArgs g{};
    g.M = d.rows; g.N = H;
    const DrTerm t[1] = {{&d.v_sa[cur], &d.w_img1, 32, 0}};
    dr_build(d, maps, g, t, 1, 1, nullptr, nullptr, 1, 4);
    g.step = d.step; g.bias = d.b_img1; g.out = d.x1.p[0]; g.out_lo = d.x1.p[1]; g.ldo = H; g.act = 1;
    maps.o[0] = d.x1.m[0]; maps.o[1] = d.x1.m[1];
    if (d.x3) DR_TRY((gm_launch<EPI_DENSE, 1, 4, 2, true, DR_EW_WIDE>(maps, g, s)));
    else DR_TRY((gm_launch<EPI_DENSE, 1, 4, 4>(maps, g, s)));
    ++*launched;
  }
  // 2. GRU cell [REF models.py:81-82]: z and r accumulate both products, the candidate keeps its halves apart
  {
    GemmArgs g{};
    g.M = d.rows; g.N = D;
    const DrTerm t[2] = {{&d.x1, &d.w_gruk, H, 0}, {&d.v_det[cur], &d.w_grur, D, 0}};
    const int rows[3] = {0, D, 2 * D};
    const int gate[2][3] = {{0, 1, 2}, {0, 1, 3}};
    dr_build(d, maps, g, t, 2, 3, rows, gate, 4, d.x3 ? 8 : 4);   // one main group (every gate slot must be fed), one small
    g.step = d.step; g.bias = d.b_gru; g.out = d.v_det[nxt].p[0]; g.out_lo = d.v_det[nxt].p[1]; g.ldo = d.ldf;
    g.hold = d.v_det[cur].p[0]; g.hold_lo = d.v_det[cur].p[1]; g.ldh = d.ldf;
    maps.o[0] = d.v_det[nxt].m[0]; maps.o[1] = d.v_det[nxt].m[1];
    if (d.x3) DR_TRY((gm_launch<EPI_GRU, 3, 8, 2, true, DR_EW_WIDE>(maps, g, s)));
    else DR_TRY((gm_launch<EPI_GRU, 3, 8, 4>(maps, g, s)));
    ++*launched;
  }
  // 3. obs1 = elu(concat([deter, embed]) @ W + b) [REF models.py:66-67]: two K ranges over one weight matrix
  {
    GemmArgs g{};
    g.M = d.rows; g.N = H;
    const DrTerm t[2] = {{&d.v_det[nxt], &d.w_obs1, D, 0}, {&d.lidar, &d.w_obs1, d.embed, D}};
    dr_build(d, maps, g, t, 2, 1, nullptr, nullptr, 1, 8);
    g.step = d.step; g.bias = d.b_obs1; g.out = d.hobs.p[0]; g.out_lo = d.hobs.p[1]; g.ldo = H; g.act = 1;
    maps.o[0] = d.hobs.m[0]; maps.o[1] = d.hobs.m[1];
    if (d.x3) DR_TRY((gm_launch<EPI_DENSE, 1, 8, 4, true, DR_EW_WIDE>(maps, g, s)));
    else DR_TRY((gm_launch<EPI_DENSE, 1, 8, 8>(maps, g, s)));
    ++*launched;
  }
  // 4. obs2 + posterior sample [REF models.py:68-72]
  {
    GemmArgs g{};
    g.M = d.rows; g.N = 2 * GM_STOCH;
    const DrTerm t[1] = {{&d.hobs, &d.w_obs2, H, 0}};
    dr_build(d, maps, g, t, 1, 1, nullptr, nullptr, 1, 4);
    g.bias = d.b_obs2; g.feat = d.feat[nxt].p[0]; g.feat_lo = d.feat[nxt].p[1]; g.ldf = d.ldf;
    g.noise = noise; g.eps = eps_stoch; g.ld_eps = GM_STOCH;
    g.key0 = (uint32_t)seed; g.key1 = (uint32_t)(seed >> 32) ^ RD_STREAM_STOCH; g.step = d.step; g.gid0 = gid0;
    g.dbg = debug; g.env_of_row = d.env_of_row;
    if (d.x3) DR_TRY((gm_launch<EPI_STOCH, 1, 4, 4, true, DR_EW_WIDE>(maps, g, s)));
    else DR_TRY((gm_launch<EPI_STOCH, 1, 4, 4>(maps, g, s)));
    ++*launched;
  }
  // 5. actor trunk [REF models.py:321-322]: float32-grade mode runs up to GM_CHAIN_MAX layers per launch (k_dense_chain)
  const bool chain = d.x3 && d.chain;
  for (int i0 = 0; chain && i0 < d.layers; i0 += GM_CHAIN_MAX) {
    ChainMaps cm;
    ChainArgs c{};
    c.M = d.rows; c.N = U; c.ldo = U; c.n_layers = std::min(GM_CHAIN_MAX, d.layers - i0);
    c.row_blocks = (d.rows + GM_BM - 1) / GM_BM;
    c.ag = d.ag;
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
    DR_TRY((gm_launch_chain<DR_ACT_STAGES, DR_ACT_EW, DR_ACT_BN>(cm, c, d.sm_count, s)));
    ++*launched;
  }
  for (int i = 0; !chain && i < d.layers; ++i) {
    GemmArgs g{};
    g.M = d.rows; g.N = U;
    const DrTerm t[1] = {{i == 0 ? &d.feat[nxt] : &d.hid[(i - 1) & 1], &d.w_act[i], i == 0 ? d.ldf : U, 0}};
    dr_build(d, maps, g, t, 1, 1, nullptr, nullptr, 1, 4);
    g.bias = d.b_act[i]; g.out = d.hid[i & 1].p[0]; g.out_lo = d.hid[i & 1].p[1]; g.ldo = U; g.act = 1;
    maps.o[0] = d.hid[i & 1].m[0]; maps.o[1] = d.hid[i & 1].m[1];
    if (d.x3) DR_TRY((gm_launch<EPI_DENSE, 1, 4, DR_ACT_STAGES, true, DR_ACT_EW, DR_ACT_BN>(maps, g, s)));
    else DR_TRY((gm_launch<EPI_DENSE, 1, 4, 4>(maps, g, s)));
    ++*launched;
  }
  // 6. hout + distribution head + SampleDist.mode() [REF models.py:323-346; tools.py:70-73]
  {
    GemmArgs g{};
    g.M = d.rows; g.N = 4;
    const DrTerm t[1] = {{&d.hid[(d.layers - 1) & 1], &d.w_act[d.layers], U, 0}};
    dr_build(d, maps, g, t, 1, 1, nullptr, nullptr, 1, 4);
    g.bias = d.b_act[d.layers]; g.actions = actions; g.feat = d.feat[nxt].p[0]; g.feat_lo = d.feat[nxt].p[1]; g.ldf = d.ldf;
    g.noise = noise; g.eps = eps_actor; g.ld_eps = 2 * d.n_samples;
    g.key0 = (uint32_t)seed; g.key1 = (uint32_t)(seed >> 32) ^ RD_STREAM_ACTOR; g.step = d.step; g.gid0 = gid0;
    g.bn = d.bn; g.bn_mask = (int)d.bn_mask; g.env_of_row = d.env_of_row; g.raw_init_std = d.raw_init_std; g.min_std = d.min_std; g.mean_scale = d.mean_scale; g.bn_eps = d.bn_eps;
    g.n_samples = d.n_samples;
    g.dbg = debug ? debug + (size_t)d.n * 2 * GM_STOCH : nullptr;
    g.out = d.head_raw;
    if (d.x3) DR_TRY((gm_launch<EPI_ACTOR, 1, 4, 4, true>(maps, g, s)));
    else DR_TRY((gm_launch<EPI_ACTOR, 1, 4, 4>(maps, g, s)));
    ++*launched;
    {
      cudaLaunchConfig_t cfg = {};
      cfg.gridDim = dim3((unsigned)((d.rows + 7) / 8));
      cfg.blockDim = dim3(256);
      cfg.stream = s;
      cudaLaunchAttribute attrs[1];
      attrs[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;   // griddepcontrol.wait in k_actor_mode / k_actor_train
      attrs[0].val.programmaticStreamSerializationAllowed = 1;
      cfg.attrs = attrs;
      cfg.numAttrs = 1;
      if (train) {
        cfg.gridDim = dim3((unsigned)((d.rows + 255) / 256));   // one thread per row
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
    k_latent_copy<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(f.p[0], f.p[1], d.ldf, p.col0, p.width, p.ext, d.n, dir,
                                                                  d.row_of_env);
    DR_TRY(cudaGetLastError());
  }
  return RD_OK;
}
