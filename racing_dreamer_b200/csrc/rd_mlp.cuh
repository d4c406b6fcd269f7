// rd_mlp.cuh -- the feed-forward Gaussian actor of the model-free baselines on the tensor cores (SURVEY.md §8-f2), and
// uniform random actions.
//
// One actor step (rd_policy_mlp) for every env:
//   k_embed_lidar (split only: the env already normalised the scan to [0, 1]) -> one k_dense<EPI_DENSE_RELU | TANH> per
//   trunk layer -> k_dense<EPI_ACTOR> writing the head's four pre-activations [N][4] -> k_mlp_head (clamp, exp, sample,
//   squash) writing the actions where k_step reads them.
// Every product is tf32x3 (float32-grade).  The trunk's activations live in one [N][width] array (hi, lo) per layer,
// read by the next layer through the same TMA view the epilogue stores through.  Widths are padded to multiples of 4
// (the TMA row pitch): the padded weight rows, K slots and biases are zero, so a padded column is act(0) = 0 and feeds
// nothing.  K = n_beams (1080) is not a multiple of the 32-float K block: the views' extent zero-fills the tail.
// The head's rows are mean0, mean1, log_std0, log_std1 (RD_HEAD_SQUASHED) or mean0, mean1, 0, 0 (RD_HEAD_DIAG, whose
// log_std is a vector read by k_mlp_head).
#pragma once
#include <algorithm>
#include <string>
#include <vector>

#include "rd_dreamer.cuh"

struct MlpPolicy {
  bool ready = false;
  static constexpr bool x3 = true;   // dr_alloc / dr_view / dr_build: three-pass products
  GmAgents ag{};                     // one actor for every env (zero value: a single agent)
  std::vector<float*> owned;         // every device allocation of this policy
  rd_mlp_actor arch{};               // the init's architecture (pointers cleared)
  int n = 0, in_pad = 0, wpad[RD_MLP_MAX_LAYERS] = {};
  DreamerPolicy::Operand lidar, act[RD_MLP_MAX_LAYERS], w[RD_MLP_MAX_LAYERS], w_head;
  float* b[RD_MLP_MAX_LAYERS] = {};
  float* b_head = nullptr;           // [4]
  float* log_std = nullptr;          // [2] (RD_HEAD_DIAG)
  float* head_raw = nullptr;         // [n][4]
  float* stage = nullptr;            // device copy of host-pointer weights for mlp_pack
  int sm_count = 148;
  uint32_t step = 0;                 // actor steps taken (Philox counter)
  std::string err;
};

static inline void mlp_free(MlpPolicy& d) {
  for (float* p : d.owned) cudaFree(p);
  d.owned.clear();
  d.ready = false;
}

static inline int mlp_pad4(int x) { return (x + 3) & ~3; }

// The actor's weight layout: each source array and where it goes.  Matrices (src [out][in], K-major) become TF32 hi/lo
// rows of pitch ld from dst row 0 of hi / lo; vectors are copied as they are.
struct MlpPart { const float* src; float* hi; float* lo; int in, out, ld; };
static inline int mlp_parts(const MlpPolicy& d, const rd_mlp_actor* a, MlpPart* p) {
  int k = 0;
  const int L = a->n_layers;
  for (int l = 0; l < L; ++l) {
    const int in = l ? a->width[l - 1] : a->in_features, ld = l ? d.wpad[l - 1] : d.in_pad;
    p[k++] = MlpPart{a->w[l], d.w[l].p[0], d.w[l].p[1], in, a->width[l], ld};
    p[k++] = MlpPart{a->b[l], d.b[l], nullptr, 1, a->width[l], 0};
  }
  const int U = a->width[L - 1], ld = d.wpad[L - 1];
  p[k++] = MlpPart{a->mean_w, d.w_head.p[0], d.w_head.p[1], U, 2, ld};
  p[k++] = MlpPart{a->mean_b, d.b_head, nullptr, 1, 2, 0};
  if (a->head == RD_HEAD_SQUASHED) {
    p[k++] = MlpPart{a->log_std_w, d.w_head.p[0] + 2 * (size_t)ld, d.w_head.p[1] + 2 * (size_t)ld, U, 2, ld};
    p[k++] = MlpPart{a->log_std_b, d.b_head + 2, nullptr, 1, 2, 0};
  } else {
    p[k++] = MlpPart{a->log_std, d.log_std, nullptr, 1, 2, 0};
  }
  return k;
}
#define MLP_MAX_PARTS (2 * RD_MLP_MAX_LAYERS + 4)
static_assert(MLP_MAX_PARTS <= GM_PACK_MAX, "mlp_pack packs the whole table in one k_pack_weights launch");

// Everything init and refresh check before any device work: the architecture (against the init's, `same`) and that
// every source is non-null host memory (!on_device) or memory of the current device (on_device).
static inline int mlp_check(MlpPolicy& d, const rd_mlp_actor* a, int n_beams, const rd_mlp_actor* same, bool on_device) {
  if (!a) { d.err = "null actor"; return RD_ERR_INVALID; }
  if (a->n_layers < 1 || a->n_layers > RD_MLP_MAX_LAYERS) {
    d.err = "n_layers " + std::to_string(a->n_layers) + " is not in 1.." + std::to_string(RD_MLP_MAX_LAYERS);
    return RD_ERR_INVALID;
  }
  for (int l = 0; l < a->n_layers; ++l)
    if (a->width[l] < 1 || a->width[l] > RD_MLP_MAX_WIDTH) {
      d.err = "width[" + std::to_string(l) + "] = " + std::to_string(a->width[l]) + " is not in 1.." + std::to_string(RD_MLP_MAX_WIDTH);
      return RD_ERR_INVALID;
    }
  if (a->in_features != n_beams) {
    d.err = "in_features " + std::to_string(a->in_features) + " != the env's n_beams " + std::to_string(n_beams);
    return RD_ERR_INVALID;
  }
  if (n_beams % 4) { d.err = "n_beams must be a multiple of 4 (the scan rows are read by TMA)"; return RD_ERR_INVALID; }
  if (a->activation != RD_ACT_RELU && a->activation != RD_ACT_TANH) { d.err = "bad activation"; return RD_ERR_INVALID; }
  if (a->head != RD_HEAD_SQUASHED && a->head != RD_HEAD_DIAG) { d.err = "bad head kind"; return RD_ERR_INVALID; }
  if (a->head == RD_HEAD_SQUASHED && !(a->log_std_min <= a->log_std_max)) { d.err = "log_std_min > log_std_max"; return RD_ERR_INVALID; }
  if (same) {
    bool eq = a->n_layers == same->n_layers && a->in_features == same->in_features && a->activation == same->activation &&
              a->head == same->head && (a->head != RD_HEAD_SQUASHED ||
                                        (a->log_std_min == same->log_std_min && a->log_std_max == same->log_std_max));
    for (int l = 0; eq && l < a->n_layers; ++l) eq = a->width[l] == same->width[l];
    if (!eq) { d.err = "the weights' architecture, activation or head differ from the ones the actor was initialised with"; return RD_ERR_INVALID; }
  }
  MlpPart parts[MLP_MAX_PARTS];
  const int n_parts = mlp_parts(d, a, parts);
  int dev = 0;
  DR_TRY(cudaGetDevice(&dev));
  for (int k = 0; k < n_parts; ++k) {
    if (!parts[k].src) { d.err = "null weight pointer"; return RD_ERR_INVALID; }
    cudaPointerAttributes at{};
    DR_TRY(cudaPointerGetAttributes(&at, parts[k].src));
    const bool device_ptr = at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged;
    if (on_device && (!device_ptr || at.device != dev)) { d.err = "on_device: a weight pointer is not memory of the policy's device"; return RD_ERR_INVALID; }
    if (!on_device && at.type == cudaMemoryTypeDevice) { d.err = "a weight pointer is device memory where host memory is expected (init, or on_device = 0)"; return RD_ERR_INVALID; }
  }
  return RD_OK;
}

// Packs a (checked by mlp_check) into the buffers init allocated, on `s`: host sources are first copied to d.stage,
// then one k_pack_weights<KMAJOR = true> launch packs the table.
static inline int mlp_pack(MlpPolicy& d, const rd_mlp_actor* a, bool on_device, cudaStream_t s) {
  MlpPart parts[MLP_MAX_PARTS];
  const int n_parts = mlp_parts(d, a, parts);
  PackArgs pa{};
  pa.n_jobs = n_parts;
  size_t off = 0;
  for (int k = 0; k < n_parts; ++k) {
    const MlpPart& p = parts[k];
    const size_t count = (size_t)p.in * p.out;
    const float* src = p.src;
    if (!on_device) {
      DR_TRY(cudaMemcpyAsync(d.stage + off, p.src, count * sizeof(float), cudaMemcpyHostToDevice, s));
      src = d.stage + off;
    }
    PackJob& J = pa.job[k];
    J.src = src; J.hi = p.hi; J.lo = p.lo;
    J.in = p.in; J.out = p.out; J.ld = p.ld; J.k_from = 1 << 30; J.k_shift = 0; J.raw = p.ld ? 0 : 1;
    J.begin = (long long)off;
    off += count;
  }
  pa.total = (long long)off;
  const unsigned grid = (unsigned)std::min<size_t>((off + 255) / 256, (size_t)d.sm_count * 8);
  k_pack_weights<true><<<grid, 256, 0, s>>>(pa);
  DR_TRY(cudaGetLastError());
  return RD_OK;
}

static inline int mlp_init(MlpPolicy& d, int n, int n_beams, const rd_mlp_actor* a) {
  if (int rc = mlp_check(d, a, n_beams, nullptr, false)) return rc;
  if (!gm_get_encoder()) { d.err = "cuTensorMapEncodeTiled is not available from this driver"; return RD_ERR_CUDA; }
  mlp_free(d);
  d.arch = *a;
  for (auto& p : d.arch.w) p = nullptr;
  for (auto& p : d.arch.b) p = nullptr;
  d.arch.mean_w = d.arch.mean_b = d.arch.log_std_w = d.arch.log_std_b = d.arch.log_std = nullptr;
  const int L = a->n_layers;
  d.n = n;
  d.in_pad = n_beams;
  for (int l = 0; l < RD_MLP_MAX_LAYERS; ++l) d.wpad[l] = l < L ? mlp_pad4(a->width[l]) : 0;
  int dev = 0;
  DR_TRY(cudaGetDevice(&dev));
  DR_TRY(cudaDeviceGetAttribute(&d.sm_count, cudaDevAttrMultiProcessorCount, dev));
  auto vec = [&](float*& p, size_t count) -> cudaError_t {
    cudaError_t e = cudaMalloc(&p, count * sizeof(float));
    if (e != cudaSuccess) return e;
    d.owned.push_back(p);
    return cudaMemset(p, 0, count * sizeof(float));
  };
  size_t stage_floats = 0;
  for (int l = 0; l < L; ++l) {
    const int ld = l ? d.wpad[l - 1] : d.in_pad;
    DR_TRY(dr_alloc(d, d.w[l], (size_t)d.wpad[l], (size_t)ld));
    DR_TRY(vec(d.b[l], (size_t)d.wpad[l]));
    stage_floats += (size_t)(l ? a->width[l - 1] : a->in_features) * a->width[l] + a->width[l];
  }
  DR_TRY(dr_alloc(d, d.w_head, 4, (size_t)d.wpad[L - 1]));
  DR_TRY(vec(d.b_head, 4));
  DR_TRY(vec(d.log_std, 2));
  stage_floats += (size_t)4 * a->width[L - 1] + 4;
  DR_TRY(vec(d.stage, stage_floats));
  if (int rc = mlp_pack(d, a, false, 0)) return rc;
  DR_TRY(cudaDeviceSynchronize());
  const size_t N = (size_t)n;
  DR_TRY(dr_alloc(d, d.lidar, N, (size_t)d.in_pad));
  DR_MAP(dr_view(d, d.lidar, d.lidar, 0, d.in_pad, N, d.in_pad, GM_BM));
  for (int l = 0; l < L; ++l) {
    DR_TRY(dr_alloc(d, d.act[l], N, (size_t)d.wpad[l]));
    DR_MAP(dr_view(d, d.act[l], d.act[l], 0, d.wpad[l], N, d.wpad[l], GM_BM));
    const int ld = l ? d.wpad[l - 1] : d.in_pad;
    DR_MAP(dr_view(d, d.w[l], d.w[l], 0, ld, d.wpad[l], ld, DR_ACT_BN));
  }
  DR_MAP(dr_view(d, d.w_head, d.w_head, 0, d.wpad[L - 1], 4, d.wpad[L - 1], GM_BN));
  DR_TRY(vec(d.head_raw, N * 4));
  d.step = 0;
  d.ready = true;
  return RD_OK;
}

// New weights of the init's architecture (mlp_check), packed on `s`; the step counter is kept.
static inline int mlp_set_weights(MlpPolicy& d, const rd_mlp_actor* a, int n_beams, bool on_device, cudaStream_t s) {
  if (int rc = mlp_check(d, a, n_beams, &d.arch, on_device)) return rc;
  return mlp_pack(d, a, on_device, s);
}

// The head of one actor step, one thread per env: mean, std = exp(log_std) (clamped per-state log_std for
// RD_HEAD_SQUASHED, the vector for RD_HEAD_DIAG), u = mean + std e, a = tanh(u) (squashed) or u (diag, unclipped).
// e = 0 when deterministic; else the noise mode's normal (Philox block (env id, step, 0, RD_STREAM_MLP) -> z0, z1, drawn
// before griddepcontrol.wait as in k_actor_train: the draws do not depend on the head's k_dense).
struct MlpHeadArgs {
  const float* raw;       // [n][4] head pre-activations (k_dense<EPI_ACTOR>)
  const float* log_std;   // [2] (diag)
  float* actions;         // [n][2]
  float* dbg;             // [n][RD_MLP_DEBUG_FLOATS] or null
  const float* eps;       // [n][2] (explicit)
  int n, squashed, deterministic, noise;
  float ls_min, ls_max;
  uint32_t key0, key1, step, gid0;
};
__global__ void __launch_bounds__(256) k_mlp_head(const MlpHeadArgs h) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= h.n) return;
  float z[4] = {0.f, 0.f, 0.f, 0.f};
  const bool draw = !h.deterministic && h.noise == GM_NOISE_PHILOX;
  if (draw) gm_normal4(h.gid0 + (uint32_t)e, h.step, 0u, RD_STREAM_MLP, h.key0, h.key1, z);
  asm volatile("griddepcontrol.wait;" ::: "memory");
  if (!h.deterministic && h.noise == GM_NOISE_EXPLICIT) { z[0] = h.eps[2 * (size_t)e]; z[1] = h.eps[2 * (size_t)e + 1]; }
  const float4 x = *reinterpret_cast<const float4*>(h.raw + (size_t)e * 4);
  const float mean[2] = {x.x, x.y};
  float ls[2];
  if (h.squashed) { ls[0] = fminf(fmaxf(x.z, h.ls_min), h.ls_max); ls[1] = fminf(fmaxf(x.w, h.ls_min), h.ls_max); }
  else { ls[0] = h.log_std[0]; ls[1] = h.log_std[1]; }
  float a[2], sd[2];
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    sd[k] = expf(ls[k]);
    const float u = h.deterministic ? mean[k] : __fadd_rn(mean[k], __fmul_rn(sd[k], z[k]));
    a[k] = h.squashed ? tanhf(u) : u;
  }
  h.actions[2 * (size_t)e] = a[0];
  h.actions[2 * (size_t)e + 1] = a[1];
  if (h.dbg) {
    float* d = h.dbg + (size_t)e * RD_MLP_DEBUG_FLOATS;
    d[0] = mean[0]; d[1] = mean[1]; d[2] = sd[0]; d[3] = sd[1];
  }
}

// Uniform random actions: Philox block (env id, step, 0, RD_STREAM_RANDOM), a_k = 2 (x_k >> 8) 2^-24 - 1 (exact).
__global__ void __launch_bounds__(256) k_random_actions(float* __restrict__ actions, int n, uint32_t key0, uint32_t key1,
                                                        uint32_t step, uint32_t gid0) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  uint32_t c[4] = {gid0 + (uint32_t)e, step, 0u, RD_STREAM_RANDOM};
  philox4x32_10(c, key0, key1);
  actions[2 * (size_t)e] = 2.0f * ((float)(c[0] >> 8) * (1.0f / 16777216.0f)) - 1.0f;
  actions[2 * (size_t)e + 1] = 2.0f * ((float)(c[1] >> 8) * (1.0f / 16777216.0f)) - 1.0f;
}

// Enqueues one actor step on `s`; *launched = the kernels launched.
static inline int mlp_step(MlpPolicy& d, const float* obs, float* actions, int deterministic, int noise, const float* eps,
                           float* debug, uint64_t seed, uint32_t gid0, cudaStream_t s, int* launched) {
  *launched = 0;
  const int L = d.arch.n_layers;
  {   // 0. the scan's TF32 split (the env already normalised it)
    const size_t count4 = (size_t)d.n * d.in_pad / 4;
    const unsigned grid = (unsigned)std::min<size_t>((count4 + 255) / 256, 148 * 8);
    k_embed_lidar<<<grid, 256, 0, s>>>(reinterpret_cast<const float4*>(obs), reinterpret_cast<float4*>(d.lidar.p[0]),
                                       reinterpret_cast<float4*>(d.lidar.p[1]), count4, 0, nullptr, d.in_pad / 4);
    DR_TRY(cudaGetLastError());
    ++*launched;
  }
  GemmMaps maps;
  for (int l = 0; l < L; ++l) {   // 1. trunk: act(x W^T + b)
    GemmArgs g{};
    g.M = d.n; g.N = d.wpad[l];
    const DreamerPolicy::Operand& a = l ? d.act[l - 1] : d.lidar;
    const DrTerm t[1] = {{&a, &d.w[l], l ? d.wpad[l - 1] : d.in_pad, 0}};
    dr_build(d, maps, g, t, 1, 1, nullptr, nullptr, 1, 4);
    g.bias = d.b[l]; g.out = d.act[l].p[0]; g.out_lo = d.act[l].p[1]; g.ldo = d.wpad[l];
    maps.o[0] = d.act[l].m[0]; maps.o[1] = d.act[l].m[1];
    if (d.arch.activation == RD_ACT_RELU)
      DR_TRY((gm_launch<EPI_DENSE_RELU, 1, 4, DR_ACT_STAGES, true, DR_ACT_EW, DR_ACT_BN>(maps, g, s)));
    else
      DR_TRY((gm_launch<EPI_DENSE_TANH, 1, 4, DR_ACT_STAGES, true, DR_ACT_EW, DR_ACT_BN>(maps, g, s)));
    ++*launched;
  }
  {   // 2. head pre-activations [n][4] (the Dreamer hout launch's instantiation)
    GemmArgs g{};
    g.M = d.n; g.N = 4;
    const DrTerm t[1] = {{&d.act[L - 1], &d.w_head, d.wpad[L - 1], 0}};
    dr_build(d, maps, g, t, 1, 1, nullptr, nullptr, 1, 4);
    g.bias = d.b_head; g.out = d.head_raw;
    DR_TRY((gm_launch<EPI_ACTOR, 1, 4, 4, true>(maps, g, s)));
    ++*launched;
  }
  {   // 3. k_mlp_head, launched while the head's k_dense drains (griddepcontrol.wait in the kernel)
    MlpHeadArgs h{};
    h.raw = d.head_raw; h.log_std = d.log_std; h.actions = actions; h.dbg = debug; h.eps = eps;
    h.n = d.n; h.squashed = d.arch.head == RD_HEAD_SQUASHED; h.deterministic = deterministic; h.noise = noise;
    h.ls_min = d.arch.log_std_min; h.ls_max = d.arch.log_std_max;
    h.key0 = (uint32_t)seed; h.key1 = (uint32_t)(seed >> 32) ^ RD_STREAM_MLP; h.step = d.step; h.gid0 = gid0;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)((d.n + 255) / 256));
    cfg.blockDim = dim3(256);
    cfg.stream = s;
    cudaLaunchAttribute attrs[1];
    attrs[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attrs[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attrs;
    cfg.numAttrs = 1;
    DR_TRY(cudaLaunchKernelEx(&cfg, k_mlp_head, h));
    ++*launched;
  }
  d.step++;
  return RD_OK;
}
