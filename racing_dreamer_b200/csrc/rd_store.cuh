// rd_store.cuh -- device-resident episode store (SURVEY.md §8-f1: "device-side ring buffer -> batched npz flush").
//
// Rows are the reference's Collect rows [REF dreamer/wrappers.py:198-250] as episodes.EpisodeRecorder stores them:
// the observation keys, then action, reward, discount = 1 - done, progress = lap + progress - 1 and time, at precision
// 32 or 16 (_convert: float64 values rounded once, straight to the target type).
//
// Layout: one ring of `cap` rows per env and key, [n_envs][cap][row bytes].  head[e] counts the rows env e has ever
// written (row r lives in slot r % cap), ep_start[e] is the first row of its episode in progress.  An episode that ends
// is committed to a table indexed by its global id modulo M; it stays held while none of its rows has been overwritten
// (start >= head[env] - cap), so an env's oldest episodes are evicted as its ring wraps.  M = n_envs * (cap + 2) table
// slots: a held episode's env writes at most cap rows before the episode is evicted, and no env commits more than
// cap + 1 episodes in that time, so a held episode's slot is never reused.
//
// Import arena (rd_store_import): one more ring of icap rows per key, written from staged host episodes.  Imported
// episode k has id RD_STORE_IMPORTED_ID0 + k, env -1 and its entry in a table of Mi = icap + 1 slots at k mod Mi; it is
// held while its first row has not been overwritten (start >= imp_head - icap).  Every episode has at least one row, so
// a held episode's slot is reused only after icap + 1 later imports, and those overwrite its rows first.  Imports are
// host-driven, so the arena's counters (imp_head, imp_next) are host values passed in StoreDev: every launch sees the
// arena as the imports enqueued before it left it.  The recorded table's bound M relies on the envs stepping in lockstep,
// which imports do not, so imported episodes never go there.
#pragma once
#include <thrust/iterator/counting_iterator.h>
#include <thrust/iterator/transform_iterator.h>
#include <cub/block/block_scan.cuh>
#include <cub/device/device_select.cuh>

#include "rd_common.cuh"

// stored keys, in the order of the episode dicts (EpisodeRecorder: observation keys, then EXTRA_KEYS)
enum { SK_LIDAR = 0, SK_POSE, SK_VELOCITY, SK_SPEED, SK_OCC, SK_ACTION, SK_REWARD, SK_DISCOUNT, SK_PROGRESS, SK_TIME,
       SK_N };

struct StoreEp {          // one committed episode (24 B)
  int64_t id;             // global id; -1 = empty slot
  int64_t start;          // absolute row index of its first row in the env's ring
  int32_t env, len;       // env index, rows
};

struct StoreDev {
  unsigned char* rows[SK_N];   // [n][cap][rb[k]] or null (key not kept)
  int32_t rb[SK_N];            // row bytes per key
  int64_t* head;               // [n] rows written so far
  int64_t* ep_start;           // [n] first row of the episode in progress
  StoreEp* table;              // [M]
  int64_t M;
  int64_t* next_id;            // [1] episodes committed so far
  uint8_t* fin;                // [n] env committed an episode in this step (= reset mask)
  int cap, n, nb, A;
  int half;                    // precision 16: float keys stored as IEEE half
  int lidar_in_half;           // the env emits half scans (RD_OBS_LIDAR_F16)
  // import arena (icap = 0: none)
  unsigned char* imp[SK_N];    // [icap][rb[k]] or null
  StoreEp* itable;             // [Mi]
  int64_t Mi, imp_head, imp_next;   // table slots; arena rows written, episodes imported so far
  int icap;
};

struct StoreSrc {                 // the env's outputs of the step / reset being recorded
  const void* lidar; const uint8_t* occ; const float* pose; const float* vel; const float* speed;
  const float* reward; const uint8_t* done; const float* progress; const int32_t* lap; const float* time;
  const float* actions;
};

// float64 -> IEEE half in one rounding (numpy's astype(float16) of a float64 value)
__device__ __forceinline__ uint16_t st_f64_to_f16(double v) {
  uint16_t h;
  asm("cvt.rn.f16.f64 %0, %1;" : "=h"(h) : "d"(v));
  return h;
}
__device__ __forceinline__ void st_put(unsigned char* row, int i, float v, int half) {
  if (half) reinterpret_cast<__half*>(row)[i] = __float2half_rn(v);
  else reinterpret_cast<float*>(row)[i] = v;
}
__device__ __forceinline__ void st_put_f64(unsigned char* row, int i, double v, int half) {
  if (half) reinterpret_cast<uint16_t*>(row)[i] = st_f64_to_f16(v);
  else reinterpret_cast<float*>(row)[i] = __double2float_rn(v);
}

// byte copy / clear of one row by the threads of a CTA: 16-byte accesses where size and both addresses allow it
// (a float32 LiDAR row of 1080 beams is 4320 B, an occupancy row 4096 B), else 4- or 2-byte ones (rows are whole
// halves at least)
__device__ __forceinline__ void st_copy(unsigned char* dst, const unsigned char* src, int bytes) {
  const unsigned al = (unsigned)bytes | (unsigned)(uintptr_t)dst | (unsigned)(uintptr_t)src;
  if ((al & 15u) == 0) {
    for (int i = threadIdx.x; i < bytes / 16; i += blockDim.x)
      reinterpret_cast<uint4*>(dst)[i] = __ldg(reinterpret_cast<const uint4*>(src) + i);
  } else if ((al & 3u) == 0) {
    for (int i = threadIdx.x; i < bytes / 4; i += blockDim.x)
      reinterpret_cast<uint32_t*>(dst)[i] = __ldg(reinterpret_cast<const uint32_t*>(src) + i);
  } else {
    for (int i = threadIdx.x; i < bytes / 2; i += blockDim.x)
      reinterpret_cast<uint16_t*>(dst)[i] = __ldg(reinterpret_cast<const uint16_t*>(src) + i);
  }
}
__device__ __forceinline__ void st_zero(unsigned char* dst, int bytes) {
  const unsigned al = (unsigned)bytes | (unsigned)(uintptr_t)dst;
  if ((al & 15u) == 0) {
    for (int i = threadIdx.x; i < bytes / 16; i += blockDim.x) reinterpret_cast<uint4*>(dst)[i] = make_uint4(0, 0, 0, 0);
  } else if ((al & 3u) == 0) {
    for (int i = threadIdx.x; i < bytes / 4; i += blockDim.x) reinterpret_cast<uint32_t*>(dst)[i] = 0u;
  } else {
    for (int i = threadIdx.x; i < bytes / 2; i += blockDim.x) reinterpret_cast<uint16_t*>(dst)[i] = 0;
  }
}

// table entry of a recorded or imported id (the caller has checked id >= 0)
__device__ __forceinline__ StoreEp st_entry(const StoreDev& S, int64_t id) {
  if (id < RD_STORE_IMPORTED_ID0) return S.table[id % S.M];
  if (S.Mi == 0) { StoreEp r; r.id = -1; r.start = 0; r.env = -1; r.len = 0; return r; }
  return S.itable[(id - RD_STORE_IMPORTED_ID0) % S.Mi];
}
__device__ __forceinline__ bool st_held(const StoreDev& S, const StoreEp& r, int64_t id) {
  if (r.id != id) return false;
  return r.env < 0 ? r.start >= S.imp_head - (int64_t)S.icap : r.start >= S.head[r.env] - (int64_t)S.cap;
}

// One row per env (one CTA per env): the step's row of every env (reset_rows = 0), or the reset row of every env that
// committed an episode in this step (reset_rows = 1: first row of its next episode).  The reset row is the reset
// observation with speed 0, zero action, reward 0, discount 1, progress -1, time 0 [REF dreamer/wrappers.py:228-238].
__global__ void __launch_bounds__(128) k_store_record(StoreDev S, StoreSrc o, int reset_rows) {
  const int e = blockIdx.x;
  if (reset_rows && !S.fin[e]) return;
  const int64_t h = S.head[e];
  const size_t slot = (size_t)e * (size_t)S.cap + (size_t)(h % S.cap);
  const int nb = S.nb;
  if (unsigned char* dst = S.rows[SK_LIDAR]) {
    dst += slot * (size_t)S.rb[SK_LIDAR];
    if (S.lidar_in_half == S.half) {
      st_copy(dst, reinterpret_cast<const unsigned char*>(o.lidar) + (size_t)e * S.rb[SK_LIDAR], S.rb[SK_LIDAR]);
    } else if (S.half) {         // float32 scans -> half, round to nearest even
      const float* src = reinterpret_cast<const float*>(o.lidar) + (size_t)e * nb;
      for (int i = threadIdx.x; i < nb; i += blockDim.x) reinterpret_cast<__half*>(dst)[i] = __float2half_rn(__ldg(src + i));
    } else {                     // half scans -> float32 (exact)
      const __half* src = reinterpret_cast<const __half*>(o.lidar) + (size_t)e * nb;
      for (int i = threadIdx.x; i < nb; i += blockDim.x) reinterpret_cast<float*>(dst)[i] = __half2float(src[i]);
    }
  }
  if (unsigned char* dst = S.rows[SK_OCC])
    st_copy(dst + slot * (size_t)S.rb[SK_OCC], o.occ + (size_t)e * (RD_OCC_OUT * RD_OCC_OUT), RD_OCC_OUT * RD_OCC_OUT);
  // the small keys: one element per thread
  const int t = threadIdx.x;
  const int hf = S.half;
  if (t < 6) {
    if (S.rows[SK_POSE]) st_put(S.rows[SK_POSE] + slot * (size_t)S.rb[SK_POSE], t, o.pose[(size_t)e * 6 + t], hf);
  } else if (t < 12) {
    if (S.rows[SK_VELOCITY]) st_put(S.rows[SK_VELOCITY] + slot * (size_t)S.rb[SK_VELOCITY], t - 6, o.vel[(size_t)e * 6 + t - 6], hf);
  } else if (t == 12) {
    if (S.rows[SK_SPEED]) st_put(S.rows[SK_SPEED] + slot * (size_t)S.rb[SK_SPEED], 0, reset_rows ? 0.f : o.speed[e], hf);
  } else if (t < 15) {
    st_put(S.rows[SK_ACTION] + slot * (size_t)S.rb[SK_ACTION], t - 13, reset_rows ? 0.f : o.actions[(size_t)e * 2 + t - 13], hf);
  } else if (t == 15) {
    st_put(S.rows[SK_REWARD] + slot * (size_t)S.rb[SK_REWARD], 0, reset_rows ? 0.f : o.reward[e], hf);
  } else if (t == 16) {         // 1 - done in float64 [REF dreamer/wrappers.py:216]
    st_put_f64(S.rows[SK_DISCOUNT] + slot * (size_t)S.rb[SK_DISCOUNT], 0, reset_rows ? 1.0 : (o.done[e] ? 0.0 : 1.0), hf);
  } else if (t == 17) {         // float64(lap) + float64(progress) - 1 [REF dreamer/wrappers.py:218]
    const double p = reset_rows ? -1.0 : __dadd_rn(__dadd_rn((double)o.lap[e], (double)o.progress[e]), -1.0);
    st_put_f64(S.rows[SK_PROGRESS] + slot * (size_t)S.rb[SK_PROGRESS], 0, p, hf);
  } else if (t == 18) {
    st_put(S.rows[SK_TIME] + slot * (size_t)S.rb[SK_TIME], 0, reset_rows ? 0.f : o.time[e], hf);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    if (reset_rows) S.ep_start[e] = h;
    S.head[e] = h + 1;
  }
}

// Commit (one CTA): an env whose world has a car that is done in this step ends its episode; the episodes get
// consecutive ids in env-index order (a world's cars consecutively, agent A first: EpisodeRecorder._flush's order).
// fin[] becomes the reset mask of the step.
constexpr int RD_COMMIT_THREADS = 1024;
__global__ void __launch_bounds__(RD_COMMIT_THREADS) k_store_commit(StoreDev S, const uint8_t* __restrict__ done) {
  using Scan = cub::BlockScan<int, RD_COMMIT_THREADS>;
  __shared__ typename Scan::TempStorage tmp;
  __shared__ int64_t base_s;
  if (threadIdx.x == 0) base_s = *S.next_id;
  __syncthreads();
  for (int c0 = 0; c0 < S.n; c0 += RD_COMMIT_THREADS) {
    const int e = c0 + (int)threadIdx.x;
    int f = 0;
    if (e < S.n) {
      const int w0 = e - e % S.A;
      for (int j = 0; j < S.A; ++j) f |= done[w0 + j] != 0;
    }
    int pre = 0, tot = 0;
    Scan(tmp).ExclusiveSum(f, pre, tot);
    const int64_t base = base_s;
    if (e < S.n) {
      S.fin[e] = (uint8_t)f;
      if (f) {
        StoreEp r;
        r.id = base + pre;
        r.start = S.ep_start[e];
        r.env = e;
        r.len = (int32_t)(S.head[e] - r.start);
        S.table[r.id % S.M] = r;
      }
    }
    __syncthreads();
    if (threadIdx.x == 0) base_s = base + tot;
    __syncthreads();
  }
  if (threadIdx.x == 0) *S.next_id = base_s;
}

// eligibility compaction: the window of the last Mi imported ids in import order, then the window of the last M recorded
// ids in commit order, kept when held and at least min_len rows long (without an arena Mi = 0: the recorded window alone)
struct StoreIdOf {
  const int64_t* next_id; int64_t M, Mi, imp_next;
  __device__ int64_t operator()(int64_t i) const {
    if (i < Mi) {
      const int64_t k = imp_next - Mi + i;
      return k < 0 ? -1 : RD_STORE_IMPORTED_ID0 + k;
    }
    return *next_id - M + (i - Mi);
  }
};
struct StoreEligible {
  StoreDev S; int min_len;
  __device__ bool operator()(int64_t id) const {
    if (id < 0) return false;
    const StoreEp r = st_entry(S, id);
    return st_held(S, r, id) && r.len >= min_len;
  }
};
using StoreIdIter = thrust::transform_iterator<StoreIdOf, thrust::counting_iterator<int64_t>>;

// The draw law [NEW-SPEC; the reference's load_episodes uses numpy's RandomState]: entry b of sample call k takes
// Philox4x32-10(key (seed_lo, seed_hi ^ RD_STREAM_STORE), counter (b, k, 0, 0)) -> x0, x1; episode
// eligible[(x0 * n_elig) >> 32]; start (x1 * (total - L + 1)) >> 32, or with balance min((x1 * total) >> 32, total - L)
// [REF dreamer/tools.py:256-262].
__global__ void __launch_bounds__(128) k_store_draw(StoreDev S, const int64_t* __restrict__ elig, const int* __restrict__ n_elig,
                                                    int B, int L, int balance, uint32_t k0, uint32_t k1, uint32_t call,
                                                    int64_t* req_id, int32_t* req_start) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const int ne = *n_elig;
  if (ne <= 0) { req_id[b] = -1; req_start[b] = -1; return; }
  uint32_t c[4] = {(uint32_t)b, call, 0u, 0u};
  philox4x32_10(c, k0, k1);
  const int64_t id = elig[(uint32_t)(((uint64_t)c[0] * (uint64_t)(uint32_t)ne) >> 32)];
  const uint32_t total = (uint32_t)st_entry(S, id).len;
  uint32_t st;
  if (balance) {
    st = (uint32_t)(((uint64_t)c[1] * (uint64_t)total) >> 32);
    st = min(st, total - (uint32_t)L);
  } else {
    st = (uint32_t)(((uint64_t)c[1] * (uint64_t)(total - (uint32_t)L + 1u)) >> 32);
  }
  req_id[b] = id;
  req_start[b] = (int32_t)st;
}

struct StoreOut {
  unsigned char* p[SK_N];       // [B][L][rb[k]] or null
  int64_t* id; int32_t* start;  // [B]
};

// Gather of [B, L] chunks, one CTA per (entry, row), every key.  Requests are checked here: an id that is not held, or
// a chunk outside its episode, reads nothing from the store, yields zero rows and id / start -1, and (count_invalid:
// caller-given indices) is counted.
__global__ void __launch_bounds__(128) k_store_gather(StoreDev S, StoreOut O, const int64_t* __restrict__ req_id,
                                                      const int32_t* __restrict__ req_start, int L, int count_invalid,
                                                      unsigned long long* invalid) {
  const int64_t row = blockIdx.x;
  const int b = (int)(row / L), t = (int)(row % L);
  const int64_t id = req_id[b];
  const int32_t st = req_start[b];
  bool ok = false;
  StoreEp r{};
  if (id >= 0) {
    r = st_entry(S, id);
    ok = st_held(S, r, id) && st >= 0 && (int64_t)st + L <= (int64_t)r.len;
  }
  const bool imported = r.env < 0;
  if (t == 0 && threadIdx.x == 0) {
    O.id[b] = ok ? id : -1;
    O.start[b] = ok ? st : -1;
    if (!ok && count_invalid) atomicAdd(invalid, 1ull);
  }
  size_t src_slot = 0;
  if (ok) src_slot = imported ? (size_t)((r.start + st + t) % S.icap)
                              : (size_t)r.env * (size_t)S.cap + (size_t)((r.start + st + t) % S.cap);
#pragma unroll
  for (int k = 0; k < SK_N; ++k) {   // unrolled: the key descriptors stay in the parameter space
    unsigned char* dst = O.p[k];
    if (!dst || !S.rows[k]) continue;
    const int rb = S.rb[k];
    dst += (size_t)row * rb;
    if (ok) st_copy(dst, (imported ? S.imp[k] : S.rows[k]) + src_slot * rb, rb);
    else st_zero(dst, rb);
  }
}

// (id, env, rows) of the first n compacted ids (export)
__global__ void k_store_export(StoreDev S, const int64_t* __restrict__ ids, int n, int64_t* out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const StoreEp r = st_entry(S, ids[i]);
  out[3 * i] = r.id; out[3 * i + 1] = r.env; out[3 * i + 2] = r.len;
}

// Import of staged rows, one CTA per staged row: row r of the call goes to arena row imp_head + r, converted from the
// staged type to the store's (numpy astype: one rounding); the first CTAs also write the table entries of the call's
// episodes.  A call of more than icap rows writes only its last icap rows and the entries of its last icap episodes:
// the others are overwritten within the call (an episode held afterwards has fewer than icap rows after its first, so
// fewer than icap episodes after it).
struct StoreStaged {
  const unsigned char* p[SK_N];   // [rows][elements of the key] or null (key not kept)
  int32_t type[SK_N];             // RD_STORE_U8 | F16 | F32 | F64 (element bytes)
  int32_t ne[SK_N];               // elements per row
};

template <typename T> __device__ __forceinline__ double st_ld(const T* p, int i);
template <> __device__ __forceinline__ double st_ld<__half>(const __half* p, int i) { return (double)__half2float(p[i]); }
template <> __device__ __forceinline__ double st_ld<float>(const float* p, int i) { return (double)p[i]; }
template <> __device__ __forceinline__ double st_ld<double>(const double* p, int i) { return p[i]; }

// one row of n elements of type T into the store's float type; groups of 8 elements as 16-byte loads and stores where
// n and both addresses allow it (a LiDAR row of 1080 beams), element by element otherwise.  Every value takes the path of
// st_put_f64: widening to double is exact, so this is one rounding from the staged value.
template <typename T>
__device__ __forceinline__ void st_convert_row(unsigned char* dst, const unsigned char* src, int n, int half) {
  const T* s = reinterpret_cast<const T*>(src);
  const unsigned al = (unsigned)(uintptr_t)dst | (unsigned)(uintptr_t)src;
  if ((n & 7) == 0 && (al & 15u) == 0) {
    for (int g = threadIdx.x; g < n / 8; g += blockDim.x) {
      alignas(16) T v[8];
#pragma unroll
      for (int q = 0; q < (int)(8 * sizeof(T)) / 16; ++q)
        reinterpret_cast<uint4*>(v)[q] = __ldg(reinterpret_cast<const uint4*>(s + 8 * g) + q);
      if (half) {
        alignas(16) uint16_t h[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) h[j] = st_f64_to_f16(st_ld(v, j));
        reinterpret_cast<uint4*>(dst)[g] = *reinterpret_cast<const uint4*>(h);
      } else {
        alignas(16) float f[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) f[j] = __double2float_rn(st_ld(v, j));
        reinterpret_cast<uint4*>(dst)[2 * g] = *reinterpret_cast<const uint4*>(f);
        reinterpret_cast<uint4*>(dst)[2 * g + 1] = *reinterpret_cast<const uint4*>(f + 4);
      }
    }
  } else {
    for (int i = threadIdx.x; i < n; i += blockDim.x) st_put_f64(dst, i, st_ld(s, i), half);
  }
}

__global__ void __launch_bounds__(128) k_store_import(StoreDev S, StoreStaged in, int64_t rows, const int32_t* __restrict__ lens,
                                                      const int64_t* __restrict__ first, int n_ep) {
  const int64_t r = (int64_t)blockIdx.x + (rows > S.icap ? rows - S.icap : 0);
  const int n_w = min(n_ep, S.icap);   // <= gridDim.x = min(rows, icap)
  if ((int)blockIdx.x < n_w && threadIdx.x == 0) {
    const int j = (int)blockIdx.x + (n_ep - n_w);
    StoreEp e;
    e.id = RD_STORE_IMPORTED_ID0 + S.imp_next + j;
    e.start = S.imp_head + first[j];
    e.env = -1;
    e.len = lens[j];
    S.itable[(S.imp_next + j) % S.Mi] = e;
  }
  if (r >= rows) return;
  const size_t slot = (size_t)((S.imp_head + r) % S.icap);
#pragma unroll
  for (int k = 0; k < SK_N; ++k) {
    unsigned char* dst = S.imp[k];
    if (!dst) continue;
    const int rb = S.rb[k];
    dst += slot * rb;
    const int ne = in.ne[k], ty = in.type[k];
    const unsigned char* src = in.p[k] + (size_t)r * (size_t)ne * (size_t)ty;
    const int store_ty = k == SK_OCC ? RD_STORE_U8 : (S.half ? RD_STORE_F16 : RD_STORE_F32);
    if (ty == store_ty) st_copy(dst, src, rb);
    else if (ty == RD_STORE_F16) st_convert_row<__half>(dst, src, ne, S.half);
    else if (ty == RD_STORE_F32) st_convert_row<float>(dst, src, ne, S.half);
    else st_convert_row<double>(dst, src, ne, S.half);
  }
}
