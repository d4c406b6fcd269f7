// rd_policy.cuh -- on-device policies: the follow-the-gap controller, one warp per env (SURVEY.md §8-f2).
//
// Replaces AgentNode.laserscan_callback + publish_drive_from_heading + PID.calculate
// [REF ros_agent/agents/follow_the_gap/src/agent.py:128-193, 200-238, 45-55] for a batch of envs whose scans are
// already in HBM (the rows k_lidar just wrote), so a closed-loop rollout never leaves the device.
//
// Per env (one warp, lanes over beams; the forward arc of the scan and its "adjusted" copy live in shared memory):
//   clip to the lookahead distance -> |first difference| -> candidates = differences that are the maximum of their
//   10-degree window (reflected border), exceed 9 x the window median (clamped border) and 0.2 m -> every candidate
//   lowers the adjusted ranges inside the arc a vehicle-width chord subtends at the nearer side -> the 83.3rd
//   percentile of the adjusted ranges (np.percentile's linear rule) -> heading = mean angle of the beams at or above
//   it, heading distance = their mean range -> PID -> steering angle, speed -> env action.
// The median test needs no sort: d > 9*median  <=>  at least w/2+1 window elements x satisfy 9*x < d.
// The percentile needs two order statistics of ~721 values: bisection on the bit patterns of their float32 codes
// (monotone for non-negative floats) with warp-wide counts, skipped when both are the lookahead distance itself.
// All arithmetic is float64 in the reference's operation order (translation unit compiled with -fmad=false); the only
// differences to NumPy are the summation order of the two means and acos() vs libm (<= 2 ulp).
#pragma once
#include "rd_common.cuh"

struct PolicyState {
  double* f64;    // [4][n]: PID previous input (NaN = none), PID integral, steering_angle, vehicle_speed
  int32_t* i32;   // [2][n]: scans seen, headings seen (the two "first message" gates of the node)
  float* dr_feat; // Dreamer agent: current latent rows [n][dr_ld] = stoch | previous action | deter (null: not attached)
  float* dr_feat_lo;   // their TF32 remainder parts (null in single-pass mode)
  int dr_ld;
  const int* dr_row;   // env -> latent row (several agents: rows ordered by agent); null: row = env
};
enum { RD_P_PREV = 0, RD_P_INT, RD_P_STEER, RD_P_SPEED, RD_NP_F64 };
enum { RD_P_SCANS = 0, RD_P_HEADINGS, RD_NP_I32 };

__device__ __forceinline__ void rd_policy_clear(const PolicyState& ps, int n, int e) {
  if (ps.dr_feat) {   // `state is None`: zero latent, zero previous action [REF ros_agent/models/dreamer/racing_dreamer.py:66-68]
    const size_t r = ps.dr_row ? (size_t)ps.dr_row[e] : (size_t)e;
    float4* row = reinterpret_cast<float4*>(ps.dr_feat + r * ps.dr_ld);
    for (int k = 0; k < ps.dr_ld / 4; ++k) row[k] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (ps.dr_feat_lo) {
      float4* lo = reinterpret_cast<float4*>(ps.dr_feat_lo + r * ps.dr_ld);
      for (int k = 0; k < ps.dr_ld / 4; ++k) lo[k] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
  }
  if (!ps.i32) return;
  ps.f64[(size_t)RD_P_PREV * n + e] = __longlong_as_double(0x7ff8000000000000ll);
  ps.f64[(size_t)RD_P_INT * n + e] = 0.0;
  ps.f64[(size_t)RD_P_STEER * n + e] = 0.0;
  ps.f64[(size_t)RD_P_SPEED * n + e] = 0.0;
  ps.i32[(size_t)RD_P_SCANS * n + e] = 0;
  ps.i32[(size_t)RD_P_HEADINGS * n + e] = 0;
}

struct GapArgs {
  rd_gap_follower g;
  PolicyState ps;
  const float* lidar;     // [n][n_beams], metres, index 0 = left
  const float* speed;     // [n] or null
  const double2* state_sv; // env state group (steer, v) (v is used when speed is null)
  float* actions;         // [n][2]
  double* debug;          // [n][4] or null
  int n, n_beams, m_pad;  // m_pad: floats per shared-memory row
  int rescale;
  double low[2], high[2];
  double a_drive, c_drag, steer_scale;   // steer_scale = steer_gain * steer_max
};

__device__ __forceinline__ double rd_warp_sum(double v) {
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
  return v;
}

// numpy float64 -> int64 cast followed by np.clip(., 0, hi): truncation toward zero; NaN and out-of-range values
// become INT64_MIN on x86 and therefore clip to 0.
__device__ __forceinline__ int rd_trunc_clip(double x, int hi) {
  if (!(x > -9.0e18 && x < 9.0e18)) return 0;
  long long k = (long long)x;
  return k < 0 ? 0 : (k > hi ? hi : (int)k);
}

// Ranges are kept in shared memory as float32 codes: the LiDAR's float32 value itself, or +inf for "clipped to the
// lookahead distance" (which is not a float32 number).  The code order equals the value order, so min() and the
// percentile selection work on the codes; rd_decode() gives back the exact float64 the reference computes with.
#define RD_CLIP_CODE 0x7f800000u
__device__ __forceinline__ double rd_decode(float f, double lookahead) {
  return (__float_as_uint(f) == RD_CLIP_CODE) ? lookahead : (double)f;
}

// ITEMS: adjusted ranges per lane held in registers for the percentile selection (32 * ITEMS >= beams in the arc)
template <int WARPS, int ITEMS>
__global__ void __launch_bounds__(WARPS * 32) k_gap_follower(GapArgs A) {
  extern __shared__ float sm_pol[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int e = blockIdx.x * WARPS + warp;
  if (e >= A.n) return;   // warps are independent: no block-wide barrier below
  const rd_gap_follower& g = A.g;
  const int n = A.n;
  float* rng = sm_pol + (size_t)warp * 2 * A.m_pad;
  float* adj = rng + A.m_pad;
  const int M = g.arc_last - g.arc_first + 1;
  const double look = g.lookahead;
  int scans = A.ps.i32[(size_t)RD_P_SCANS * n + e] + 1;
  int headings = A.ps.i32[(size_t)RD_P_HEADINGS * n + e];
  double steering_angle = A.ps.f64[(size_t)RD_P_STEER * n + e];
  double vehicle_speed = A.ps.f64[(size_t)RD_P_SPEED * n + e];
  double heading = 0.0, heading_dist = 0.0;
  if (scans >= 2) {   // the first scan after a reset only arms the node's timestamp [REF agent.py:132-134]
    const float* row = A.lidar + (size_t)e * A.n_beams;
    for (int j = lane; j < M; j += 32) {
      float r = row[(A.n_beams - 1) - (g.arc_first + j)];
      r = r < 0.0f ? 0.0f : r;
      if ((double)r >= look) r = __uint_as_float(RD_CLIP_CODE);   // np.clip(ranges, 0, lookahead_distance)
      rng[j] = r;
      adj[j] = r;
    }
    __syncwarp();
    const int nd = M - 1, w = g.filter_width, half = w >> 1;
    const double inc = g.angle_increment, amin = g.angle_min;
    const double ang0 = (double)g.arc_first * inc + amin;
    const double w2 = g.vehicle_width * g.vehicle_width;
    for (int base = 0; base < nd; base += 32) {
      const int i = base + lane;
      bool cand = false;
      if (i < nd) {
        const double d = fabs(rd_decode(rng[i + 1], look) - rd_decode(rng[i], look));
        if (d > g.minimum_gap_length) {
          bool ismax = true;
          int below = 0;
          for (int k = 0; k < w; ++k) {
            const int j = i - half + k;
            const int jr = j < 0 ? -j - 1 : (j >= nd ? 2 * nd - j - 1 : j);   // maximum_filter1d: mode 'reflect'
            const int jc = j < 0 ? 0 : (j >= nd ? nd - 1 : j);                // median_filter: mode 'nearest'
            const double dr = fabs(rd_decode(rng[jr + 1], look) - rd_decode(rng[jr], look));
            const double dc = (jc == jr) ? dr : fabs(rd_decode(rng[jc + 1], look) - rd_decode(rng[jc], look));
            if (dr > d) ismax = false;
            if (dc * g.median_dev_threshold < d) ++below;
          }
          cand = ismax && below >= half + 1;
        }
      }
      unsigned bal = __ballot_sync(0xffffffffu, cand);
      while (bal) {   // every lane handles the same candidate: its chord lowers a run of adjusted ranges
        const int ii = base + (__ffs(bal) - 1);
        bal &= bal - 1;
        float Lc = rng[ii];
        if (ii > 0) Lc = fminf(Lc, rng[ii - 1]);   // the reference's slice is empty (and raises) for ii == 0
        Lc = fminf(Lc, rng[ii + 1]);
        const double L = rd_decode(Lc, look);
        const double theta = (double)(g.arc_first + ii) * inc + amin;
        const double L2 = L * L;
        const double beta = acos((2.0 * L2 - w2) / (2.0 * L2));
        const int k0 = rd_trunc_clip(((theta - beta) - ang0) / inc, M - 1);
        const int k1 = rd_trunc_clip(((theta + beta) - ang0) / inc, M - 1);
        for (int k = k0 + lane; k <= k1; k += 32) adj[k] = fminf(adj[k], Lc);
        __syncwarp();   // the next candidate's run overlaps this one's with a different lane -> element mapping
      }
    }
    __syncwarp();
    // two order statistics of adj[0..M): when enough beams are still clipped both are the lookahead distance itself
    // (open track ahead); otherwise bisection on the codes' bit patterns (monotone for non-negative floats)
    double x, y;
    unsigned key[ITEMS];   // codes of this lane's adjusted ranges; slots past the arc hold the maximum code
    unsigned n_clip = 0;
#pragma unroll
    for (int t = 0; t < ITEMS; ++t) {
      const int j = lane + 32 * t;
      key[t] = (j < M) ? __float_as_uint(adj[j]) : 0xffffffffu;
      n_clip += (key[t] == RD_CLIP_CODE) ? 1u : 0u;
    }
    n_clip = __reduce_add_sync(0xffffffffu, n_clip);
    if ((int)n_clip >= M - g.pct_lo) {
      x = y = look;
    } else {
      unsigned lo = 0xffffffffu, hi = 0;
#pragma unroll
      for (int t = 0; t < ITEMS; ++t) {
        lo = key[t] < lo ? key[t] : lo;
        if (key[t] != 0xffffffffu) hi = key[t] > hi ? key[t] : hi;
      }
      lo = __reduce_min_sync(0xffffffffu, lo);
      hi = __reduce_max_sync(0xffffffffu, hi);
      while (lo < hi) {
        const unsigned mid = lo + ((hi - lo) >> 1);
        unsigned c = 0;
#pragma unroll
        for (int t = 0; t < ITEMS; ++t) c += (key[t] <= mid) ? 1u : 0u;
        c = __reduce_add_sync(0xffffffffu, c);
        if ((int)c >= g.pct_lo + 1) hi = mid; else lo = mid + 1;
      }
      unsigned nxt = lo;
      if (g.pct_hi > g.pct_lo) {
        unsigned c = 0, up = 0xffffffffu;
#pragma unroll
        for (int t = 0; t < ITEMS; ++t) {
          c += (key[t] <= lo) ? 1u : 0u;
          if (key[t] > lo && key[t] < up) up = key[t];
        }
        c = __reduce_add_sync(0xffffffffu, c);
        up = __reduce_min_sync(0xffffffffu, up);
        if ((int)c < g.pct_hi + 1) nxt = up;
      }
      x = rd_decode(__uint_as_float(lo), look);
      y = rd_decode(__uint_as_float(nxt), look);
    }
    const double dxy = y - x;   // numpy _lerp
    const double pct = (g.pct_gamma >= 0.5) ? (y - dxy * (1.0 - g.pct_gamma)) : (x + dxy * g.pct_gamma);
    double sa = 0.0, sr = 0.0, cnt = 0.0;
#pragma unroll
    for (int t = 0; t < ITEMS; ++t) {
      const int j = lane + 32 * t;
      if (j >= M) break;
      const double a = rd_decode(__uint_as_float(key[t]), look);
      if (a >= pct && a < g.range_max) {   // np.digitize(adjusted, [0, pct, range_max]) == 2
        sa += (double)(g.arc_first + j) * inc + amin;
        sr += rd_decode(rng[j], look);
        cnt += 1.0;
      }
    }
    sa = rd_warp_sum(sa); sr = rd_warp_sum(sr); cnt = rd_warp_sum(cnt);
    heading = sa / cnt;
    heading_dist = sr / cnt;
    headings += 1;
    if (headings >= 2) {   // the first heading only arms the PID clock [REF agent.py:206-208]
      const double prev = A.ps.f64[(size_t)RD_P_PREV * n + e];
      double integ = A.ps.f64[(size_t)RD_P_INT * n + e];
      const double err = 0.0 - heading;   // PID.calculate [REF agent.py:45-55]
      const double P = g.kp * err;
      integ = integ + g.ki * err * g.scan_dt;
      const double D = (prev != prev) ? 0.0 : (g.kd * (prev - heading) / g.scan_dt);
      const double control = (g.kp + g.ki + g.kd > 0.0) ? ((P + integ) + D) : heading;
      double ang = -control;
      const double lim = fabs(g.max_steering_angle);
      ang = ang < -lim ? -lim : (ang > lim ? lim : ang);
      const double aabs = fabs(ang);
      double spd = g.max_vehicle_speed;
      if (aabs > g.speed_limit_angle) spd = g.max_vehicle_speed - (aabs / g.max_steering_angle) * (g.max_vehicle_speed * 0.30);
      if (heading_dist < 5.0) spd = fmin(spd, heading_dist / 5.0 * 4.0);
      spd = fmax(spd, 1.5);
      steering_angle = ang;
      vehicle_speed = spd;
      if (lane == 0) {
        A.ps.f64[(size_t)RD_P_PREV * n + e] = heading;
        A.ps.f64[(size_t)RD_P_INT * n + e] = integ;
        A.ps.f64[(size_t)RD_P_STEER * n + e] = ang;
        A.ps.f64[(size_t)RD_P_SPEED * n + e] = spd;
      }
    }
  }
  if (lane == 0) {
    A.ps.i32[(size_t)RD_P_SCANS * n + e] = scans;
    A.ps.i32[(size_t)RD_P_HEADINGS * n + e] = headings;
    // drive command -> env action
    const double v = A.speed ? (double)A.speed[e] : A.state_sv[e].y;
    const double vt = vehicle_speed * g.speed_scale;
    double motor = vt * A.c_drag / A.a_drive + g.speed_gain * (vt - v);
    double steer = steering_angle / A.steer_scale;
    motor = motor < A.low[0] ? A.low[0] : (motor > A.high[0] ? A.high[0] : motor);
    steer = steer < A.low[1] ? A.low[1] : (steer > A.high[1] ? A.high[1] : steer);
    if (A.rescale) {   // inverse of ReduceActionSpace._normalize [REF dreamer/wrappers.py:129-134]
      motor = (motor - A.low[0]) / (A.high[0] - A.low[0]) * 2.0 - 1.0;
      steer = (steer - A.low[1]) / (A.high[1] - A.low[1]) * 2.0 - 1.0;
    }
    A.actions[2 * (size_t)e] = (float)motor;
    A.actions[2 * (size_t)e + 1] = (float)steer;
    if (A.debug) {
      double* d = A.debug + 4 * (size_t)e;
      d[0] = steering_angle; d[1] = vehicle_speed; d[2] = heading; d[3] = heading_dist;
    }
  }
}
