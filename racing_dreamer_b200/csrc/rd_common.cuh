// rd_common.cuh -- shared device-side types and helpers of librd_env.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <stdint.h>

#include "../../include/rd_env.h"

#define RD_MAX_MAPS 8
#include "rd_march.cuh"           // RD_SUB_BITS = 12 (origin quantum 2^-12 cell), RD_DIR_BITS = 18 (direction 2^-18)
#define RD_COARSE_SHIFT 2         // clearance field block = 4 x 4 cells
#define RD_OCC_IN 220             // OccupancyMapObs crop [REF dreamer/wrappers.py:398-399]
#define RD_OCC_MID 200
#define RD_OCC_OUT 64

// One track on the device.  bits: y-up rows of rw u32 words, bit = drivable.  dist: y-up u16.
struct DevMap {
  const uint32_t* bits;  // followed, at byte offset coarse_off, by the block clearance field (one allocation)
  const uint16_t* dist;
  const double* start;   // [n_start][3]
  const double* reset;   // [n_reset][3]
  const int32_t* ball_next;  // [n_reset] the reset pose cfg.ball_spacing metres further along the lap (multi-agent resets)
  int h, w, rw, col0, row0, full_h, dmax, n_start, n_reset;
  int bits_bytes;        // bytes of bits + clearance field, each rounded up to 16 (bulk-copy granularity)
  int coarse_off;        // byte offset of the clearance field u8[ch][cw] (rd_march.cuh)
  int cw, ch, cshift;
  double res, inv_res, ox, oy;
  double inv_dmax;       // RN(1 / dmax): progress = dist / dmax by one multiply + two fma (rdv_div_by, correctly rounded)
};

// Per-env record handed from the dynamics/reset kernel to the LiDAR and occupancy kernels (48 B, 16-B aligned).
struct __align__(16) OriginRec {
  int32_t px, py;        // sensor origin in 2^-12 cells relative to the crop
  int32_t valid;         // bit0: origin inside a drivable cell; bit1: px/py hold the position
  uint32_t gid;          // global env id (noise counter)
  uint32_t episode, step;
  int32_t was_reset;     // env was reset in this call (occupancy obs = zeros) ; 2 = frozen (leave outputs)
  int32_t pad;
  double c, s;           // cos/sin of the heading
};

struct LidarParams {
  int n_beams;
  int groups;            // ceil(n_beams / 32)
  int gpi;               // beam groups per work item (1 or 2, see k_lidar)
  int units;             // work items per env: ceil(groups / gpi)
  unsigned groups_magic; // ceil(2^32 / units): item / units == umulhi(item, groups_magic) (k_lidar)
  unsigned envs_magic;   // ceil(2^32 / n_env of the launch), centre_first order
  int centre_first;      // work order: beam groups from the centre of the scan outwards, envs innermost
  int normalize;         // 1: RD_OBS_LIDAR_NORM (r / range_max - 0.5); 2: RD_OBS_NORM_BASELINES ((r - norm_lo) * norm_sc)
  double norm_lo, norm_sc;
  int f16;               // RD_OBS_LIDAR_F16: rows are stored as IEEE half
  float range_min, range_max, noise;
  float scale;           // metres per (sub-cell / direction unit) = 2^(DIR-SUB) * resolution
  int64_t rsub;          // range_max in sub-cells
  uint32_t key0, key1;   // Philox key of the noise stream
  // multi-agent worlds: the other cars of the world are seen by the scan (agents <= 1: off)
  int agents;            // cars per world; env e belongs to world e / agents
  int car_reach;         // |origin difference| (sub-cells, per axis) beyond which a car cannot be within range
  int car_radius_sub;    // radius (sub-cells) of a disc around a car's SENSOR origin that contains its body box
  float car_ulo, car_uhi, car_hw;  // body box in the OTHER car's sensor frame, cells: u in [ulo, uhi], |v| <= hw
  float res;             // metres per cell
};

// ---- Philox4x32-10 (counter-based RNG; identical integer arithmetic in the oracle) ----
__device__ __forceinline__ void philox4x32_10(uint32_t (&c)[4], uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
    uint32_t hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
    uint32_t n0 = hi1 ^ c[1] ^ k0, n2 = hi0 ^ c[3] ^ k1;
    c[0] = n0; c[1] = lo1; c[2] = n2; c[3] = lo0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
}
#define RD_STREAM_RESET 0x52455345u
#define RD_STREAM_LIDAR 0x4c494441u
#define RD_STREAM_STORE 0x53544f52u   // episode-store sampler (rd_store.cuh)

// ---- map lookups (global memory, read-only path) ----
__device__ __forceinline__ bool rd_cell_of(const DevMap& m, double x, double y, int& cx, int& cy) {
  double u = (x - m.ox) * m.inv_res;
  double v = (y - m.oy) * m.inv_res;
  double fu = floor(u), fv = floor(v);
  if (!(fu > -1.0e9 && fu < 1.0e9 && fv > -1.0e9 && fv < 1.0e9)) { cx = -1; cy = -1; return false; }
  cx = (int)fu - m.col0;
  cy = (int)fv - m.row0;
  return cx >= 0 && cx < m.w && cy >= 0 && cy < m.h;
}
__device__ __forceinline__ int rd_drivable_at(const DevMap& m, int cx, int cy) {
  if (cx < 0 || cx >= m.w || cy < 0 || cy >= m.h) return 0;
  return (__ldg(m.bits + (size_t)cy * m.rw + (cx >> 5)) >> (cx & 31)) & 1u;
}

// ---- float64 helpers for the dynamics integrator (k_step): short, branch-free, no slow paths ----
// sin/cos on [-pi/4, pi/4] (fdlibm __kernel_sin / __kernel_cos minimax polynomials, < 1 ulp)
__device__ __forceinline__ void rd_sincos_kernel(double r, double& s, double& c) {
  const double z = r * r;
  double ps = fma(z, 1.58969099521155010221e-10, -2.50507602534068634195e-08);
  double pc = fma(z, -1.13596475577881948265e-11, 2.08757232129817482790e-09);
  ps = fma(z, ps, 2.75573137070700676789e-06);
  pc = fma(z, pc, -2.75573143513906633035e-07);
  ps = fma(z, ps, -1.98412698298579493134e-04);
  pc = fma(z, pc, 2.48015872894767294178e-05);
  ps = fma(z, ps, 8.33333333332248946124e-03);
  pc = fma(z, pc, -1.38888888888741095749e-03);
  ps = fma(z, ps, -1.66666666666666324348e-01);
  pc = fma(z, pc, 4.16666666666666019037e-02);
  s = fma(r * z, ps, r);
  c = fma(z * z, pc, fma(z, -0.5, 1.0));
}
// sincos for |x| < ~1e5 rad (three-term Cody-Waite reduction by pi/2, then the kernels; quadrant fix-up by selects).
// Larger arguments (a car that has spun thousands of times) take the library path.
__device__ __forceinline__ void rd_sincos(double x, double* sn, double* cs) {
  if (!(fabs(x) < 1.0e5)) { sincos(x, sn, cs); return; }
  const double k = rint(x * 6.36619772367581382433e-01);
  double r = fma(-k, 1.57079632679489655800e+00, x);
  r = fma(-k, 6.12323399573676603587e-17, r);
  r = fma(-k, -1.49738490485916983294e-33, r);
  double s, c;
  rd_sincos_kernel(r, s, c);
  const int q = (int)k;
  const double s1 = (q & 1) ? c : s, c1 = (q & 1) ? s : c;
  *sn = (q & 2) ? -s1 : s1;
  *cs = ((q + 1) & 2) ? -c1 : c1;
}
// 1/x for normal, finite x (speeds, cosines of small angles): hardware seed + three Newton steps, <= 1 ulp
__device__ __forceinline__ double rd_rcp(double x) {
  double y;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
  double e = fma(-x, y, 1.0);
  y = fma(y, e, y);
  e = fma(-x, y, 1.0);
  y = fma(y, e, y);
  e = fma(-x, y, 1.0);
  return fma(y, e, y);
}

// ---- mbarrier / bulk-copy (TMA, 1-D) wrappers ----
__device__ __forceinline__ uint32_t rd_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void rd_mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(rd_smem_u32(bar)), "r"(count));
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void rd_mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(rd_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void rd_bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   rd_smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(rd_smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void rd_mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(rd_smem_u32(bar)),
      "r"(parity)
      : "memory");
}
