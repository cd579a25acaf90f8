// sg_traj.cuh -- kernels on the trajectory buffer [N][T][C] that the step kernel writes (the data format downstream of
// the hot path, SURVEY section 8 rows f1/f4): what the reference's trainer does to a dataset before it reaches a net.
//
//   sg_traj_noise_kernel     functions/optimization.py:6-14 `noised_modality`: accelerometer channels += N(0, 0.7),
//                            gyro channels += N(0, 0.06); optionally fused with the standardisation (x - mean) / std of
//                            functions/optimization.py:38.
//   sg_traj_stats_*_kernel   functions/utils.py:39-40: per-channel mean / standard deviation over axes (0, 1).
//
//   sg_traj_mask_kernel      create_dataset.py:43-44,57-58 `--mask-contact`: rows recorded without finger-object contact are
//                            zeroed, with the contact flag of manenv.py:65-83 in its intended and its literal meaning.
//
// The first two are streaming, HBM-bound passes (no reuse): 128-bit loads/stores of four consecutive channels per thread, grids
// sized as SM count x resident CTAs, grid-stride loops.  Algorithmic bytes: noise 2*s per element (read + write),
// stats s per element (read once), s = 4 (fp32) or 8 (fp64).
//
// Random numbers: Philox4x32-10 (Salmon et al., SC'11; the generator behind tf.random / curand / torch.cuda) keyed by the
// 64-bit seed, counter = index of the 4-element group (plus the caller's row offset when the buffer is a shard of a larger
// tensor), so a draw depends only on (seed, global element index): not on the grid, the sharding of worlds over GPUs or
// launches, or the batch precision.  Normals by Box-Muller in fp32 from the four words.
#pragma once
#include <stdint.h>

#include "sg_rt.hpp"

namespace sg {

struct Philox4 { uint32_t x, y, z, w; };

// ten rounds of Philox4x32 (multipliers 0xD2511F53 / 0xCD9E8D57, Weyl key increments 0x9E3779B9 / 0xBB67AE85)
__device__ __forceinline__ Philox4 philox4x32_10(Philox4 c, uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; r++) {
    const uint64_t p0 = (uint64_t)0xD2511F53u * c.x, p1 = (uint64_t)0xCD9E8D57u * c.z;
    Philox4 n;
    n.x = (uint32_t)(p1 >> 32) ^ c.y ^ k0;
    n.y = (uint32_t)p1;
    n.z = (uint32_t)(p0 >> 32) ^ c.w ^ k1;
    n.w = (uint32_t)p0;
    c = n;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  return c;
}

// uniform in (0, 1]: never 0, so the logarithm below is finite (x * 2^-32 is exact in fp32, so fma or mul+add agree)
__device__ __forceinline__ float u01(uint32_t x) { return (float)x * 2.3283064365386963e-10f + 1.1641532182693481e-10f; }

// two standard normals from two words: Box-Muller, z0 = r cos(2 pi ub), z1 = r sin(2 pi ub), r = sqrt(-2 ln ua).
// Default: the special-function unit, arranged so that the absolute error on z stays below 8e-6 for every input (typically
// 1e-6; the oracle evaluates the same formula in float64 from the same fp32 uniforms):
//   * ln ua by lg2.approx (relative error 2^-22 below 0.5, absolute 2^-22 above) except within 2^-5 of 1, where the relative
//     error of a logarithm near zero would blow up: there 1 - ua is exact in fp32 and -ln(1 - t) is its series to t^5
//     (truncation t^5 / 6 < 5e-9 relative);
//   * sqrt.approx (2^-23 relative);
//   * the angle is taken in (-pi, pi] (cos and sin of 2 pi u are minus those of 2 pi (u - 0.5), and u - 0.5 is exact above
//     0.25), where sin.approx / cos.approx are good to 2^-20.9 absolute.
// About 50 instructions per pair instead of ~170 with the FFMA polynomials of logf / sincospif: the kernel is bound by
// HBM instead of by issue slots (DESIGN.md 3b).  The host build (the SIMT emulator of the tests) keeps the libm formulas.
__device__ __forceinline__ void box_muller(uint32_t a, uint32_t b, float& z0, float& z1) {
#if !defined(__CUDA_ARCH__)
  const float r = sqrtf(-2.0f * logf(u01(a)));
  float s, c;
  sincospif(2.0f * u01(b), &s, &c);
  z0 = r * c;
  z1 = r * s;
#else
  const float ua = u01(a), t = 1.0f - ua;
  float lg, L, r, s, c;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(lg) : "f"(ua));
  L = -1.3862943611198906f * lg;                                       // -2 ln 2 * log2(ua)
  const float ser = 2.0f * t * fmaf(t, fmaf(t, fmaf(t, fmaf(t, 0.2f, 0.25f), 0.33333334f), 0.5f), 1.0f);
  L = t < 0.03125f ? ser : L;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(L));
  const float th = 6.2831853071795865f * (u01(b) - 0.5f);
  asm("sin.approx.ftz.f32 %0, %1;" : "=f"(s) : "f"(th));
  asm("cos.approx.ftz.f32 %0, %1;" : "=f"(c) : "f"(th));
  z0 = -r * c;
  z1 = -r * s;
#endif
}

template <typename T> struct Vec4 { T v[4]; };
__device__ __forceinline__ Vec4<float> load4(const float* p) { const float4 q = *(const float4*)p; return {{q.x, q.y, q.z, q.w}}; }
__device__ __forceinline__ Vec4<double> load4(const double* p) {
  const double2 a = *(const double2*)p, b = *(const double2*)(p + 2);
  return {{a.x, a.y, b.x, b.y}};
}
__device__ __forceinline__ void store4(float* p, const Vec4<float>& v) { float4 q; q.x = v.v[0]; q.y = v.v[1]; q.z = v.v[2]; q.w = v.v[3]; *(float4*)p = q; }
__device__ __forceinline__ void store4(double* p, const Vec4<double>& v) {
  double2 a, b; a.x = v.v[0]; a.y = v.v[1]; b.x = v.v[2]; b.y = v.v[3];
  *(double2*)p = a; *(double2*)(p + 2) = b;
}

template <typename T>
struct TrajNoiseArgs {
  const T* in;          // [nelem], 16-byte aligned; may alias out
  T* out;
  long long nelem;      // rows * nchan, nchan % 4 == 0
  int nchan, nacc;      // channels < nacc get sigma_acc, the others sigma_gyro
  float sigma_acc, sigma_gyro;
  uint32_t k0, k1;      // seed
  unsigned long long first_quad;   // counter of this buffer's first quad (a shard of a larger tensor continues its stream)
  const double* mean;   // [nchan] or null: fused (x - mean) / std after the noise
  const double* stdev;
};

// per-channel constants in shared memory (kernel prologue): sigma, and for the fused standardisation mean and 1 / std in the
// batch precision -- one 128-bit shared-memory load per table and quad instead of a compare + select per element, two
// fp64 loads, two conversions and a division per element
template <typename T>
__device__ __forceinline__ void traj_noise_quad(const TrajNoiseArgs<T>& A, const T* tabs, Vec4<T>& v, long long q, int g) {
  const unsigned long long ctr = A.first_quad + (unsigned long long)q;
  const Philox4 r = philox4x32_10(Philox4{(uint32_t)ctr, (uint32_t)(ctr >> 32), 0u, 0u}, A.k0, A.k1);
  float z[4];
  box_muller(r.x, r.y, z[0], z[1]);
  box_muller(r.z, r.w, z[2], z[3]);
  const int c0 = g * 4;
  const Vec4<T> sig = load4(tabs + c0);
#pragma unroll
  for (int j = 0; j < 4; j++) v.v[j] += sig.v[j] * (T)z[j];
  if (A.mean) {
    const Vec4<T> m = load4(tabs + A.nchan + c0), is = load4(tabs + 2 * A.nchan + c0);
#pragma unroll
    for (int j = 0; j < 4; j++) v.v[j] = (v.v[j] - m.v[j]) * is.v[j];
  }
}

// Two quads per thread and iteration, both loads issued before any arithmetic.  (Measured and dropped again,
// profiles/r02r_traj_bench.jsonl: issuing the NEXT iteration's loads before the arithmetic of the current one -- 0.69 of the
// roof in fp32 instead of 0.68, but 0.79 instead of 0.90 in fp64 -- and 8 instead of 6 resident CTAs per SM at 32 registers:
// 0.67.  The fp32 instance is bound by neither issue slots (62 %) nor HBM (55 %) alone: ~150 instructions per quad, a third
// of them 32-bit multiplies of the ten Philox rounds, leave the two streams imperfectly overlapped.)
template <typename T>
__global__ void __launch_bounds__(256) sg_traj_noise_kernel(const __grid_constant__ TrajNoiseArgs<T> A) {
  SG_SHARED_BYTES(smem_raw);
  T* tabs = (T*)smem_raw;                                // [3][nchan]: sigma | mean | 1 / std
  for (int c = threadIdx.x; c < A.nchan; c += blockDim.x) {
    tabs[c] = (T)(c < A.nacc ? A.sigma_acc : A.sigma_gyro);
    tabs[A.nchan + c] = A.mean ? (T)A.mean[c] : T(0);
    tabs[2 * A.nchan + c] = A.mean ? T(1) / (T)A.stdev[c] : T(1);
  }
  __syncthreads();
  const long long nquad = A.nelem >> 2, stride = (long long)gridDim.x * blockDim.x;
  const int qpr = A.nchan >> 2;
  const long long q0 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  int g = (int)(q0 % qpr);                               // channel group of q, carried along instead of a 64-bit modulo per quad
  const int gstep = (int)(stride % qpr);
  for (long long q = q0; q < nquad; q += 2 * stride) {
    const long long qb = q + stride;
    const bool hb = qb < nquad;
    Vec4<T> va = load4(A.in + 4 * q);
    Vec4<T> vb = va;
    if (hb) vb = load4(A.in + 4 * qb);
    int gb = g + gstep;
    if (gb >= qpr) gb -= qpr;
    traj_noise_quad(A, tabs, va, q, g);
    store4(A.out + 4 * q, va);
    if (hb) { traj_noise_quad(A, tabs, vb, qb, gb); store4(A.out + 4 * qb, vb); }
    g = gb + gstep;
    if (g >= qpr) g -= qpr;
  }
}

// ---- per-channel mean / std ---------------------------------------------------------------------------------------
// Pass 1: every thread owns one 4-channel group of the row (blockDim.x and therefore the grid stride are multiples of
// nchan / 4, so the group never changes) and accumulates sum and sum of squares of (x - x[row 0]) in fp64 -- the shift
// removes the cancellation of the one-pass variance.  The CTA's threads are then added per channel in thread order and
// the per-CTA partials are added in CTA order by pass 2: the result does not depend on scheduling.
constexpr int TRAJ_STATS_MAX_CHAN = 64;

template <typename T>
struct TrajStatsArgs {
  const T* in;          // [nrows][nchan], 16-byte aligned, nchan % 4 == 0
  long long nrows;
  int nchan;
  double* partial;      // [gridDim.x][2][nchan]
  double* mean;         // [nchan]  (pass 2)
  double* stdev;        // [nchan]
  int nblocks;          // gridDim.x of pass 1 (pass 2)
};

template <typename T>
__global__ void __launch_bounds__(512) sg_traj_stats_partial_kernel(const __grid_constant__ TrajStatsArgs<T> A) {
  SG_SHARED_BYTES(smem_raw);
  double* sh = (double*)smem_raw;                      // [8][blockDim.x]
  const int qpr = A.nchan >> 2, tid = threadIdx.x, nt = blockDim.x;
  const long long nquad = A.nrows * qpr, stride = (long long)gridDim.x * nt;
  const int g = tid % qpr;                             // this thread's channel group
  const Vec4<T> sv = load4(A.in + 4 * g);
  double s[4] = {0, 0, 0, 0}, ss[4] = {0, 0, 0, 0};
#pragma unroll 8
  for (long long q = (long long)blockIdx.x * nt + tid; q < nquad; q += stride) {
    const Vec4<T> v = load4(A.in + 4 * q);
#pragma unroll
    for (int j = 0; j < 4; j++) {
      const double d = (double)v.v[j] - (double)sv.v[j];
      s[j] += d;
      ss[j] = fma(d, d, ss[j]);
    }
  }
#pragma unroll
  for (int j = 0; j < 4; j++) { sh[j * nt + tid] = s[j]; sh[(4 + j) * nt + tid] = ss[j]; }
  __syncthreads();
  if (tid < 2 * A.nchan) {
    const int which = tid / A.nchan, c = tid % A.nchan, cg = c >> 2, j = c & 3;
    const double* col = sh + (which * 4 + j) * nt;
    double acc = 0;
    for (int u = cg; u < nt; u += qpr) acc += col[u];
    A.partial[((long long)blockIdx.x * 2 + which) * A.nchan + c] = acc;
  }
}

// Pass 2, one CTA: thread (r, col) adds the partials of the CTAs b = r, r + R, r + 2R, ... of column col = (sum | sum of
// squares, channel) in increasing b -- independent loads, so the L2 latency is paid once per thread and not once per
// partial as in a single serial loop -- and the R subset sums of a column are then added in the order r = 0 .. R-1.  The
// association is fixed by (nblocks, blockDim.x) alone: bit-reproducible.
constexpr int TRAJ_STATS_FINAL_THREADS = 1024;
template <typename T>
__global__ void __launch_bounds__(TRAJ_STATS_FINAL_THREADS) sg_traj_stats_final_kernel(const __grid_constant__ TrajStatsArgs<T> A) {
  SG_SHARED_BYTES(smem_raw);
  double* sh = (double*)smem_raw;                      // [R][2 * nchan]
  const int ncol = 2 * A.nchan, R = blockDim.x / ncol, tid = threadIdx.x;
  const int r = tid / ncol, col = tid - r * ncol;
  if (r < R) {
    double acc = 0;
#pragma unroll 4
    for (int b = r; b < A.nblocks; b += R) acc += A.partial[(long long)b * ncol + col];
    sh[r * ncol + col] = acc;
  }
  __syncthreads();
  if (tid < A.nchan) {
    const int c = tid;
    double s = 0, ss = 0;
    for (int q = 0; q < R; q++) { s += sh[q * ncol + c]; ss += sh[q * ncol + A.nchan + c]; }
    const double n = (double)A.nrows * 1.0, m = s / n;
    const double var = ss / n - m * m;
    A.mean[c] = (double)A.in[c] + m;
    A.stdev[c] = sqrt(var > 0 ? var : 0.0);
  }
}

// ---- --mask-contact -------------------------------------------------------------------------------------------------
// One warp per world: 32 rows' touch words per coalesced load, the keep flag per row, then the rows without contact are
// zeroed by 128-bit stores that cover the 32 rows contiguously (a kept row costs no trajectory traffic at all).
//   mode 0 "intended": keep a row iff every finger group touched an object geom during it: (touch & allf) == allf.
//   mode 1 "reference-literal" (SURVEY App. C item 2): get_sensor_sensordata removes the fingers it has seen from a
//     class-level list that is never refilled; while fingers are left the flag is "the list ran empty during this row",
//     afterwards it is "ncon >= 1".  Per world that is a prefix-OR over the rows (warp shuffle scan + carry), with the
//     fingers still left carried in and out through `fleft` so that consecutive episodes continue the list.
template <typename T>
struct TrajMaskArgs {
  T* traj;              // [nworlds][T][nchan], 16-byte aligned, nchan % 4 == 0
  const int* touch;     // [nworlds][T]: finger-group bits of the row's object contacts | anybit when ncon >= 1
  int nworlds, T_, nchan;
  int allf, anybit, mode;
  int* fleft;           // [nworlds] or null (mode 1): fingers not yet seen, in/out
};

template <typename T>
__global__ void __launch_bounds__(256) sg_traj_mask_kernel(const __grid_constant__ TrajMaskArgs<T> A) {
  const int lane = threadIdx.x & 31, wpb = blockDim.x >> 5, qpr = A.nchan >> 2;
  const unsigned FULL = 0xffffffffu;
  Vec4<T> zero;
  zero.v[0] = zero.v[1] = zero.v[2] = zero.v[3] = T(0);
  for (long long w = (long long)blockIdx.x * wpb + (threadIdx.x >> 5); w < A.nworlds; w += (long long)gridDim.x * wpb) {
    int seen = 0;                                        // finger bits seen before this chunk (mode 1)
    if (A.mode == 1 && A.fleft) seen = A.allf & ~A.fleft[w];
    for (int r0 = 0; r0 < A.T_; r0 += 32) {
      const bool in = r0 + lane < A.T_;
      const int tv = in ? A.touch[w * A.T_ + r0 + lane] : 0;
      bool keep;
      if (A.mode == 0) {
        keep = (tv & A.allf) == A.allf;
      } else {
        int inc = tv & A.allf;                           // inclusive prefix OR over the chunk's rows
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
          const int o = __shfl_sync(FULL, inc, (lane - d) & 31);
          if (lane >= d) inc |= o;
        }
        int exc = __shfl_sync(FULL, inc, (lane - 1) & 31);
        exc = (lane ? exc : 0) | seen;
        inc |= seen;
        keep = exc == A.allf ? (tv & A.anybit) != 0 : inc == A.allf;
        seen = __shfl_sync(FULL, inc, 31);
      }
      const int kept = (keep || !in) ? 1 : 0;
      T* base = A.traj + (w * A.T_ + r0) * A.nchan;
      for (int i = 0; i < qpr; i++) {
        const int lq = i * 32 + lane;
        if (!__shfl_sync(FULL, kept, lq / qpr)) store4(base + 4 * lq, zero);
      }
    }
    if (A.mode == 1 && A.fleft && lane == 0) A.fleft[w] = A.allf & ~seen;
  }
}

}  // namespace sg
