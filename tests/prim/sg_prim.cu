// sg_prim.cu -- TEST INFRASTRUCTURE: the step kernel's small device primitives (narrowphase of sg_math.cuh, impedance,
// QCQP and friction solves of sg_kernels2.cuh) applied element by element to host arrays, so that tests/test_primitives.py
// can hold each one against the oracle's own primitive or a high-precision restatement at inputs chosen for their edges.
//
// One translation unit per precision, -DSGP_PREC=32 or 64, compiled two ways:
//   device:    nvcc with the product's NVCCFLAGS (and FASTFLAGS for fp32, as soft-grip_b200/csrc/Makefile builds the fp32
//              step kernel), so the fp32 entry points run the MUFU approximations of the product
//   emulator:  g++ -x c++ -DSG_SIMT_EMU -I tests/simt, the same source on the CPU (exact division and square root)
// Every entry point takes n elements of NI inputs and writes n elements of NO outputs (precision T unless stated), copies
// them to the device with cudaMemcpy, runs one kernel over the elements and copies the results back.  It returns 0, or
// the negated CUDA error code.  Nothing here is part of the product.
#include "sg_rt.hpp"
#include "sg_kernels2.cuh"

#include <vector>

#if SGP_PREC == 32
typedef float T;
#define SGP_FN(name) name##_f32
#elif SGP_PREC == 64
typedef double T;
#define SGP_FN(name) name##_f64
#else
#error "build with -DSGP_PREC=32 or -DSGP_PREC=64"
#endif

using namespace sg;

namespace {

struct Args { const T* in; T* out; int n; };

template <class P>
__global__ void prim_kernel(Args a) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < a.n; i += gridDim.x * blockDim.x) P::apply(a.in + P::NI * (size_t)i, a.out + P::NO * (size_t)i);
}

template <class P>
int run(const T* in, T* out, int n) {
  if (n <= 0) return 0;
  T *din = nullptr, *dout = nullptr;
  const size_t bi = sizeof(T) * P::NI * (size_t)n, bo = sizeof(T) * P::NO * (size_t)n;
  cudaError_t e = cudaMalloc((void**)&din, bi);
  if (e == cudaSuccess) e = cudaMalloc((void**)&dout, bo);
  if (e == cudaSuccess) e = cudaMemcpy(din, in, bi, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemset(dout, 0xff, bo);      // NaN pattern: an output the kernel never writes shows up
  if (e == cudaSuccess) {
    const int block = 64, grid = (int)((n + block - 1) / block < 1024 ? (n + block - 1) / block : 1024);
    Args a{din, dout, n};
    auto kp = prim_kernel<P>;
    SG_LAUNCH(kp, grid, block, 0, (cudaStream_t)0, a);
    e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
  }
  if (e == cudaSuccess) e = cudaMemcpy(out, dout, bo, cudaMemcpyDeviceToHost);
  if (din) cudaFree(din);
  if (dout) cudaFree(dout);
  return e == cudaSuccess ? 0 : -(int)e;
}

// in: spos[3] radius bpos[3] bmat[9] bsize[3]; out: n dist pos[3] nrm[3]
struct SphereBox {
  static constexpr int NI = 19, NO = 8;
  static __device__ void apply(const T* x, T* y) {
    RawCon<T> c{};
    const int n = sphere_box(c, x, x[3], x + 4, x + 7, x + 16);
    y[0] = T(n); y[1] = n ? c.dist : T(0);
    for (int k = 0; k < 3; k++) { y[2 + k] = n ? c.pos[k] : T(0); y[5 + k] = n ? c.nrm[k] : T(0); }
  }
};
// in: cpos[3] axis[3] radius halflength bpos[3] bmat[9] bsize[3]; out: n, then (dist pos[3] nrm[3]) per contact (2)
struct CapsuleBox {
  static constexpr int NI = 23, NO = 15;
  static __device__ void apply(const T* x, T* y) {
    RawCon<T> c[2] = {};
    const int n = capsule_box(c, x, x + 3, x[6], x[7], x + 8, x + 11, x + 20);
    y[0] = T(n);
    for (int i = 0; i < 2; i++) {
      y[1 + 7 * i] = i < n ? c[i].dist : T(0);
      for (int k = 0; k < 3; k++) { y[2 + 7 * i + k] = i < n ? c[i].pos[k] : T(0); y[5 + 7 * i + k] = i < n ? c[i].nrm[k] : T(0); }
    }
  }
};
// in: ppos[3] pmat[9] cpos[3] axis[3] radius halflength; out: n, then (dist pos[3] nrm[3] hint[3]) per contact (2)
struct PlaneCapsule {
  static constexpr int NI = 20, NO = 21;
  static __device__ void apply(const T* x, T* y) {
    RawCon<T> c[2] = {};
    const int n = plane_capsule(c, x, x + 3, x + 12, x + 15, x[18], x[19]);
    y[0] = T(n);
    for (int i = 0; i < 2; i++) {
      y[1 + 10 * i] = i < n ? c[i].dist : T(0);
      for (int k = 0; k < 3; k++) {
        y[2 + 10 * i + k] = i < n ? c[i].pos[k] : T(0); y[5 + 10 * i + k] = i < n ? c[i].nrm[k] : T(0); y[8 + 10 * i + k] = i < n ? c[i].hint[k] : T(0);
      }
    }
  }
};
// in: p1[3] R1[9] s1[3] p2[3] R2[9] s2[3]; out: overlap (0 / 1)
struct BoxBox {
  static constexpr int NI = 30, NO = 1;
  static __device__ void apply(const T* x, T* y) { y[0] = box_box_overlap(x, x + 3, x + 12, x + 15, x + 18, x + 27) ? T(1) : T(0); }
};
// in: normal[3] hint[3]; out: frame[9] (normal, tangent, binormal)
struct MakeFrame {
  static constexpr int NI = 6, NO = 9;
  static __device__ void apply(const T* x, T* y) {
    T f[9] = {x[0], x[1], x[2], x[3], x[4], x[5], 0, 0, 0};
    make_frame(f);
    for (int k = 0; k < 9; k++) y[k] = f[k];
  }
};
// in: si[7] (fill_si of a solimp) pos; out: impedance
struct Impedance {
  static constexpr int NI = 8, NO = 1;
  static __device__ void apply(const T* x, T* y) { y[0] = impedance2<T>(x, x[7]); }
};
#if SGP_PREC == 32
// in: a11n a12n kb bc1 bc2 frc f0 la (the arguments of friction_fast); out: f1 f2 la
struct FrictionFast {
  static constexpr int NI = 8, NO = 3;
  static __device__ void apply(const T* x, T* y) {
    float f1, f2, la = x[7];
    friction_fast(f1, f2, la, x[0], x[1], x[2], x[3], x[4], x[5], x[6]);
    y[0] = f1; y[1] = f2; y[2] = la;
  }
};
#else
// in: A11 A12 A22 b1 b2 d1 d2 r; out: res1 res2 active (the fp64 branch: MuJoCo's iteration)
struct Qcqp2 {
  static constexpr int NI = 8, NO = 3;
  static __device__ void apply(const T* x, T* y) {
    T res[2];
    const int active = qcqp2_fast<T>(res, x[0], x[1], x[2], x + 3, x[5], x[6], x[7]);
    y[0] = res[0]; y[1] = res[1]; y[2] = T(active);
  }
};
// in: A11 A12 A22 bc1 bc2 frc f0; out: f1 f2.  The fp64 branch of the step kernel's friction() (a member of its world struct,
// so restated here line for line): mju_QCQP2 through qcqp2_fast, then the rescaling onto the cone of mj_solPGS.
struct Friction {
  static constexpr int NI = 7, NO = 2;
  static __device__ void apply(const T* x, T* y) {
    const T A11 = x[0], A12 = x[1], A22 = x[2], frc = x[5], f0 = x[6];
    const T bc[2] = {x[3], x[4]};
    T vv[2];
    const int active = qcqp2_fast<T>(vv, A11, A12, A22, bc, frc, frc, f0);
    if (active) {
      const T ifr2 = tdiv(T(1), frc * frc);
      T s = vv[0] * vv[0] * ifr2 + vv[1] * vv[1] * ifr2;
      s = tsqrt(tdiv(f0 * f0, tmax(T(SG_MINVAL), s)));
      vv[0] *= s; vv[1] *= s;
    }
    y[0] = vv[0]; y[1] = vv[1];
  }
};
#endif

}  // namespace

extern "C" {
int SGP_FN(sgp_sphere_box)(const T* in, T* out, int n) { return run<SphereBox>(in, out, n); }
int SGP_FN(sgp_capsule_box)(const T* in, T* out, int n) { return run<CapsuleBox>(in, out, n); }
int SGP_FN(sgp_plane_capsule)(const T* in, T* out, int n) { return run<PlaneCapsule>(in, out, n); }
int SGP_FN(sgp_box_box_overlap)(const T* in, T* out, int n) { return run<BoxBox>(in, out, n); }
int SGP_FN(sgp_make_frame)(const T* in, T* out, int n) { return run<MakeFrame>(in, out, n); }
// solimp: n x 5 (double, as the model holds it), pos: n; the constants go through the host-side fill_si as in make_cst
int SGP_FN(sgp_impedance2)(const double* solimp, const T* pos, T* out, int n) {
  std::vector<T> in(8 * (size_t)(n > 0 ? n : 0));
  for (int i = 0; i < n; i++) { fill_si(&in[8 * (size_t)i], solimp + 5 * (size_t)i); in[8 * (size_t)i + 7] = pos[i]; }
  return run<Impedance>(in.data(), out, n);
}
#if SGP_PREC == 32
int sgp_friction_fast_f32(const T* in, T* out, int n) { return run<FrictionFast>(in, out, n); }
#else
int sgp_qcqp2_f64(const T* in, T* out, int n) { return run<Qcqp2>(in, out, n); }
int sgp_friction_f64(const T* in, T* out, int n) { return run<Friction>(in, out, n); }
#endif
}
