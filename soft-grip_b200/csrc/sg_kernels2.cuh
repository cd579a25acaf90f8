// sg_kernels2.cuh -- sm_100a device code of the batched soft-gripper simulator (sub-warp worlds).
//
// A warp is split into 32/LPW groups of LPW lanes; each group owns one world (LPW = 8: four worlds per
// warp).  The whole mj_step of a world (SURVEY.md section 3.2 / App. A; ref call site:
// environment/manenv.py:49 `self.env.step()`) runs without leaving the SM:
//
//   gripper()         finger-chain kinematics, inertia, bias, actuation, sensor pre-data   (1 lane / chain)
//   collide()         broadphase (lane / pair) -> candidates -> narrowphase (lane / candidate); contacts are
//                     emitted in MuJoCo's canonical order by ballot compaction, then scheduled per lane
//   rows_and_smooth() equality / tendon / limit rows (impedance, R, aref) and the smooth forces
//   warmstart()       forces from qacc_warmstart, dual cost test, qacc = qacc_smooth + M^-1 J^T f
//   pgs()             projected Gauss-Seidel in exact MuJoCo row order.  Equality rows are swept by a
//                     *list schedule* built on the host (sg_plan.hpp build_step_tables: rows of a step touch
//                     disjoint sliders, so lanes update them at once with the result of the sequential sweep);
//                     the dense volume-tendon row is a sub-warp shuffle reduction; limits and elliptic contact
//                     blocks run one lane per finger chain with the chain's accelerations in registers
//   finish()/euler()  accelerometers, implicit-damping Euler, NaN checks
//
// What the sweeps touch stays in shared memory ("hot": the running qacc, two words per equality row, finger
// inverse inertia).  The matrix AR = J M^-1 J^T + R is never formed.  Per equality row only u = R f - aref and
// n = -1 / (1/m1 + 1/m2 + R) are kept: the residual is J.qacc + u, and neither f nor R is needed (no clamp on
// equality rows).  Between the solve and the next rows_and_smooth() the row pairs are dead and serve gripper() and
// collide() as scratch.  Everything that is touched once per step ("aux": qpos, qvel, smooth forces, contact
// records) lives in an L2-resident global scratch slot of the group.
//
// No tensor-core math: nothing here is a dense contraction (largest dense objects: 4x4 finger inertia blocks,
// 3x3 contact blocks).  The kernel is bound by issue slots / dependent-issue latency of the Gauss-Seidel
// sweep; sub-warp worlds raise the useful lanes per issued instruction, small hot state raises resident warps.
// The tensor cores' memory is used, though (KArgs2::tm_cols, when every resident CTA of an SM gets its window): during
// the solve the (u, n) pairs live in tensor memory, one TMEM lane per thread (tcgen05.ld / st, see tm_ld2), and the
// shared-memory region they leave free holds a two-entry ring of contact records per lane, filled by cp.async one
// contact block ahead (chain_phase<RING>).  Without the window the pairs stay in shared memory and the records are read
// from the scratch; both paths compute the same bits (tests/test_simt.py, tests/test_gpu.py).
#pragma once
#include <stdint.h>

#include "../../include/softgrip.h"
#include "sg_plan.hpp"
#include "sg_math.cuh"

namespace sg {

// contact record: 32 words of T, 16-byte aligned groups
// Words 15, 26, 27 carry the tangential 2x2 block the way the friction solve wants it -- scaled by the friction coefficient and
// normalised by its trace (a22n = 1 - a11n), and the matching scale of the right-hand side -- so that none of it is redone
// in each of the 30 sweeps; kb = 0 marks a singular block (mju_QCQP2: zero friction).  R1 = R0 / impratio and the slider's
// 1 / m, which used to sit there, are a multiply resp. one shared-memory load away.
enum { CR_JG = 0 /*12*/, CR_NS = 12 /*3*/, CR_A12N = 15, CR_AREF = 16 /*3*/, CR_R0 = 19, CR_A = 20 /*6: 00 01 02 11 12 22*/,
       CR_A11N = 26, CR_KB = 27, CR_F = 28 /*3, then the friction multiplier*/, CR_STRIDE = 32 };

// per-world memory plan.  Offsets are in elements (T for the real arrays, int for the int arrays).
struct Layout2 {
  // hot, always shared memory
  int a;                 // nv (+ pad)
  int row2;              // 2*(nrow+1) : (u, R) per equality row, schedule order; the last pair is the dummy row (0, 1)
  int minv;              // 16*MAXCHAIN
  int hlim;              // 4*MAXFD : f, aref, R, sign per finger dof (meaningful where the limit is active)
  int h_impr;            // 1 (unused since team mode was removed; keeps the layout of the hot block)
  int hotT;
  int h_misc;            // 8 ints
  int hotI;
  // aux: global scratch
  int q, v, qs, jtf, a0; // nv each (qs: qacc_smooth; a0: qacc_warmstart at step entry, for the re-run after a divergence reset)
  int qv_in_smem, hq, hv; // unused, 0 (qpos / qvel in the hot region: a removed variant)
  int act, ctrl, actdot; // nu each
  int s_jv, s_ab, s_rot; // per sensor: 12, 3, 9
  int sens;              // nsd
  int crec;              // CR_STRIDE * maxcon
  int auxT;
  int i_con;             // maxcon : (chain+1) | (slider+1) << 4
  int i_tl;              // maxcon : time | lane << 16
  int i_order;           // maxcon : contact index | time << 8 | (slider + 1) << 16, segmented by lane
  int i_cand;            // (unused since the schedule's time slots moved to the shared-memory scratch)
  int i_lmask;           // MAXCHAIN : active-limit masks (bit jl: lower, bit 4+jl: upper)
  int auxI;
  int aux_in_smem;       // unused, 0 (aux in shared memory: a removed variant)
  // collision scratch: the (u, n) pairs of the equality rows are dead between the end of the solve and the next
  // rows_and_smooth(), so gripper() and collide() keep their per-step data there (offsets in T words from row2)
  int sc_cen;            // 3*ns : capsule centres
  int sc_gbox;           // 12 per moving box : geom position, rotation
  int sc_gaxis, sc_ganchor;  // 3*MAXFD each : world-frame joint axes / anchors of the finger chains
  int sc_cand;           // candidate list (ints): pair type | collider << 3 | second geom << 8
  int cand_cap;          // capacity of the candidate list (<= 0: the model does not fit the scratch)
  int smem_stride;       // bytes per world in shared memory (multiple of 16, bank-skewed)
  int smem_tables;       // bytes of the CTA-shared level-sweep step tables at the start of shared memory
  int gs_stride;         // bytes per world in the global scratch
};

enum { M2_NCON = 0, M2_STATUS = 1, M2_TOUCH = 2, M2_NCONTOT = 3, M2_ITERS = 4, M2_NCAND = 5, M2_TMAX = 6, M2_NLIM = 7, M2_DONE = 8,
       M2_LMASK = 9 /* MAXCHAIN entries */ };

template <typename T>
inline Layout2 make_layout2(const PlanDims& D, int wpw, int lpw) {
  Layout2 L{};
  int o = 0;
  auto take = [&](int n) { int r = o; o += (n + 3) & ~3; return r; };   // keep every array 16-byte aligned (float4 loads)
  auto pack = [&](int n) { int r = o; o += n; return r; };               // scalar-access arrays: no padding (shared memory is the
                                                                         // occupancy limit, every 16 bytes per world count)
  L.row2 = pack(2 * (D.nrow + 1));       // 2-vector loads; at offset 0 so that the sweep addresses the pairs off the world's base register
  o = (o + 3) & ~3;
  L.minv = take(16 * MAXCHAIN);          // 4-vector loads
  L.a = pack(D.nv + 1); L.hlim = pack(4 * MAXFD); L.h_impr = pack(1);
  o = (o + 1) & ~1;                      // the int block (and a double-precision aux block) stays 8-byte aligned
  L.hotT = o;
  L.h_misc = 0; L.hotI = 12;
  while ((sizeof(T) * (size_t)L.hotT + 4 * (size_t)L.hotI) % 16) L.hotI++;   // what follows (aux in shared memory) is 16-byte aligned
  o = 0;
  L.q = take(D.nv); L.v = take(D.nv); L.qs = take(D.nv); L.jtf = take(D.nv); L.a0 = take(D.nv);
  const int nu = D.nu > 0 ? D.nu : 1;
  L.act = take(nu); L.ctrl = take(nu); L.actdot = take(nu);
  L.s_jv = take(12 * MAXSENS); L.s_ab = take(3 * MAXSENS); L.s_rot = take(9 * MAXSENS); L.sens = take(D.nsd > 0 ? D.nsd : 1);
  L.crec = take(CR_STRIDE * D.maxcon);
  L.auxT = o;
  int io = 0;
  auto takei = [&](int n) { int r = io; io += (n + 3) & ~3; return r; };
  L.i_con = takei(D.maxcon); L.i_tl = takei(D.maxcon); L.i_order = takei(D.maxcon);
  L.i_cand = takei(D.ns); L.i_lmask = takei(MAXCHAIN);
  L.auxI = io;
  size_t hot = sizeof(T) * (size_t)L.hotT + sizeof(int) * (size_t)L.hotI;
  size_t aux = sizeof(T) * (size_t)L.auxT + sizeof(int) * (size_t)L.auxI;
  size_t sb = (hot + 15) & ~(size_t)15;
  // skew consecutive worlds of a warp by 32/wpw banks so that the same offset in different groups hits different banks
  if (wpw > 1) { const size_t unit = (size_t)(128 / wpw) < 16 ? 16 : (size_t)(128 / wpw); while ((sb / unit) % 2 == 0 || sb % unit) sb += 16; }
  L.smem_stride = (int)sb;
  L.gs_stride = (int)((aux + 127) & ~(size_t)127);
  {
    int so = 0;
    L.sc_cen = so; so += 3 * D.ns > D.ns + 32 ? 3 * D.ns : D.ns + 32;   // later reused for the contact schedule's time slots
    L.sc_gbox = so; so += 12 * MAXCHAIN * MAXCB;
    L.sc_gaxis = so; so += 3 * MAXFD;
    L.sc_ganchor = so; so += 3 * MAXFD;
    L.sc_cand = so;
    L.cand_cap = (2 * D.nrow - so) * (int)(sizeof(T) / sizeof(int));
    if (L.cand_cap > D.maxcand) L.cand_cap = D.maxcand;
  }
  // CTA-shared tables: step slots (8 bytes) | tendon coefficients, coefficient / mass, 1 / mass (ns each) | slider axes
  // (3 ns) | collider table | broadphase runs | row -> sliders
  L.smem_tables = (int)(((size_t)(D.nstep + 1) * lpw * 8 + (6 * (size_t)D.ns + (size_t)MAXCOLL * CO_STRIDE) * sizeof(T) +
                         (4 * (size_t)D.nrun + (size_t)D.nrow) * sizeof(int) + 127) & ~(size_t)127);
  return L;
}

// model constants in kernel precision
template <typename T>
struct Cst {
  T h, g[3], tol, impratio, inv_impratio, impr_scale;
  T eqj_K, eqj_B, eqj_si[7];
  T eqt_K, eqt_B, eqt_si[7], ten_iw, ten_k0, ten_d0, ten_lspring, ten_l0;
  T lim_K, lim_B, lim_si[7];
  T con_K, con_B, con_si[7], con_fr;
  T cap_r, cap_hl, sph_r, sph_pos[3], obj_pos[3];
  int cap_mask, sph_mask;
};

template <typename T>
inline void fill_si(T* o, const double* si) {
  for (int k = 0; k < 5; k++) o[k] = (T)si[k];
  o[5] = (T)(1.0 / std::pow(si[3], si[4] - 1.0));
  o[6] = (T)(1.0 / std::pow(1.0 - si[3], si[4] - 1.0));
}
template <typename T>
inline Cst<T> make_cst(const PlanDims& D) {
  Cst<T> C{};
  C.h = (T)D.h; for (int k = 0; k < 3; k++) { C.g[k] = (T)D.g[k]; C.sph_pos[k] = (T)D.sph_pos[k]; C.obj_pos[k] = (T)D.obj_pos[k]; }
  C.tol = (T)D.tol; C.impratio = (T)D.impratio; C.impr_scale = (T)D.impr_scale;
  C.inv_impratio = (T)(1.0 / (D.impratio > SG_MINVAL ? D.impratio : SG_MINVAL));
  C.eqj_K = (T)D.eqj_K; C.eqj_B = (T)D.eqj_B; fill_si(C.eqj_si, D.eqj_solimp);
  C.eqt_K = (T)D.eqt_K; C.eqt_B = (T)D.eqt_B; fill_si(C.eqt_si, D.eqt_solimp);
  C.ten_iw = (T)D.ten_iw; C.ten_k0 = (T)D.ten_k0; C.ten_d0 = (T)D.ten_d0; C.ten_lspring = (T)D.ten_lspring; C.ten_l0 = (T)D.ten_l0;
  C.lim_K = (T)D.lim_K; C.lim_B = (T)D.lim_B; fill_si(C.lim_si, D.lim_solimp);
  C.con_K = (T)D.con_K; C.con_B = (T)D.con_B; fill_si(C.con_si, D.con_solimp); C.con_fr = (T)D.con_fr;
  C.cap_r = (T)D.cap_r; C.cap_hl = (T)D.cap_hl; C.sph_r = (T)D.sph_r;
  C.cap_mask = (int)D.cap_mask; C.sph_mask = (int)D.sph_mask;
  return C;
}

template <typename T>
struct KArgs2 {
  PlanDims D;
  Cst<T> C;
  Layout2 L;
  const T* tab;
  const int* itab;
  int nworlds;
  int step_barrier;            // 1: the warps of a CTA start every physics step together (CTA barrier per step)
  int tm_cols;                 // tensor-memory columns the CTA allocates (power of two >= 32), 0: the (u, n) rows stay in shared memory
  int tm_stride;               // columns per warp: warp w owns [tm_stride (w / 4), +tm_stride) of its lane quarter
  int rec_ring;                // 1: contact records reach the chain phase through a two-entry shared-memory ring per lane (needs tm_cols)
  unsigned char* scratch;      // global aux slots [gridDim.x * WPW][L.gs_stride]
  int* batch_counter;          // persistent CTAs take their batches of worlds from this counter (zeroed before the launch);
                               // null: batch i of CTA c is i * gridDim.x + c
  // state, world-major
  T *qpos, *qvel, *warm, *act, *ctrl;
  const double *p_stiff, *p_damp, *p_tdamp, *p_objoff;
  int* status;
  T* sens_out;          // step: [W][nsd]; rollout: [W][nrows][nsd] (traj_soa = 0) or [nrows][nsd][W] (traj_soa = 1)
  int* touch_out;       // step: [W];      rollout: [W][nrows]
  int traj_soa;         // rollout only: 1 = structure-of-arrays trajectory, world index fastest
  int nsub, integrate;
  int rollout, sim_start, sim_step, nrows;
  const int* ctrl_event;
  const double* ctrl_value;
  int debug_world;
  double* debug_out;
  int debug_cap;
  // development aid (null in production): SM-clock cycles per phase summed over warps, [PH_COUNT] sums followed by
  // one time stamp per warp of the grid
  unsigned long long* prof;
};
enum { PH_GRIPPER = 0, PH_COLLIDE, PH_ROWS, PH_WARMSTART, PH_PGS_SETUP, PH_PGS_EQUALITY, PH_PGS_CHAIN, PH_SENSORS, PH_EULER, PH_OTHER,
       PH_COUNT = 16 };

// reciprocal used inside the sweeps: one MUFU on the fp32 fast path, an IEEE division in the verification build
template <typename T> __device__ __forceinline__ T trcp(T x);
template <> __device__ __forceinline__ double trcp<double>(double x) { return 1.0 / x; }
template <> __device__ __forceinline__ float trcp<float>(float x) {
#ifdef __CUDA_ARCH__
  float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r;
#else
  return 1.0f / x;
#endif
}

// Pins a loop-invariant pointer / value in registers: without it ptxas rebuilds such values from the kernel-parameter
// bank inside the contact loop (three constant loads plus 64-bit address arithmetic per record pointer, per block).
// (the OFFSET is pinned, not the pointer: a pointer that went through an asm statement loses its address space and every
// access through it becomes a generic load)
__device__ __forceinline__ long long keep_off(long long o) {
#if defined(__CUDA_ARCH__)
  asm volatile("" : "+l"(o));
#endif
  return o;
}
__device__ __forceinline__ int keep_off(int o) {
#if defined(__CUDA_ARCH__)
  asm volatile("" : "+r"(o));
#endif
  return o;
}
__device__ __forceinline__ float keep_val(float x) {
#if defined(__CUDA_ARCH__)
  asm volatile("" : "+f"(x));
#endif
  return x;
}
__device__ __forceinline__ double keep_val(double x) {
#if defined(__CUDA_ARCH__)
  asm volatile("" : "+d"(x));
#endif
  return x;
}

// one 128-byte contact record ahead into L1 (global scratch only)
__device__ __forceinline__ void prefetch_l1(const void* p) {
#ifdef __CUDA_ARCH__
  asm volatile("prefetch.global.L1 [%0];" ::"l"(p));
#else
  (void)p;
#endif
}
// ---- tensor memory as per-thread scratch --------------------------------------------------------------------------
// The kernel has no matrix work for the tensor cores, but their 256 KB of tensor memory per SM is the one on-chip store
// that shared memory (full) and the register file (full) leave unused.  In the 32x32b access shape every thread of a warp
// reads and writes its own TMEM lane (warp w of the CTA: lanes 32 (w % 4) ..), at a column address that is uniform over
// the warp -- which is exactly the access pattern of the equality sweep: every lane handles the row of ITS slot of step
// `st`, so the (u, n) pair of slot (st, lane) lives in the lane's TMEM lane at column 2 st (4 st in double precision).
// Measured with the sweep's load -> flops -> store -> warp-barrier pattern (scripts/tmem_probe.cu, 16 warps per SM):
// 50.6 cycles per step from tensor memory against 64.3 from shared memory, bit-identical results.
// The loads are asynchronous: the registers are only valid after tm_wait_ld, which takes them as operands so that the
// compiler cannot move a use above the wait.
template <typename T> struct TmPair;   // columns per (u, n) pair
template <> struct TmPair<float> { static constexpr int cols = 2; };
template <> struct TmPair<double> { static constexpr int cols = 4; };
#if defined(SG_SIMT_EMU)
// emulator: simt.h keeps a [128][512] word array per CTA and checks that the column address is uniform over the warp
__device__ __forceinline__ void tm_ld2(unsigned ta, float& x, float& y) { unsigned w[2]; simt_tm_ld(ta, 2, w); memcpy(&x, w, 4); memcpy(&y, w + 1, 4); }
__device__ __forceinline__ void tm_ld2(unsigned ta, double& x, double& y) { unsigned w[4]; simt_tm_ld(ta, 4, w); memcpy(&x, w, 8); memcpy(&y, w + 2, 8); }
__device__ __forceinline__ void tm_st1(unsigned ta, float x) { unsigned w[1]; memcpy(w, &x, 4); simt_tm_st(ta, 1, w); }
__device__ __forceinline__ void tm_st1(unsigned ta, double x) { unsigned w[2]; memcpy(w, &x, 8); simt_tm_st(ta, 2, w); }
__device__ __forceinline__ void tm_st2(unsigned ta, float x, float y) { unsigned w[2]; memcpy(w, &x, 4); memcpy(w + 1, &y, 4); simt_tm_st(ta, 2, w); }
__device__ __forceinline__ void tm_st2(unsigned ta, double x, double y) { unsigned w[4]; memcpy(w, &x, 8); memcpy(w + 2, &y, 8); simt_tm_st(ta, 4, w); }
template <typename T> __device__ __forceinline__ void tm_wait_ld(T&, T&) {}
__device__ __forceinline__ void tm_wait_st() {}
#elif defined(__CUDA_ARCH__)
__device__ __forceinline__ void tm_ld2(unsigned ta, float& x, float& y) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0, %1}, [%2];" : "=f"(x), "=f"(y) : "r"(ta));
}
__device__ __forceinline__ void tm_ld2(unsigned ta, double& x, double& y) {
  unsigned a, b, c, d;
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(a), "=r"(b), "=r"(c), "=r"(d) : "r"(ta));
  // (the words are only valid after tm_wait_ld: the wait below is part of the load for the two-register type)
  asm volatile("tcgen05.wait::ld.sync.aligned;" : "+r"(a), "+r"(b), "+r"(c), "+r"(d)::"memory");
  x = __hiloint2double((int)b, (int)a); y = __hiloint2double((int)d, (int)c);
}
__device__ __forceinline__ void tm_st1(unsigned ta, float x) { asm volatile("tcgen05.st.sync.aligned.32x32b.x1.b32 [%0], {%1};" ::"r"(ta), "f"(x)); }
__device__ __forceinline__ void tm_st1(unsigned ta, double x) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x2.b32 [%0], {%1, %2};" ::"r"(ta), "r"(__double2loint(x)), "r"(__double2hiint(x)));
}
__device__ __forceinline__ void tm_st2(unsigned ta, float x, float y) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x2.b32 [%0], {%1, %2};" ::"r"(ta), "f"(x), "f"(y));
}
__device__ __forceinline__ void tm_st2(unsigned ta, double x, double y) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};" ::"r"(ta), "r"(__double2loint(x)), "r"(__double2hiint(x)),
               "r"(__double2loint(y)), "r"(__double2hiint(y)));
}
__device__ __forceinline__ void tm_wait_ld(float& x, float& y) { asm volatile("tcgen05.wait::ld.sync.aligned;" : "+f"(x), "+f"(y)::"memory"); }
__device__ __forceinline__ void tm_wait_ld(double&, double&) {}     // waited inside tm_ld2<double>
__device__ __forceinline__ void tm_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
#else   // host pass of nvcc: never executed
template <typename T> __device__ __forceinline__ void tm_ld2(unsigned, T&, T&) {}
template <typename T> __device__ __forceinline__ void tm_st1(unsigned, T) {}
template <typename T> __device__ __forceinline__ void tm_st2(unsigned, T, T) {}
template <typename T> __device__ __forceinline__ void tm_wait_ld(T&, T&) {}
__device__ __forceinline__ void tm_wait_st() {}
#endif

// ---- the record ring of the chain phase ---------------------------------------------------------------------------
// cp_rec: asynchronous copy of one contact record (NB bytes, 16-byte pieces) from the global scratch into shared memory.
// No registers are held while the record is on its way from L2 (cp.async.cg: straight from L2, which is where the
// record's force words were last written); cp_wait: the lane's copies have landed.
// The ring is addressed through its 32-bit shared-window address, pinned in a register (see keep_off): with a generic
// pointer ptxas rebuilds the window base (S2UR CgaCtaId, ULEA ..) and the lane's offset in every block.  The explicit
// ld.shared statements are volatile, i.e. they stay behind the cp_wait that precedes them; every other access to the
// region is separated from them by a warp barrier.
__device__ __forceinline__ void cp_wait() {
#if defined(__CUDA_ARCH__)
  asm volatile("cp.async.wait_group 0;" ::: "memory");
#endif
}
#if defined(__CUDA_ARCH__)
typedef unsigned ring_t;
__device__ __forceinline__ ring_t ring_of(unsigned char* p) { return (unsigned)keep_off((int)__cvta_generic_to_shared(p)); }
template <int NB>
__device__ __forceinline__ void cp_rec(ring_t d, const unsigned char* src) {
#pragma unroll
  for (int i = 0; i < NB; i += 16) asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d + i), "l"(src + i) : "memory");
  asm volatile("cp.async.commit_group;" ::: "memory");
}
__device__ __forceinline__ void lds4(ring_t a, float* o) {
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(o[0]), "=f"(o[1]), "=f"(o[2]), "=f"(o[3]) : "r"(a));
}
__device__ __forceinline__ void lds4(ring_t a, double* o) {
  asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(o[0]), "=d"(o[1]) : "r"(a));
  asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(o[2]), "=d"(o[3]) : "r"(a + 16));
}
#else
typedef unsigned char* ring_t;
__device__ __forceinline__ ring_t ring_of(unsigned char* p) { return p; }
template <int NB> __device__ __forceinline__ void cp_rec(ring_t d, const unsigned char* src) { memcpy(d, src, NB); }
template <typename T> __device__ __forceinline__ void lds4(ring_t a, T* o) { memcpy(o, a, 4 * sizeof(T)); }
#endif
// division inside the contact blocks: MUFU.RCP + FMUL on the fp32 fast path (2 ulp), IEEE in the verification build
template <typename T> __device__ __forceinline__ T tdiv(T a, T b);
template <> __device__ __forceinline__ double tdiv<double>(double a, double b) { return a / b; }
template <> __device__ __forceinline__ float tdiv<float>(float a, float b) {
#ifdef __CUDA_ARCH__
  float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(b)); return a * r;   // one MUFU + one FMUL (no range scaling:
                                                                                  // every divisor here is guarded against tiny values)
#else
  return a / b;
#endif
}

// square root inside the contact blocks: MUFU.SQRT on the fp32 fast path, IEEE in the verification build
template <typename T> __device__ __forceinline__ T tfsqrt(T x);
template <> __device__ __forceinline__ double tfsqrt<double>(double x) { return sqrt(x); }
template <> __device__ __forceinline__ float tfsqrt<float>(float x) {
#ifdef __CUDA_ARCH__
  float r; asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r;
#else
  return sqrtf(x);
#endif
}

// mju_QCQP2: min 0.5 v'Av + b'v  s.t. |v| <= r  in the friction-scaled variables.
// Verification build (double): MuJoCo's own iteration (same algorithm as sg_math.cuh qcqp2) -- Newton on
// |v(la)|^2 - r^2 from la = 0, at most 20 steps, absolute thresholds 1e-10.
// Fast path (float): the same root of the same secular equation, found by Newton on 1/r - 1/|v(la)| (More-Sorensen:
// convex and nearly linear in la, so the iterates rise monotonically to the root and 2-3 steps reach float accuracy
// where MuJoCo's iteration needs 6-20), started from the lower bound |b|/r - trace(A) of the root when that is positive.
// MuJoCo's thresholds (1e-10 absolute) are below float resolution; the fast path stops at |v| - r <= 2e-6 r.  The
// caller rescales v onto the cone afterwards, as MuJoCo does.
template <typename T> __device__ __forceinline__ int qcqp2_fast(T* res, T A11i, T A12i, T A22i, const T* bin, T d0, T d1, T r) {
  T b1 = bin[0] * d0, b2 = bin[1] * d1;
  T A11 = A11i * d0 * d0, A22 = A22i * d1 * d1, A12 = A12i * d0 * d1;
  T la = 0, v1 = 0, v2 = 0;
  if (sizeof(T) == 4) {
    const T lb = tdiv(tfsqrt(b1 * b1 + b2 * b2), r) - (A11 + A22);
    if (lb > T(0)) la = lb;
    for (int iter = 0; iter < 8; iter++) {
      T det = (A11 + la) * (A22 + la) - A12 * A12;
      if (det < T(1e-10)) { res[0] = 0; res[1] = 0; return 0; }
      T detinv = tdiv(T(1), det), P11 = (A22 + la) * detinv, P22 = (A11 + la) * detinv, P12 = -A12 * detinv;
      v1 = -P11 * b1 - P12 * b2; v2 = -P12 * b1 - P22 * b2;
      const T n2 = v1 * v1 + v2 * v2, gap = tfsqrt(n2) - r;
      if (gap <= T(2e-6) * r) break;
      const T q = P11 * v1 * v1 + T(2) * P12 * v1 * v2 + P22 * v2 * v2;
      const T delta = tdiv(n2 * gap, q * r);
      if (!(delta > T(1e-10))) break;
      la += delta;
    }
    res[0] = v1 * d0; res[1] = v2 * d1;
    return la != T(0);
  }
  for (int iter = 0; iter < 20; iter++) {
    T det = (A11 + la) * (A22 + la) - A12 * A12;
    if (det < T(1e-10)) { res[0] = 0; res[1] = 0; return 0; }
    T detinv = tdiv(T(1), det), P11 = (A22 + la) * detinv, P22 = (A11 + la) * detinv, P12 = -A12 * detinv;
    v1 = -P11 * b1 - P12 * b2; v2 = -P12 * b1 - P22 * b2;
    T val = v1 * v1 + v2 * v2 - r * r;
    if (val < T(1e-10)) break;
    T deriv = T(-2) * (P11 * v1 * v1 + T(2) * P12 * v1 * v2 + P22 * v2 * v2);
    T delta = -tdiv(val, deriv);
    if (delta < T(1e-10)) break;
    la += delta;
  }
  res[0] = v1 * d0; res[1] = v2 * d1;
  return la != T(0);
}

// reciprocal square root for the fast friction update
__device__ __forceinline__ float trsqrt(float x) {
#ifdef __CUDA_ARCH__
  float r; asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r;
#else
  return 1.0f / sqrtf(x);
#endif
}

// Friction forces of one elliptic contact with the normal force f0 fixed (the QCQP of mj_solPGS followed by the
// rescaling onto the cone), fp32 fast path.  Same problem as qcqp2_fast + rescale, arranged for latency: the problem is
// normalised by trace(A); with w = adj(A + la) b, v = -w / det, every step needs |w|^2, det and w' adj w only, so its
// three special-function ops (1/det, sqrt |w|^2, 1/(Q r)) are independent of each other, and the final rescaling is one
// more reciprocal square root:  f = -w r / |w|  when the cone is active.
#if defined(SG_FRIC_STATS) && !defined(__CUDA_ARCH__)
static long sg_fric_evals = 0, sg_fric_calls = 0;     // development statistics under the emulator (Newton evaluations per call)
#endif
#if defined(SG_FRIC_DOMAIN) && !defined(__CUDA_ARCH__)
// development statistics under the emulator (scripts/dev_fric_domain.py): the range of friction_fast's arguments that the
// step kernel produces -- the domain tests/test_primitives.py asserts its error bounds on.  Per quantity: count, min, max
// and a histogram in quarter decades, written as one JSON line to $SG_FRIC_DOMAIN_OUT when the process exits.
struct FricDomain {
  enum { F0, BKF, COND, COND_INACTIVE, WARM, NQ, NBIN = 320 };     // bins: log10 from -40 to +40
  long n[NQ] = {}, hist[NQ][NBIN] = {};
  double lo[NQ], hi[NQ];
  long calls = 0, active = 0, kb0 = 0;
  FricDomain() { for (int q = 0; q < NQ; q++) { lo[q] = 1e300; hi[q] = -1e300; } }
  void add(int q, double x) {
    if (!(x > 0)) return;
    n[q]++; lo[q] = x < lo[q] ? x : lo[q]; hi[q] = x > hi[q] ? x : hi[q];
    int b = (int)std::floor(4.0 * (std::log10(x) + 40.0)); b = b < 0 ? 0 : b >= NBIN ? NBIN - 1 : b;
    hist[q][b]++;
  }
  void record(float a11, float a12, float kb, float bc0, float bc1, float f0, float la_in, float la_out) {
    calls++;
    if (kb == 0.0f) { kb0++; return; }
    const double a22 = 1.0 - (double)a11, tr = (double)a11 + a22, det = (double)a11 * a22 - (double)a12 * a12;
    const double disc = std::sqrt(std::fmax(0.0, 0.25 * tr * tr - det)), lmax = 0.5 * tr + disc, lmin = det / lmax;
    const double cond = lmin > 0 ? lmax / lmin : 1e300;
    add(F0, f0);
    add(BKF, std::sqrt((double)bc0 * bc0 + (double)bc1 * bc1) * kb / f0);
    add(COND, cond);
    if (la_out != 0.0f) { active++; if (la_in != 0.0f) add(WARM, (double)la_in / la_out); }   // warm start over the root it settled on
    else add(COND_INACTIVE, cond);
  }
  ~FricDomain() {
    const char* path = getenv("SG_FRIC_DOMAIN_OUT");
    FILE* f = path ? fopen(path, "a") : nullptr;
    if (!f) return;
    static const char* names[NQ] = {"f0", "bc_kb_over_f0", "cond", "cond_inactive", "warm_over_root"};
    fprintf(f, "{\"calls\": %ld, \"active\": %ld, \"singular\": %ld", calls, active, kb0);
    for (int q = 0; q < NQ; q++) {
      fprintf(f, ", \"%s\": {\"n\": %ld, \"min\": %.6g, \"max\": %.6g, \"hist_log10_quarter\": {", names[q], n[q], lo[q], hi[q]);
      bool first = true;
      for (int b = 0; b < NBIN; b++) if (hist[q][b]) { fprintf(f, "%s\"%.2f\": %ld", first ? "" : ", ", b / 4.0 - 40.0, hist[q][b]); first = false; }
      fprintf(f, "}}");
    }
    fprintf(f, "}\n");
    fclose(f);
  }
};
inline FricDomain sg_fric_domain;
#endif
__device__ __forceinline__ void friction_fast(float& f1, float& f2, float& la_io, float a11, float a12, float kb, float bc0, float bc1, float frc, float f0) {
#if defined(SG_FRIC_STATS) && !defined(__CUDA_ARCH__)
  sg_fric_calls++;
  if ((sg_fric_calls & 0x3ffff) == 0) fprintf(stderr, "friction_fast: %ld calls, %.3f evaluations per call\n", sg_fric_calls, (double)sg_fric_evals / (double)sg_fric_calls);
#endif
#if defined(SG_FRIC_DOMAIN) && !defined(__CUDA_ARCH__)
  // recorded on every return, with the multiplier the call settled on
  struct Rec { float* la; float a11, a12, kb, bc0, bc1, f0, la_in; ~Rec() { sg_fric_domain.record(a11, a12, kb, bc0, bc1, f0, la_in, *la); } }
      rec_{&la_io, a11, a12, kb, bc0, bc1, f0, la_io};
#endif
  // (a11, a12, 1 - a11) = frc^2 A_tt / trace and kb = frc / trace come ready-made from the contact record (contact_rows);
  // kb = 0 marks a singular block
  if (kb == 0.0f) { f1 = 0; f2 = 0; la_io = 0; return; }                  // mju_QCQP2: singular -> zero, inactive
  const float a22 = 1.0f - a11, b1 = bc0 * kb, b2 = bc1 * kb;
  const float rr = trcp<float>(f0);
  float lo = tfsqrt<float>(b1 * b1 + b2 * b2) * rr - 1.0f;               // lower bound |b|/r - trace of the root
  if (!(lo > 0.0f)) lo = 0.0f;
  // start from the root of the previous sweep (la_io, in the same normalised units; 0 on the first sweep) when it lies
  // above the bound: the problem changes little between sweeps, and a start to the right of the root costs one extra step
  // (the tangent of the convex function lands left of the root, from where the iterates rise monotonically)
  float la = fmaxf(lo, la_io);
  float w1 = 0, w2 = 0, rdet = 0, N2 = 0;
#pragma unroll 1
  for (int iter = 0; iter < 8; iter++) {                                  // a lower cap changes the results
#if defined(SG_FRIC_STATS) && !defined(__CUDA_ARCH__)
    sg_fric_evals++;
#endif
    const float c11 = a22 + la, c22 = a11 + la;
    const float det = c11 * c22 - a12 * a12;
    w1 = c11 * b1 - a12 * b2; w2 = c22 * b2 - a12 * b1;
    N2 = w1 * w1 + w2 * w2;
    const float Q = c11 * w1 * w1 - 2.0f * a12 * w1 * w2 + c22 * w2 * w2;
    rdet = trcp<float>(det);
    const float gap = tfsqrt<float>(N2) * rdet - f0;
    if (fabsf(gap) <= 2e-6f * f0) break;                 // on the cone
    if (gap < 0.0f && la <= lo) break;                   // inside the cone at the lowest admissible la (inactive when lo = 0)
    float nl = la + N2 * det * trcp<float>(Q * f0) * gap;
    if (!(nl > lo)) nl = lo;
    if (nl == la) break;
    la = nl;
  }
  const float s = la != 0.0f ? f0 * trsqrt(fmaxf(N2, 1e-30f)) : rdet;   // active: onto the cone; inactive: the free minimiser
  f1 = -w1 * s * frc; f2 = -w2 * s * frc;
  la_io = la;
}

template <typename T> __device__ __forceinline__ T powp(T x, T pw) { return pw == T(2) ? x * x : tpow(x, pw); }
// getimpedance with pre-sanitised solimp and host-precomputed 1/mid^(p-1), 1/(1-mid)^(p-1)  (SURVEY App. A1)
template <typename T> __device__ __forceinline__ T impedance2(const T* si, T pos) {
  const T d0 = si[0], d1 = si[1], w = si[2], mid = si[3], pw = si[4];
  if (d0 == d1 || w <= T(SG_MINVAL)) return T(0.5) * (d0 + d1);
  const T x = tabs(pos / w);
  if (x >= T(1)) return d1;
  if (x <= T(0)) return d0;
  T y;
  if (pw == T(1)) y = x;
  else if (x <= mid) y = powp(x, pw) * si[5];
  else y = T(1) - powp(T(1) - x, pw) * si[6];
  return d0 + y * (d1 - d0);
}

template <typename T> __device__ __forceinline__ void ld4(const T* p, T* o);
template <> __device__ __forceinline__ void ld4<float>(const float* p, float* o) {
  const float4 v = *reinterpret_cast<const float4*>(p); o[0] = v.x; o[1] = v.y; o[2] = v.z; o[3] = v.w;
}
template <> __device__ __forceinline__ void ld4<double>(const double* p, double* o) {
  const double2 v0 = *reinterpret_cast<const double2*>(p), v1 = *reinterpret_cast<const double2*>(p + 2);
  o[0] = v0.x; o[1] = v0.y; o[2] = v1.x; o[3] = v1.y;
}
template <typename T> __device__ __forceinline__ void st4(T* p, T a, T b, T c, T d);
template <> __device__ __forceinline__ void st4<float>(float* p, float a, float b, float c, float d) {
  float4 v; v.x = a; v.y = b; v.z = c; v.w = d; *reinterpret_cast<float4*>(p) = v;
}
template <> __device__ __forceinline__ void st4<double>(double* p, double a, double b, double c, double d) {
  double2 v0, v1; v0.x = a; v0.y = b; v1.x = c; v1.y = d; *reinterpret_cast<double2*>(p) = v0; *reinterpret_cast<double2*>(p + 2) = v1;
}
template <typename T> __device__ __forceinline__ void ld2(const T* p, T& x, T& y);
template <> __device__ __forceinline__ void ld2<float>(const float* p, float& x, float& y) { const float2 v = *reinterpret_cast<const float2*>(p); x = v.x; y = v.y; }
template <> __device__ __forceinline__ void ld2<double>(const double* p, double& x, double& y) { const double2 v = *reinterpret_cast<const double2*>(p); x = v.x; y = v.y; }

// four consecutive ints of a 16-byte aligned per-world int array (contact tables: one L2 round trip per four entries)
__device__ __forceinline__ void ldi4(const int* p, int* o) {
  const int4* q = reinterpret_cast<const int4*>(p);
  const int4 v = *q; o[0] = v.x; o[1] = v.y; o[2] = v.z; o[3] = v.w;
}
template <typename T> __device__ __forceinline__ void ldg2(const T* p, T& x, T& y);
template <> __device__ __forceinline__ void ldg2<float>(const float* p, float& x, float& y) { const float2 v = __ldg(reinterpret_cast<const float2*>(p)); x = v.x; y = v.y; }
template <> __device__ __forceinline__ void ldg2<double>(const double* p, double& x, double& y) { const double2 v = __ldg(reinterpret_cast<const double2*>(p)); x = v.x; y = v.y; }
static_assert(MAXCD == 4, "finger chain blocks are loaded as 4-vectors");

// one slot of the level-sweep step tables in shared memory (host encoding: sg_plan.hpp build_step_tables).  The shell is
// uniform (every slider has the same mass and tendon coefficient 1, as every MuJoCo composite has; checked by the host,
// sg_api.cu), so the slot is the 8-byte descriptor alone -- one 64-bit shared-memory load, two wavefronts per warp
template <typename T> struct alignas(8) Slot { unsigned x, y; };
template <typename T> __device__ __forceinline__ Slot<T> ld_slot(const Slot<T>* p) { return *p; }

// Once-per-step loops over the sliders / rows of a lane: ptxas does not move the global loads of iteration i + 1 above
// the stores (or the divergent arithmetic) of iteration i, so a plain loop pays one L2 round trip (~400 cycles at this
// occupancy) per iteration -- 41 of them in the row loop, 14 in every slider loop, ~140 per step, a tenth of a
// contact-free step.  batched() runs such a loop in two phases per NB elements: every load of the batch first (into a
// small struct per element, no stores in between), then the arithmetic and the stores.  Same operations per element, same
// element order: bit-identical results.
// (the lambdas are force-inlined: inside this very large kernel the inliner otherwise leaves some of them as calls, and
// their by-reference captures then live in local memory)
#define SG_INL __attribute__((always_inline))
template <int NB, typename V, typename LoadF, typename UseF>
__device__ __forceinline__ void batched(int first, int limit, int stride, LoadF load, UseF use) {
  for (int e0 = first; e0 < limit; e0 += stride * NB) {
    V v[NB];
#pragma unroll
    for (int b = 0; b < NB; b++) { const int e = e0 + b * stride; V x{}; if (e < limit) load(e, x); v[b] = x; }   // (always written: stays in registers)
#pragma unroll
    for (int b = 0; b < NB; b++) { const int e = e0 + b * stride; if (e < limit) use(e, v[b]); }
  }
}
template <typename T> struct V1 { T a; };
template <typename T> struct V2 { T a, b; };
template <typename T> struct V3 { T a, b, c; };
template <typename T> struct V5 { T a, b, c, d, e; };

// ---------------------------------------------------------------------------------------------
// the world
// ---------------------------------------------------------------------------------------------
template <typename T, int LPW>
struct World2 {
  static_assert(LPW >= MAXCHAIN && LPW <= 32 && (LPW & (LPW - 1)) == 0, "lanes per world: power of two, one lane per finger chain");
  static constexpr int WPW = 32 / LPW;
  static constexpr unsigned LOWMASK = LPW == 32 ? 0xffffffffu : ((1u << (LPW & 31)) - 1u);
  const KArgs2<T>& K;
  const PlanDims& D;
  const Cst<T>& C;
  const Layout2& L;
  T* hot; int* hoti; T* aux; int* auxi;
  int lane, grp, sl, gshift, w;
  bool valid;
  T kw, dw, tdw, off[3];

  unsigned char* smem_base;
  unsigned tm;            // this warp's tensor-memory window: lane quarter << 16 | first column (see tm_ld2)
  const Slot<T>* slots;  // CTA-shared step tables of the level sweep (shared memory), already offset to this lane
  const T *stc, *stciw;   // CTA-shared copies of the tendon coefficients and coefficient / mass
  const T* stim;          // CTA-shared 1 / slider mass
  const T* sax;           // CTA-shared slider axes (3 per slider)
  const T* scoll;         // CTA-shared collider table
  const int* sruns;       // CTA-shared broadphase runs
  const int* srd;         // CTA-shared row -> (first slider | second slider << 16, 0xffff: none), storage order
  __device__ __forceinline__ T stiw(int e) const { return stim[e]; }

  // vwarp / vnwarp: position of this warp's worlds in the CTA in units of WPW worlds (the real warp index, except
  // for the 2-lanes-per-world view that one warp of a team takes of the team's 16 worlds)
  __device__ World2(const KArgs2<T>& k, unsigned char* smem, int wid, bool ok, int vwarp = -1, int vnwarp = -1)
      : K(k), D(k.D), C(k.C), L(k.L), w(wid), valid(ok) {
    lane = threadIdx.x & 31; grp = lane / LPW; sl = lane % LPW; gshift = grp * LPW;
    const int warp = vwarp >= 0 ? vwarp : (int)(threadIdx.x >> 5), nwarp = vnwarp >= 0 ? vnwarp : (int)(blockDim.x >> 5);
    smem_base = smem;
    tm = 0;
    slots = reinterpret_cast<const Slot<T>*>(smem) + sl;
    stc = reinterpret_cast<const T*>(smem + (size_t)(D.nstep + 1) * LPW * sizeof(Slot<T>));
    stciw = stc + D.ns;
    stim = stciw + D.ns;
    sax = stim + D.ns;
    scoll = sax + 3 * D.ns;
    sruns = reinterpret_cast<const int*>(scoll + MAXCOLL * CO_STRIDE);
    srd = sruns + 4 * D.nrun;
    // storage slot of the group: consecutive slots sit LPW banks apart (Layout2::smem_stride); the two (or more) groups
    // of a half-warp take slots that are 16 banks apart, so that a 64-bit access of the whole warp to the same row pair
    // of every world is conflict-free as well
    const int gslot = WPW > 1 ? (grp % (WPW / 2)) * 2 + grp / (WPW / 2) : 0;
    unsigned char* base = smem + L.smem_tables + (size_t)(warp * WPW + gslot) * L.smem_stride;
    hot = reinterpret_cast<T*>(base);
    hoti = reinterpret_cast<int*>(hot + L.hotT);
    // the once-per-step data always lives in the global scratch (a shared-memory variant was measured slower and is gone:
    // with one possible address space the compiler emits global loads instead of generic ones)
    aux = reinterpret_cast<T*>(K.scratch + (((size_t)blockIdx.x * nwarp + warp) * WPW + gslot) * (size_t)L.gs_stride);
    auxi = reinterpret_cast<int*>(aux + L.auxT);
  }

  // loop-invariant base pointers pinned in registers (see keep_off): scratch-relative, table-relative, shared-memory-relative
  template <typename P> __device__ __forceinline__ P* pin_g(P* p) const {
    return reinterpret_cast<P*>(K.scratch + keep_off((long long)(reinterpret_cast<unsigned char*>(p) - K.scratch)));
  }
  __device__ __forceinline__ const T* pin_t(const T* p) const { return K.tab + keep_off((long long)(p - K.tab)); }
  template <typename P> __device__ __forceinline__ P* pin_s(P* p) const {
    return reinterpret_cast<P*>(smem_base + keep_off((int)(reinterpret_cast<unsigned char*>(p) - smem_base)));
  }
  __device__ __forceinline__ const T* tab(int o) const { return K.tab + o; }
  __device__ __forceinline__ const int* itab(int o) const { return K.itab + o; }
  __device__ __forceinline__ T* q() { return aux + L.q; }
  __device__ __forceinline__ T* v() { return aux + L.v; }
  __device__ __forceinline__ T* a() { return hot + L.a; }
  __device__ __forceinline__ T* qs() { return aux + L.qs; }
  __device__ __forceinline__ int& misc(int i) { return hoti[L.h_misc + i]; }
  __device__ __forceinline__ T* crec(int i) { return aux + L.crec + CR_STRIDE * i; }
  __device__ __forceinline__ T* scr(int o) { return hot + L.row2 + o; }     // collision scratch (see Layout2)
  __device__ __forceinline__ int* scand() { return reinterpret_cast<int*>(hot + L.row2 + L.sc_cand); }

  // phase clock (development aid): charges the cycles since the warp's previous tick to phase `ph`
  __device__ __forceinline__ void tick(int ph) {
#if defined(__CUDA_ARCH__)
    if (K.prof && lane == 0) {
      unsigned long long* stamp = K.prof + PH_COUNT + (size_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
      const unsigned long long t = clock64();
      atomicAdd(K.prof + ph, t - *stamp);
      *stamp = t;
    }
#else
    (void)ph;
#endif
  }

  // sub-warp collectives (every lane of the warp takes part; results are per group)
  __device__ __forceinline__ T gsum(T x) const {
#pragma unroll
    for (int o = LPW / 2; o > 0; o >>= 1) x += __shfl_xor_sync(FULLMASK, x, o);
    return x;
  }
  __device__ __forceinline__ int gmax(int x) const {
#pragma unroll
    for (int o = LPW / 2; o > 0; o >>= 1) { const int y = __shfl_xor_sync(FULLMASK, x, o); x = x > y ? x : y; }
    return x;
  }
  __device__ __forceinline__ int gor(int x) const {
#pragma unroll
    for (int o = LPW / 2; o > 0; o >>= 1) x |= __shfl_xor_sync(FULLMASK, x, o);
    return x;
  }
  __device__ __forceinline__ unsigned gballot(bool p) const { return (__ballot_sync(FULLMASK, p) >> gshift) & LOWMASK; }
  __device__ __forceinline__ int wmax(int x) const { return __reduce_max_sync(FULLMASK, x); }

  __device__ void load_params() {
    kw = K.p_stiff ? T(K.p_stiff[w]) : T(-1);
    dw = K.p_damp ? T(K.p_damp[w]) : T(-1);
    tdw = K.p_tdamp ? T(K.p_tdamp[w]) : T(-1);
#pragma unroll
    for (int k = 0; k < 3; k++) off[k] = C.obj_pos[k] + (K.p_objoff ? T(K.p_objoff[3 * (size_t)w + k]) : T(0));
  }
  __device__ __forceinline__ T stiffness(int e) const { return (kw >= T(0) && itab(D.io_kmask)[e]) ? kw : tab(D.o_sl_k0)[e]; }
  __device__ __forceinline__ T damping(int e) const { return dw >= T(0) ? dw : tab(D.o_sl_d0)[e]; }
  __device__ __forceinline__ T ten_stiffness() const { return (kw >= T(0) && D.stiff_tendon0) ? kw : C.ten_k0; }
  __device__ __forceinline__ T ten_damping() const { return tdw >= T(0) ? tdw : C.ten_d0; }

  // ------------------------------------------------------------------------------------------
  // finger chains: kinematics, inertia, bias, actuation, sensors (one lane per chain)
  // world-frame Jacobian formulation (independent of the oracle's com-based spatial algebra)
  // ------------------------------------------------------------------------------------------
  __device__ void gripper(int c) {
    const T* ch = tab(D.o_chain + c * CH_STRIDE);
    const int nd = D.ncd[c], nb = D.ncb[c], dof0 = D.chain_dof0[c];
    T P[3], R[9];
#pragma unroll
    for (int k = 0; k < 3; k++) P[k] = ch[CH_BASEPOS + k];
#pragma unroll
    for (int k = 0; k < 9; k++) R[k] = ch[CH_BASEROT + k];
    T axis[MAXCD][3], anch[MAXCD][3], bpos[MAXCB][3], brot[MAXCB][9], com[MAXCB][3], Iw[MAXCB][6], om[MAXCB][3];
    int nsup[MAXCB];
    int j = 0;
#pragma unroll
    for (int k = 0; k < MAXCB; k++) {
      if (k >= nb) break;
      const T* cb = ch + CH_BODY + k * CB_STRIDE;
      T pos[3], Rc[9], t[3];
      matvec3(t, R, cb + CB_POS);
#pragma unroll
      for (int i = 0; i < 3; i++) pos[i] = P[i] + t[i];
      matmul3(Rc, R, cb + CB_ROT);
#pragma unroll
      for (int jj = 0; jj < MAXCD; jj++) {
        if (jj != j || j >= nd) continue;
        const T* cd = ch + CH_DOF + j * CD_STRIDE;
        if ((int)cd[CD_BODY] != k) continue;
        matvec3(axis[j], Rc, cd + CD_AXIS);
        matvec3(t, Rc, cd + CD_JPOS);
#pragma unroll
        for (int i = 0; i < 3; i++) anch[j][i] = pos[i] + t[i];
        // Rodrigues rotation about the local axis by q
        T s, co; tsincos(q()[dof0 + j], &s, &co);
        const T ux = cd[CD_AXIS], uy = cd[CD_AXIS + 1], uz = cd[CD_AXIS + 2], oc = T(1) - co;
        T Rj[9] = {co + ux * ux * oc, ux * uy * oc - uz * s, ux * uz * oc + uy * s,
                   uy * ux * oc + uz * s, co + uy * uy * oc, uy * uz * oc - ux * s,
                   uz * ux * oc - uy * s, uz * uy * oc + ux * s, co + uz * uz * oc};
        matmul3(Rc, Rc, Rj);
        matvec3(t, Rc, cd + CD_JPOS);
#pragma unroll
        for (int i = 0; i < 3; i++) pos[i] = anch[j][i] - t[i];
        j++;
      }
      nsup[k] = j;
#pragma unroll
      for (int i = 0; i < 3; i++) { bpos[k][i] = pos[i]; P[i] = pos[i]; }
#pragma unroll
      for (int i = 0; i < 9; i++) { brot[k][i] = Rc[i]; R[i] = Rc[i]; }
      matvec3(t, Rc, cb + CB_IPOS);
#pragma unroll
      for (int i = 0; i < 3; i++) com[k][i] = pos[i] + t[i];
      T Ri[9]; matmul3(Ri, Rc, cb + CB_IROT);
      const T I0 = cb[CB_INERTIA], I1 = cb[CB_INERTIA + 1], I2 = cb[CB_INERTIA + 2];
      Iw[k][0] = Ri[0] * Ri[0] * I0 + Ri[1] * Ri[1] * I1 + Ri[2] * Ri[2] * I2;   // xx
      Iw[k][1] = Ri[3] * Ri[3] * I0 + Ri[4] * Ri[4] * I1 + Ri[5] * Ri[5] * I2;   // yy
      Iw[k][2] = Ri[6] * Ri[6] * I0 + Ri[7] * Ri[7] * I1 + Ri[8] * Ri[8] * I2;   // zz
      Iw[k][3] = Ri[0] * Ri[3] * I0 + Ri[1] * Ri[4] * I1 + Ri[2] * Ri[5] * I2;   // xy
      Iw[k][4] = Ri[0] * Ri[6] * I0 + Ri[1] * Ri[7] * I1 + Ri[2] * Ri[8] * I2;   // xz
      Iw[k][5] = Ri[3] * Ri[6] * I0 + Ri[4] * Ri[7] * I1 + Ri[5] * Ri[8] * I2;   // yz
      // box geom pose -> aux
      T* gb = scr(L.sc_gbox) + 12 * (c * MAXCB + k);
      matvec3(t, Rc, cb + CB_GPOS);
#pragma unroll
      for (int i = 0; i < 3; i++) gb[i] = pos[i] + t[i];
      T Rg[9]; matmul3(Rg, Rc, cb + CB_GROT);
#pragma unroll
      for (int i = 0; i < 9; i++) gb[3 + i] = Rg[i];
    }
#pragma unroll
    for (int jj = 0; jj < MAXCD; jj++) {
      if (jj >= nd) break;
#pragma unroll
      for (int i = 0; i < 3; i++) { scr(L.sc_gaxis)[3 * (dof0 + jj) + i] = axis[jj][i]; scr(L.sc_ganchor)[3 * (dof0 + jj) + i] = anch[jj][i]; }
    }
    // velocity-dependent terms
    T qv[MAXCD], da[MAXCD][3], va[MAXCD][3];
#pragma unroll
    for (int jj = 0; jj < MAXCD; jj++) qv[jj] = jj < nd ? v()[dof0 + jj] : T(0);
#pragma unroll
    for (int jj = 0; jj < MAXCD; jj++) {
      T wb[3] = {0, 0, 0};
      va[jj][0] = va[jj][1] = va[jj][2] = 0;
      if (jj < nd) {
#pragma unroll
        for (int i = 0; i < MAXCD; i++) {
          if (i >= jj) break;
          T r[3] = {anch[jj][0] - anch[i][0], anch[jj][1] - anch[i][1], anch[jj][2] - anch[i][2]}, t[3];
          cross3(t, axis[i], r);
#pragma unroll
          for (int k = 0; k < 3; k++) { wb[k] += axis[i][k] * qv[i]; va[jj][k] += t[k] * qv[i]; }
        }
        cross3(da[jj], wb, axis[jj]);
      } else { da[jj][0] = da[jj][1] = da[jj][2] = 0; }
    }
    auto point_terms = [&](const T* p, int ns_, T Jv[MAXCD][3], T* vp, T* ab) {
      vp[0] = vp[1] = vp[2] = 0; ab[0] = ab[1] = ab[2] = 0;
#pragma unroll
      for (int jj = 0; jj < MAXCD; jj++) {
        if (jj >= ns_) { Jv[jj][0] = Jv[jj][1] = Jv[jj][2] = 0; continue; }
        T r[3] = {p[0] - anch[jj][0], p[1] - anch[jj][1], p[2] - anch[jj][2]};
        cross3(Jv[jj], axis[jj], r);
#pragma unroll
        for (int k = 0; k < 3; k++) vp[k] += Jv[jj][k] * qv[jj];
      }
#pragma unroll
      for (int jj = 0; jj < MAXCD; jj++) {
        if (jj >= ns_) continue;
        T r[3] = {p[0] - anch[jj][0], p[1] - anch[jj][1], p[2] - anch[jj][2]}, t1[3], t2[3];
        T dv[3] = {vp[0] - va[jj][0], vp[1] - va[jj][1], vp[2] - va[jj][2]};
        cross3(t1, da[jj], r); cross3(t2, axis[jj], dv);
#pragma unroll
        for (int k = 0; k < 3; k++) ab[k] += (t1[k] + t2[k]) * qv[jj];
      }
    };
    T M[MAXCD][MAXCD], frc[MAXCD];
#pragma unroll
    for (int i = 0; i < MAXCD; i++) { frc[i] = 0;
#pragma unroll
      for (int jj = 0; jj < MAXCD; jj++) M[i][jj] = (i == jj && i >= nd) ? T(1) : T(0); }
    const T g[3] = {C.g[0], C.g[1], C.g[2]};
#pragma unroll
    for (int k = 0; k < MAXCB; k++) {
      if (k >= nb) break;
      const T* cb = ch + CH_BODY + k * CB_STRIDE;
      const T mass = cb[CB_MASS];
      T Jv[MAXCD][3], vc[3], ac[3], al[3] = {0, 0, 0};
      om[k][0] = om[k][1] = om[k][2] = 0;
      point_terms(com[k], nsup[k], Jv, vc, ac);
#pragma unroll
      for (int jj = 0; jj < MAXCD; jj++) {
        if (jj >= nsup[k]) break;
#pragma unroll
        for (int i = 0; i < 3; i++) { om[k][i] += axis[jj][i] * qv[jj]; al[i] += da[jj][i] * qv[jj]; }
      }
      auto Imul = [&](const T* x, T* y) {
        y[0] = Iw[k][0] * x[0] + Iw[k][3] * x[1] + Iw[k][4] * x[2];
        y[1] = Iw[k][3] * x[0] + Iw[k][1] * x[1] + Iw[k][5] * x[2];
        y[2] = Iw[k][4] * x[0] + Iw[k][5] * x[1] + Iw[k][2] * x[2];
      };
      T F[3] = {mass * (ac[0] - g[0]), mass * (ac[1] - g[1]), mass * (ac[2] - g[2])};
      T Ial[3], Iom[3], N[3];
      Imul(al, Ial); Imul(om[k], Iom); cross3(N, om[k], Iom);
#pragma unroll
      for (int i = 0; i < 3; i++) N[i] += Ial[i];
#pragma unroll
      for (int i = 0; i < MAXCD; i++) {
        if (i >= nsup[k]) break;
        frc[i] -= dot3(Jv[i], F) + dot3(axis[i], N);       // -qfrc_bias
        T Ia[3]; Imul(axis[i], Ia);
#pragma unroll
        for (int jj = 0; jj < MAXCD; jj++) {
          if (jj > i) break;
          T mij = mass * dot3(Jv[i], Jv[jj]) + dot3(axis[jj], Ia);
          M[i][jj] += mij;
          if (jj != i) M[jj][i] += mij;
        }
      }
    }
    // actuation through the chain's spatial tendon (cylinder: filter dynamics, force = gain*act)
    const T* ct = ch + CH_TEN;
    if (ct[CT_HAS] != T(0)) {
      const int kb = (int)ct[CT_BODY], u = (int)ct[CT_ACT];
      T s1[3], t[3], dir[3];
      matvec3(t, brot[kb], ct + CT_S1);
#pragma unroll
      for (int i = 0; i < 3; i++) { s1[i] = bpos[kb][i] + t[i]; dir[i] = s1[i] - ct[CT_S0 + i]; }
      normalize3(dir);
      if (u >= 0) {
        const T actv = aux[L.act + u], ctrlv = aux[L.ctrl + u];
        aux[L.actdot + u] = (ctrlv - actv) / tmax(T(SG_MINVAL), ct[CT_TIMECONST]);
        const T force = ct[CT_GAIN] * actv;
#pragma unroll
        for (int jj = 0; jj < MAXCD; jj++) {
          if (jj >= nsup[kb]) break;
          T r[3] = {s1[0] - anch[jj][0], s1[1] - anch[jj][1], s1[2] - anch[jj][2]}, jc[3];
          cross3(jc, axis[jj], r);
          frc[jj] += ct[CT_GEAR] * dot3(dir, jc) * force;
        }
      }
    }
    // M^-1 by Gauss-Jordan on the (padded) 4x4 SPD block
    T Mi[MAXCD][MAXCD];
#pragma unroll
    for (int i = 0; i < MAXCD; i++)
#pragma unroll
      for (int jj = 0; jj < MAXCD; jj++) Mi[i][jj] = i == jj ? T(1) : T(0);
#pragma unroll
    for (int p = 0; p < MAXCD; p++) {
      const T ip = T(1) / M[p][p];
#pragma unroll
      for (int jj = 0; jj < MAXCD; jj++) { M[p][jj] *= ip; Mi[p][jj] *= ip; }
#pragma unroll
      for (int i = 0; i < MAXCD; i++) {
        if (i == p) continue;
        const T f = M[i][p];
#pragma unroll
        for (int jj = 0; jj < MAXCD; jj++) { M[i][jj] -= f * M[p][jj]; Mi[i][jj] -= f * Mi[p][jj]; }
      }
    }
#pragma unroll
    for (int i = 0; i < MAXCD; i++) {
      T s = 0;
#pragma unroll
      for (int jj = 0; jj < MAXCD; jj++) { hot[L.minv + 16 * c + 4 * i + jj] = Mi[i][jj]; s += Mi[i][jj] * frc[jj]; }
      if (i < nd) qs()[dof0 + i] = s;
    }
    // sensors on this chain (gyro now; accelerometer pre-data, finished after the solve)
    for (int s = 0; s < D.nsens; s++) {
      const T* se = tab(D.o_sens + s * SE_STRIDE);
      if ((int)se[SE_CHAIN] != c) continue;
      const int k = (int)se[SE_BODY], adr = (int)se[SE_ADR];
      T Rs[9]; matmul3(Rs, brot[k], se + SE_ROT);
      if ((int)se[SE_TYPE] == SENS_GYRO) {
        T o[3]; matTvec3(o, Rs, om[k]);
#pragma unroll
        for (int i = 0; i < 3; i++) aux[L.sens + adr + i] = o[i];
      } else {
        T p[3], t[3], Jv[MAXCD][3], vp[3], ab[3];
        matvec3(t, brot[k], se + SE_POS);
#pragma unroll
        for (int i = 0; i < 3; i++) p[i] = bpos[k][i] + t[i];
        point_terms(p, nsup[k], Jv, vp, ab);
#pragma unroll
        for (int jj = 0; jj < MAXCD; jj++)
#pragma unroll
          for (int i = 0; i < 3; i++) aux[L.s_jv + 12 * s + 3 * jj + i] = Jv[jj][i];
#pragma unroll
        for (int i = 0; i < 3; i++) aux[L.s_ab + 3 * s + i] = ab[i] - g[i];
#pragma unroll
        for (int i = 0; i < 9; i++) aux[L.s_rot + 9 * s + i] = Rs[i];
      }
    }
  }

  // ------------------------------------------------------------------------------------------
  // collision + contact rows
  // ------------------------------------------------------------------------------------------
  __device__ __forceinline__ void capsule_center(int e, T* c) {
    const T* ce = scr(L.sc_cen) + 3 * e;
#pragma unroll
    for (int k = 0; k < 3; k++) c[k] = ce[k];
  }
  __device__ __forceinline__ void collider_pose(int ci, T* pos, T* rot) {
    const T* co = scoll + ci * CO_STRIDE;
    const int c = (int)co[CO_CHAIN];
    if (c < 0) {
#pragma unroll
      for (int k = 0; k < 3; k++) pos[k] = co[CO_POS + k];
#pragma unroll
      for (int k = 0; k < 9; k++) rot[k] = co[CO_ROT + k];
    } else {
      const T* gb = scr(L.sc_gbox) + 12 * (c * MAXCB + (int)co[CO_BODY]);
#pragma unroll
      for (int k = 0; k < 3; k++) pos[k] = gb[k];
#pragma unroll
      for (int k = 0; k < 9; k++) rot[k] = gb[3 + k];
    }
  }

  // builds the three rows of one contact into record `slot` (mj_instantiateContact + mj_makeImpedance +
  // mj_referenceConstraint + the diagonal block of efc_AR)
  __device__ void contact_rows(int slot, const RawCon<T>& rc, int ci, int e, T slider_sign, bool dbg, int dbg_index) {
    const T* co = scoll + ci * CO_STRIDE;
    const int c = (int)co[CO_CHAIN];
    T fr[9];
#pragma unroll
    for (int k = 0; k < 3; k++) { fr[k] = rc.nrm[k]; fr[3 + k] = rc.hint[k]; }
    make_frame(fr);
    T Jg[3][MAXCD];
    T* cr = crec(slot);
    int nsupp = 0, dof0 = 0;
    if (c >= 0) {
      dof0 = D.chain_dof0[c];
      const T* ch = tab(D.o_chain + c * CH_STRIDE);
      const int kb = (int)co[CO_BODY];
      for (int jj = 0; jj < D.ncd[c]; jj++) if ((int)ch[CH_DOF + jj * CD_STRIDE + CD_BODY] <= kb) nsupp = jj + 1;
    }
#pragma unroll
    for (int jj = 0; jj < MAXCD; jj++) {
      T col[3] = {0, 0, 0};
      if (jj < nsupp) {
        const T* ax = scr(L.sc_gaxis) + 3 * (dof0 + jj); const T* an = scr(L.sc_ganchor) + 3 * (dof0 + jj);
        T r[3] = {rc.pos[0] - an[0], rc.pos[1] - an[1], rc.pos[2] - an[2]};
        cross3(col, ax, r);
      }
#pragma unroll
      for (int r = 0; r < 3; r++) { Jg[r][jj] = dot3(fr + 3 * r, col); cr[CR_JG + 4 * r + jj] = Jg[r][jj]; }
    }
    T ns[3] = {0, 0, 0}, iw_e = 0, biw = co[CO_BIW], ve = 0;
    if (e >= 0) {
      const T* ax = sax + 3 * e;
#pragma unroll
      for (int r = 0; r < 3; r++) ns[r] = slider_sign * dot3(fr + 3 * r, ax);
      iw_e = stiw(e);
      biw += tab(D.o_sl_biw)[e];
      ve = v()[D.nfd + e];
    }
#pragma unroll
    for (int r = 0; r < 3; r++) cr[CR_NS + r] = ns[r];
    cr[CR_F + 3] = 0;                                         // word 31: friction multiplier of the previous sweep
    const T imp = impedance2<T>(C.con_si, rc.dist);
    const T R0 = tmax(T(SG_MINVAL), (T(1) - imp) * biw / imp);
    const T R1 = R0 * C.inv_impratio;
    cr[CR_R0] = R0;
    // velocity, aref
    T vel[3];
#pragma unroll
    for (int r = 0; r < 3; r++) {
      T s = ns[r] * ve;
#pragma unroll
      for (int jj = 0; jj < MAXCD; jj++) if (jj < nsupp) s += Jg[r][jj] * v()[dof0 + jj];
      vel[r] = s;
    }
    cr[CR_AREF] = -C.con_B * vel[0] - C.con_K * imp * rc.dist;
    cr[CR_AREF + 1] = -C.con_B * vel[1];
    cr[CR_AREF + 2] = -C.con_B * vel[2];
    // A = Jg Minv Jg' + ns ns'/m + diag(R)
    T MJ[3][MAXCD];
#pragma unroll
    for (int r = 0; r < 3; r++)
#pragma unroll
      for (int i = 0; i < MAXCD; i++) {
        T s = 0;
        if (c >= 0) {
#pragma unroll
          for (int jj = 0; jj < MAXCD; jj++) s += hot[L.minv + 16 * c + 4 * i + jj] * Jg[r][jj];
        }
        MJ[r][i] = s;
      }
    int idx = 0;
    T Ab[6];
#pragma unroll
    for (int r = 0; r < 3; r++)
#pragma unroll
      for (int s2 = r; s2 < 3; s2++) {
        T s = ns[r] * ns[s2] * iw_e;
#pragma unroll
        for (int jj = 0; jj < MAXCD; jj++) s += Jg[r][jj] * MJ[s2][jj];
        if (r == s2) s += (r == 0 ? R0 : R1);
        Ab[idx] = s;
        cr[CR_A + idx++] = s;    // order: 00 01 02 11 12 22
      }
    {
      // the friction block of the fast path's solve: (frc^2 A_tt) / trace and frc / trace (see friction_fast)
      const T d2 = C.con_fr * C.con_fr, a11 = Ab[3] * d2, a12 = Ab[4] * d2, a22 = Ab[5] * d2;
      T a11n = T(0.5), a12n = 0, kb = 0;
      if (!(a11 * a22 - a12 * a12 < T(1e-10))) { const T sc = T(1) / (a11 + a22); a11n = a11 * sc; a12n = a12 * sc; kb = C.con_fr * sc; }
      cr[CR_A11N] = a11n; cr[CR_A12N] = a12n; cr[CR_KB] = kb;
    }
    auxi[L.i_con + slot] = (c + 1) | ((e + 1) << 4);
    if (dbg && K.debug_out) {
      double* o = K.debug_out + 64 + 16 * (size_t)dbg_index;   // dist, pos3, frame9
      if (64 + 16 * (dbg_index + 1) <= K.debug_cap) {
        o[0] = (double)rc.dist;
        for (int k = 0; k < 3; k++) o[1 + k] = (double)rc.pos[k];
        for (int k = 0; k < 9; k++) o[4 + k] = (double)fr[k];
      }
    }
  }

  __device__ void collide() {
    const bool dbg = valid && (w == K.debug_world);
    // ---- capsule centres into the scratch (the sliders only move along their axes) ----
    T blo[3] = {T(SG_MAXVAL), T(SG_MAXVAL), T(SG_MAXVAL)}, bhi[3] = {-T(SG_MAXVAL), -T(SG_MAXVAL), -T(SG_MAXVAL)};
    {
      const T* __restrict__ qsl = pin_g(q() + D.nfd);
      const T* __restrict__ c0 = pin_t(tab(D.o_sl_cap0));
      T* cen = scr(L.sc_cen);
      struct CenV { T q, c[3]; };
      batched<8, CenV>(sl, D.ns, LPW,
        [&](int e, CenV& x) SG_INL { x.q = qsl[e]; x.c[0] = c0[3 * e]; x.c[1] = c0[3 * e + 1]; x.c[2] = c0[3 * e + 2]; },
        [&](int e, const CenV& x) SG_INL {
#pragma unroll
          for (int k = 0; k < 3; k++) {
            const T ck = off[k] + x.c[k] + sax[3 * e + k] * x.q;
            cen[3 * e + k] = ck;
            blo[k] = ck < blo[k] ? ck : blo[k]; bhi[k] = ck > bhi[k] ? ck : bhi[k];     // a NaN centre leaves the bounds alone
            if (!(ck == ck)) { blo[k] = -T(SG_MAXVAL); bhi[k] = T(SG_MAXVAL); }          // ... so it opens them explicitly
          }
        });
      // bounding box of the capsule centres of this world (sub-warp min / max)
#pragma unroll
      for (int k = 0; k < 3; k++)
#pragma unroll
        for (int o = LPW / 2; o > 0; o >>= 1) {
          const T l2 = __shfl_xor_sync(FULLMASK, blo[k], o), h2 = __shfl_xor_sync(FULLMASK, bhi[k], o);
          blo[k] = l2 < blo[k] ? l2 : blo[k]; bhi[k] = h2 > bhi[k] ? h2 : bhi[k];
        }
      __syncwarp();
    }
    // ---- broadphase: bounding spheres, candidates compacted in pair order.  The pair list is walked by runs
    // {type, collider a, first b, count}: the collider is fetched once per run, everything else is in shared memory ----
    int ncand = 0, flags = 0;
    int* cand = scand();
    const int cand_cap = L.cand_cap;
    for (int run = 0; run < D.nrun; run++) {
      const int pt = sruns[4 * run], a0 = sruns[4 * run + 1] & 255, na = sruns[4 * run + 1] >> 8, b0 = sruns[4 * run + 2];
      const int total = na * sruns[4 * run + 3];
      const bool one = na == 1;                      // one collider against a range of second geoms: fetched once
      int pa = a0;
      const T* co = scoll + pa * CO_STRIDE;
      T c1[3], rot1[9];
      if (pt == PAIR_PLANE_CAPSULE || pt == PAIR_BOX_CAPSULE) {
        // Can any capsule of the shell pass the bounding-sphere test against a collider of this run?  The test below is
        // |centre - c1|^2 <= (rb1 + rb2)^2 (plane: signed distance <= rb2); every centre lies in [blo, bhi], so a collider
        // whose distance to that box exceeds the bound (with a relative margin for rounding) rejects every pair of the run.
        bool reach = false;
        const T rb2 = C.cap_r + C.cap_hl;
        for (int i = 0; i < na; i++) {
          const T* ci = scoll + (a0 + i) * CO_STRIDE;
          T cc[3], rr[9];
          collider_pose(a0 + i, cc, rr);
          if ((int)ci[CO_TYPE] == GEOM_PLANE) {
            T dmin = 0;
#pragma unroll
            for (int k = 0; k < 3; k++) { const T n = rr[3 * k + 2], a = n * (blo[k] - cc[k]), b = n * (bhi[k] - cc[k]); dmin += a < b ? a : b; }
            if (!(dmin > rb2 + T(1e-4) * (tabs(dmin) + rb2))) reach = true;
          } else {
            T d2 = 0;
#pragma unroll
            for (int k = 0; k < 3; k++) { const T x = cc[k] < blo[k] ? blo[k] - cc[k] : (cc[k] > bhi[k] ? cc[k] - bhi[k] : T(0)); d2 += x * x; }
            const T bound = ci[CO_RBOUND] + rb2;
            if (!(d2 > bound * bound * T(1.0001))) reach = true;
          }
        }
        // the loop below is full of warp collectives (the worlds of a warp ballot together): warp-uniform decision
        if (!__any_sync(FULLMASK, reach)) continue;
      }
      if (one) collider_pose(pa, c1, rot1);
      if (one && (pt == PAIR_PLANE_CAPSULE || pt == PAIR_BOX_CAPSULE)) {
        // one collider against a range of capsules (nearly every pair of the list): everything that does not depend on
        // the capsule is hoisted out of the chunk loop -- the same tests in the same order, a third of the instructions
        const bool plane = pt == PAIR_PLANE_CAPSULE;
        const T rb2 = C.cap_r + C.cap_hl;
        const T bound = co[CO_RBOUND] + rb2, bound2 = bound * bound;
        const T nrm[3] = {rot1[2], rot1[5], rot1[8]};
        const T hs[3] = {co[CO_SIZE] + C.cap_r, co[CO_SIZE + 1] + C.cap_r, co[CO_SIZE + 2] + C.cap_r};
        const T* cen = scr(L.sc_cen);
        for (int base = 0; base < total; base += LPW) {
          const int j = base + sl, pb = b0 + j;
          bool pass = false;
          if (j < total) {
            const T dif[3] = {cen[3 * pb] - c1[0], cen[3 * pb + 1] - c1[1], cen[3 * pb + 2] - c1[2]};
            if (plane) pass = !(dot3(dif, nrm) > rb2);
            else {
              pass = !(dot3(dif, dif) > bound2);
              if (pass) {
                // mid-phase (prunes only): the capsule's bounding box in the frame of the box must overlap the box
                T dl[3], al[3];
                matTvec3(dl, rot1, dif);
                matTvec3(al, rot1, sax + 3 * pb);
#pragma unroll
                for (int k = 0; k < 3; k++) if (tabs(dl[k]) > hs[k] + C.cap_hl * tabs(al[k])) pass = false;
              }
            }
          }
          const unsigned m = gballot(pass);
          if (pass) {
            const int slot = ncand + __popc(m & ((1u << sl) - 1));
            if (slot < cand_cap) cand[slot] = pt | (pa << 3) | (pb << 8); else flags |= SG_ST_CON_FULL;
          }
          ncand += __popc(m);
        }
        continue;
      }
      for (int base = 0; base < total; base += LPW) {
        const int j = base + sl;
        int pb = b0 + j;
        bool pass = false;
        if (j < total) {
          if (!one) { const int jb = j / na; pa = a0 + (j - jb * na); pb = b0 + jb; co = scoll + pa * CO_STRIDE; collider_pose(pa, c1, rot1); }
          const bool plane = (int)co[CO_TYPE] == GEOM_PLANE;
          const T rb1 = co[CO_RBOUND];
          T c2[3], rb2;
          if (pt == PAIR_PLANE_CAPSULE || pt == PAIR_BOX_CAPSULE) { capsule_center(pb, c2); rb2 = C.cap_r + C.cap_hl; }
          else if (pt == PAIR_SPHERE_BOX) {
#pragma unroll
            for (int k = 0; k < 3; k++) c2[k] = off[k] + C.sph_pos[k];
            rb2 = C.sph_r;
          } else { T rot[9]; collider_pose(pb, c2, rot); rb2 = scoll[pb * CO_STRIDE + CO_RBOUND]; }
          T dif[3] = {c2[0] - c1[0], c2[1] - c1[1], c2[2] - c1[2]};
          if (plane) { T nrm[3] = {rot1[2], rot1[5], rot1[8]}; pass = !(dot3(dif, nrm) > rb2); }
          else { T bound = rb1 + rb2; pass = !(dot3(dif, dif) > bound * bound); }
          if (pass && pt == PAIR_BOX_CAPSULE) {
            // mid-phase (prunes only): the capsule's bounding box in the frame of the box must overlap the box
            T dl[3], al[3];
            matTvec3(dl, rot1, dif);
            matTvec3(al, rot1, sax + 3 * pb);
#pragma unroll
            for (int k = 0; k < 3; k++) if (tabs(dl[k]) > co[CO_SIZE + k] + C.cap_r + C.cap_hl * tabs(al[k])) pass = false;
          }
        }
        const unsigned m = gballot(pass);
        if (pass) {
          const int slot = ncand + __popc(m & ((1u << sl) - 1));
          if (slot < cand_cap) cand[slot] = pt | (pa << 3) | (pb << 8); else flags |= SG_ST_CON_FULL;
        }
        ncand += __popc(m);
      }
    }
    if (ncand > cand_cap) ncand = cand_cap;
    const int ncand_w = wmax(ncand);   // also orders the candidate writes before the reads below
    // ---- narrowphase over the candidate list; contacts keep the pair order ----
    int ncon = 0, ncontot = 0, touch = 0;
    for (int base = 0; base < ncand_w; base += LPW) {
      const int ci_ = base + sl;
      RawCon<T> rc[2];
      int n = 0, pa = 0, e = -1; T ssign = 0;
      if (ci_ < ncand) {
        const int cw = cand[ci_];
        const int pt = cw & 7; pa = (cw >> 3) & 31; const int pb = cw >> 8;
        const T* co = scoll + pa * CO_STRIDE;
        T c1[3], rot1[9];
        collider_pose(pa, c1, rot1);
        T size1[3] = {co[CO_SIZE], co[CO_SIZE + 1], co[CO_SIZE + 2]};
        int mask = (int)co[CO_MASK];
        if (pt == PAIR_PLANE_CAPSULE) {
          T cc[3]; capsule_center(pb, cc);
          n = plane_capsule(rc, c1, rot1, cc, sax + 3 * pb, C.cap_r, C.cap_hl);
          e = pb; ssign = 1; mask |= C.cap_mask;
        } else if (pt == PAIR_BOX_CAPSULE) {
          T cc[3]; capsule_center(pb, cc);
          n = capsule_box(rc, cc, sax + 3 * pb, C.cap_r, C.cap_hl, c1, rot1, size1);
          e = pb; ssign = -1; mask |= C.cap_mask;
        } else if (pt == PAIR_SPHERE_BOX) {
          T sc[3];
#pragma unroll
          for (int k = 0; k < 3; k++) sc[k] = off[k] + C.sph_pos[k];
          n = sphere_box(rc[0], sc, C.sph_r, c1, rot1, size1);
          e = -1; mask |= C.sph_mask;
        } else if (pt == PAIR_BOX_BOX) {
          const T* co2 = scoll + pb * CO_STRIDE;
          T c2[3], rot2[9]; collider_pose(pb, c2, rot2);
          T size2[3] = {co2[CO_SIZE], co2[CO_SIZE + 1], co2[CO_SIZE + 2]};
          if (box_box_overlap(c1, rot1, size1, c2, rot2, size2)) flags |= SG_ST_UNSUPPORTED;
        } else flags |= SG_ST_UNSUPPORTED;
        if (n > 0) { touch |= (1 << 30); if (mask & 1) touch |= (mask >> 1); }
      }
      // contacts with dist >= 0 (== includemargin) exist but carry no constraint rows
      const int n_act = (n > 0 && rc[0].dist < T(0) ? 1 : 0) + (n > 1 && rc[1].dist < T(0) ? 1 : 0);
      const unsigned m1 = gballot(n_act >= 1), m2 = gballot(n_act >= 2);
      const unsigned t1 = gballot(n >= 1), t2 = gballot(n >= 2);
      const unsigned lt = (1u << sl) - 1;
      int slot = ncon + __popc(m1 & lt) + __popc(m2 & lt);
      int dslot = ncontot + __popc(t1 & lt) + __popc(t2 & lt);
      for (int i = 0; i < n; i++) {
        if (rc[i].dist < T(0)) {
          if (slot < D.maxcon) contact_rows(slot, rc[i], pa, e, ssign, dbg, dslot + i);
          else flags |= SG_ST_CON_FULL;
          slot++;
        }
      }
      ncon += __popc(m1) + __popc(m2);
      ncontot += __popc(t1) + __popc(t2);
    }
    if (ncon > D.maxcon) ncon = D.maxcon;
    touch = gor(touch);
    flags = gor(flags);
    if (sl == 0) { misc(M2_NCON) = ncon; misc(M2_TOUCH) = touch; misc(M2_NCONTOT) = ncontot; misc(M2_STATUS) |= flags; misc(M2_NCAND) = ncand; }
    __syncwarp();
    // ---- Gauss-Seidel schedule of the contact blocks.  A block is processed by the lane of its finger chain
    // (blocks against static colliders: the remaining lanes, round robin); its time slot is one more than the
    // latest earlier block on the same lane or on the same slider -- exactly the dependencies of the
    // sequential sweep of mj_solPGS, so the result equals the sequential one. ----
    // per-slider and per-lane latest time slots: in the scratch of the capsule centres, which are dead by now
    int* lastt = reinterpret_cast<int*>(scr(L.sc_cen));
    int* lanet = lastt + D.ns;
    const int clpw = LPW;                                         // lanes that sweep this world's limit/contact rows
    const int nfree = clpw > MAXCHAIN ? clpw - MAXCHAIN : 0;
    for (int e = sl; e < D.ns; e += LPW) lastt[e] = 0;
    lanet[sl] = 0;
    __syncwarp();
    if (sl == 0) {
      int tmax_ = 0, nstat = 0;
      const int* const icon = pin_g(auxi + L.i_con);
      int* const itl = pin_g(auxi + L.i_tl);
      int ce_next = ncon > 0 ? icon[0] : 0;
      for (int i = 0; i < ncon; i++) {
        const int ce = ce_next;
        if (i + 1 < ncon) ce_next = icon[i + 1];                 // the record index list lives in the global scratch
        const int c = (ce & 15) - 1, e = (ce >> 4) - 1;
        int ln;
        if (c >= 0) ln = c % clpw;
        else { ln = nfree > 0 ? MAXCHAIN + (nstat % nfree) : nstat % clpw; nstat++; }
        int t = lanet[ln];
        if (e >= 0) { const int te = lastt[e]; if (te > t) t = te; }
        t += 1;
        lanet[ln] = t;
        if (e >= 0) lastt[e] = t;
        itl[i] = t | (ln << 16);
        if (t > tmax_) tmax_ = t;
      }
      misc(M2_TMAX) = tmax_;
    }
    __syncwarp();
  }

  // ------------------------------------------------------------------------------------------
  // equality / tendon / limit rows and smooth dynamics of the shell
  // ------------------------------------------------------------------------------------------
  struct Tendon { T u, R, A, nA, aref; }; // group-uniform registers: u = R f - aref, nA = -1 / A
  struct ChainRows {                      // registers of the lane that owns a finger chain
    T ag[MAXCD];                          // running qacc of the chain dofs during the sweeps
    int lmask;                            // bit jl: limit of local dof jl is active
  };
  // limit rows live in shared memory (hot): f, aref, R, sign per finger dof
  __device__ __forceinline__ T& lf(int dof) { return hot[L.hlim + dof]; }
  __device__ __forceinline__ T& laref(int dof) { return hot[L.hlim + MAXFD + dof]; }
  __device__ __forceinline__ T& lR(int dof) { return hot[L.hlim + 2 * MAXFD + dof]; }
  __device__ __forceinline__ T& lsgn(int dof) { return hot[L.hlim + 3 * MAXFD + dof]; }

  __device__ void rows_and_smooth(Tendon& tn, T& Ft_out) {
    const int nfd = D.nfd, ns = D.ns;
    const bool dbg = valid && (w == K.debug_world) && K.debug_out;
    // volume tendon: L = sum c_e q_e, Ldot = sum c_e v_e
    const T* __restrict__ qp = pin_g(q() + nfd);     // qpos / qvel of the sliders are read-only in this stage
    const T* __restrict__ vp = pin_g(v() + nfd);
    T Ls = 0, Lv = 0, As = 0;
    batched<8, V2<T>>(sl, ns, LPW,
      [&](int e, V2<T>& x) SG_INL { x.a = qp[e]; x.b = vp[e]; },
      [&](int e, const V2<T>& x) SG_INL { const T tc = stc[e]; Ls += tc * x.a; Lv += tc * x.b; As += tc * stciw[e]; });
    Ls = gsum(Ls); Lv = gsum(Lv); As = gsum(As);
    const T Ft = -ten_stiffness() * (Ls - C.ten_lspring) - ten_damping() * Lv;
    Ft_out = Ft;
    // sliders: qacc_smooth = (passive - bias) / m  (bias = -m axis.g for a slider on a static parent)
    T* __restrict__ qsp = pin_g(qs() + nfd);
    batched<8, V5<T>>(sl, ns, LPW,
      [&](int e, V5<T>& x) SG_INL { x.a = qp[e]; x.b = vp[e]; x.c = tab(D.o_sl_m)[e]; x.d = stiffness(e); x.e = damping(e); },
      [&](int e, const V5<T>& x) SG_INL {
        const T* ax = sax + 3 * e;                         // (the CTA-shared copy of the slider axes)
        T f = -x.d * x.a - x.e * x.b;
        f += stc[e] * Ft;
        f -= -(x.c * (ax[0] * C.g[0] + ax[1] * C.g[1] + ax[2] * C.g[2]));
        qsp[e] = f * stiw(e);
      });
    // joint-equality rows in schedule order: row2 = (aref, R) until the warm start turns aref into u
    const int* __restrict__ rd = srd;
    const T* __restrict__ siwt = pin_t(tab(D.o_sl_iw));
    T* __restrict__ row2 = hot + L.row2;
    batched<8, V3<T>>(sl, D.nrow, LPW,
      [&](int p, V3<T>& x) SG_INL {
        const int d12 = rd[p], d1 = d12 & 0xffff, d2 = (d12 >> 16) & 0xffff;
        T pos = qp[d1], vel = vp[d1], diag = siwt[d1];     // (dof_invweight0 is not bit-uniform over the sliders: table loads)
        if (d2 != 0xffff) { pos -= qp[d2]; vel -= vp[d2]; diag += siwt[d2]; }
        x.a = pos; x.b = vel; x.c = diag;
      },
      [&](int p, const V3<T>& x) SG_INL {
        const T imp = impedance2<T>(C.eqj_si, x.a);
        const T aref = -C.eqj_B * x.b - C.eqj_K * imp * x.a;
        row2[2 * p] = aref;
        row2[2 * p + 1] = tmax(T(SG_MINVAL), (T(1) - imp) * x.c / imp);
        if (dbg) { K.debug_out[K.debug_cap - (D.nrow + 1) + p] = (double)aref; K.debug_out[K.debug_cap - 2 * (D.nrow + 1) + p] = (double)row2[2 * p + 1]; }
      });
    {
      const T pos = Ls - C.ten_l0;
      const T imp = impedance2<T>(C.eqt_si, pos);
      tn.R = tmax(T(SG_MINVAL), (T(1) - imp) * C.ten_iw / imp);
      tn.aref = -C.eqt_B * Lv - C.eqt_K * imp * pos;
      tn.A = As + tn.R;
      tn.nA = T(-1) / tn.A;
      tn.u = 0;
    }
    __syncwarp();
  }

  // joint limits of the chain owned by this lane, lower then upper, in joint order (mj_instantiateLimit)
  __device__ void chain_limits(int c, ChainRows& cr) {
    cr.lmask = 0;
    const int d0 = D.chain_dof0[c];
#pragma unroll
    for (int jl = 0; jl < MAXCD; jl++) {
      if (jl >= D.ncd[c]) continue;
      lf(d0 + jl) = 0; laref(d0 + jl) = 0; lR(d0 + jl) = 1; lsgn(d0 + jl) = 0;
      const T* cd = tab(D.o_chain + c * CH_STRIDE + CH_DOF + jl * CD_STRIDE);
      if (cd[CD_LIMITED] == T(0)) continue;
      const T qq = q()[d0 + jl];
      const T dlo = qq - cd[CD_LO], dhi = cd[CD_HI] - qq;
      T dist = 0, sgn = 0;
      if (dlo < T(0)) { dist = dlo; sgn = 1; }
      else if (dhi < T(0)) { dist = dhi; sgn = -1; }
      else continue;
      const T imp = impedance2<T>(C.lim_si, dist);
      lR(d0 + jl) = tmax(T(SG_MINVAL), (T(1) - imp) * cd[CD_IW] / imp);
      laref(d0 + jl) = -C.lim_B * (sgn * v()[d0 + jl]) - C.lim_K * imp * dist;
      lsgn(d0 + jl) = sgn;
      cr.lmask |= 1 << jl;
    }
    misc(M2_LMASK + c) = cr.lmask;
  }

  __device__ __forceinline__ int chain_of(int dof) const {
    int c = 0;
    for (int k = 1; k < D.nchain; k++) if (dof >= D.chain_dof0[k]) c = k;
    return c;
  }

  // elliptic-cone warm-start force of one contact from jar (mj_constraintUpdate zones, SURVEY App. A4)
  __device__ __forceinline__ void cone_force(const T* jar, T R0, T R1, T* f) {
    const T frc = C.con_fr, mu = frc * tsqrt(R1 / R0);
    f[0] = -(T(1) / R0) * jar[0]; f[1] = -(T(1) / R1) * jar[1]; f[2] = -(T(1) / R1) * jar[2];
    const T U0 = jar[0] * mu, U1 = jar[1] * frc, U2 = jar[2] * frc;
    const T N = U0, Tn = tsqrt(U1 * U1 + U2 * U2);
    if (N >= mu * Tn || (Tn <= T(0) && N >= T(0))) { f[0] = f[1] = f[2] = 0; }
    else if (mu * N + Tn <= T(0) || (Tn <= T(0) && N < T(0))) { }
    else {
      const T Dm = (T(1) / R0) / (mu * mu * (T(1) + mu * mu)), NT = N - mu * Tn;
      f[0] = -Dm * NT * mu;
      f[1] = -f[0] / Tn * U1 * frc; f[2] = -f[0] / Tn * U2 * frc;
    }
  }

  // warm start (SURVEY App. A4): forces from qacc_warmstart (in a()), kept only if the dual cost
  // f.b + 0.5 f'AR f is not positive; leaves a() = qacc_smooth + M^-1 J^T f and row2 = (u, R)
  __device__ void warmstart(Tendon& tn, ChainRows& cr) {
    const int nfd = D.nfd, ns = D.ns;
    const int ncon = misc(M2_NCON);
    const int* rd = srd;
    T* row2 = hot + L.row2;
    T* jtf = pin_g(aux + L.jtf);
    const int* const dof_rows = K.itab + keep_off((long long)D.io_dof_rows);
    const int* const icon = pin_g(auxi + L.i_con);
    T* const rec0 = pin_g(aux + L.crec);
    // dual cost = sum_rows (0.5 R f^2 - f aref) + (J^T f).qacc_smooth + 0.5 (J^T f)' M^-1 (J^T f): the middle term is
    // sum_rows f (J qacc_smooth) regrouped per dof, so no row ever has to gather qacc_smooth
    T cost = 0;
    // equality rows: per-dof gather of J^T f over the rows of each slider (no scatter, no atomics)
    T tja = 0;
    struct RowsV { int code[MAXDOFROWS]; };
    batched<8, RowsV>(sl, ns, LPW,
      [&](int e, RowsV& x) SG_INL {
        const int* dr = dof_rows + e * MAXDOFROWS;
#pragma unroll
        for (int k = 0; k < MAXDOFROWS; k++) x.code[k] = dr[k];
      },
      [&](int e, const RowsV& x) SG_INL {
        T s = 0;
        const T ae = a()[nfd + e];
#pragma unroll
        for (int k = 0; k < MAXDOFROWS; k++) {
          // entry (sg_api.cu host_tables): row position | other slider << 12 (0xfff: none) | "e is the second slider" << 24
          const int code = x.code[k];
          if (code >= 0) {
            const int p = code & 0xfff, other = (code >> 12) & 0xfff;
            const bool second = (code >> 24) & 1;
            const T ao = other != 0xfff ? a()[nfd + other] : T(0);
            const T ja = second ? ao - ae : ae - ao;
            T ar, R; ld2(row2 + 2 * p, ar, R);
            const T f = -(T(1) / R) * (ja - ar);
            if (second) s -= f;
            else { s += f; cost += f * (T(0.5) * R * f - ar); }   // the row's own cost: counted once, by its first dof
          }
        }
        tja += stc[e] * ae;
        jtf[nfd + e] = s;
      });
    tja = gsum(tja);
    const T tf = -(T(1) / tn.R) * (tja - tn.aref);
    if (sl == 0) cost += tf * (T(0.5) * tn.R * tf - tn.aref);
    batched<8, V1<T>>(sl, ns, LPW, [&](int e, V1<T>& x) SG_INL { x.a = jtf[nfd + e]; }, [&](int e, const V1<T>& x) SG_INL { jtf[nfd + e] = x.a + stc[e] * tf; });
    // limits (the chain lanes)
    if (sl < D.nchain) {
      const int d0 = D.chain_dof0[sl];
#pragma unroll
      for (int jl = 0; jl < MAXCD; jl++) {
        if (jl < D.ncd[sl]) jtf[d0 + jl] = 0;
        if (!(cr.lmask & (1 << jl))) continue;
        const T sgn = lsgn(d0 + jl), ar = laref(d0 + jl), R = lR(d0 + jl);
        const T jar = sgn * a()[d0 + jl] - ar;
        const T f = jar >= T(0) ? T(0) : -(T(1) / R) * jar;
        lf(d0 + jl) = f;
        jtf[d0 + jl] = sgn * f;
        cost += f * (T(0.5) * R * f - ar);
      }
    }
    // contacts
    for (int i = sl; i < ncon; i += LPW) {
      const int ce = icon[i];
      const int c = (ce & 15) - 1, e = (ce >> 4) - 1;
      T* r = rec0 + CR_STRIDE * i;
      // the words of the record in one batch of vector loads (one L2 round trip beside the one of icon[i])
      T jg[12], w1[4], w2[4];
      ld4(r + CR_JG, jg); ld4(r + CR_JG + 4, jg + 4); ld4(r + CR_JG + 8, jg + 8);
      ld4(r + CR_NS, w1); ld4(r + CR_AREF, w2);
      const T R0 = w2[3], R1 = R0 * C.inv_impratio;
      T jar[3];
#pragma unroll
      for (int k = 0; k < 3; k++) {
        T sa = 0;
        if (e >= 0) sa = w1[k] * a()[nfd + e];
        if (c >= 0) {
#pragma unroll
          for (int jj = 0; jj < MAXCD; jj++) if (jj < D.ncd[c]) sa += jg[4 * k + jj] * a()[D.chain_dof0[c] + jj];
        }
        jar[k] = sa - w2[k];
      }
      T f[3];
      cone_force(jar, R0, R1, f);
      const T Rr[3] = {R0, R1, R1};
#pragma unroll
      for (int k = 0; k < 3; k++) { r[CR_F + k] = f[k]; cost += f[k] * (T(0.5) * Rr[k] * f[k] - w2[k]); }
    }
    __syncwarp();
    // J^T f of the contacts, added after the limits.  Deterministic without atomics: the contacts of slider e are
    // summed, in contact order, by lane e % LPW (sliders are private to that lane); the finger-dof parts are kept in
    // registers per lane and then reduced over the lanes in a fixed order.
    {
      T gd[MAXCHAIN][MAXCD];
#pragma unroll
      for (int c = 0; c < MAXCHAIN; c++)
#pragma unroll
        for (int jj = 0; jj < MAXCD; jj++) gd[c][jj] = 0;
      for (int i0 = 0; i0 < ncon; i0 += 4) {
        const int4 ce4 = *reinterpret_cast<const int4*>(icon + i0);     // four table entries per L2 round trip
        for (int j = 0; j < 4 && i0 + j < ncon; j++) {
          const int i = i0 + j;
          const int ce = j == 0 ? ce4.x : j == 1 ? ce4.y : j == 2 ? ce4.z : ce4.w;
          const int c = (ce & 15) - 1, e = (ce >> 4) - 1;
          if ((e >= 0 ? e : i) % LPW != sl) continue;
          const T* r = rec0 + CR_STRIDE * i;
          T jg[12], w1[4], f[4];
          ld4(r + CR_NS, w1); ld4(r + CR_F, f);
          if (c >= 0) { ld4(r + CR_JG, jg); ld4(r + CR_JG + 4, jg + 4); ld4(r + CR_JG + 8, jg + 8); }
          if (e >= 0) jtf[nfd + e] += w1[0] * f[0] + w1[1] * f[1] + w1[2] * f[2];
          if (c >= 0) {
#pragma unroll
            for (int cc = 0; cc < MAXCHAIN; cc++)
              if (cc == c) {
#pragma unroll
                for (int jj = 0; jj < MAXCD; jj++) gd[cc][jj] += jg[jj] * f[0] + jg[4 + jj] * f[1] + jg[8 + jj] * f[2];
              }
          }
        }
      }
#pragma unroll
      for (int c = 0; c < MAXCHAIN; c++)
#pragma unroll
        for (int jj = 0; jj < MAXCD; jj++) {
          const T tot = gsum(gd[c][jj]);
          if (sl == 0 && c < D.nchain && jj < D.ncd[c]) jtf[D.chain_dof0[c] + jj] += tot;
        }
    }
    __syncwarp();
    // (J^T f).qacc_smooth + 0.5 (J^T f)' M^-1 (J^T f)
    batched<8, V2<T>>(sl, ns, LPW, [&](int e, V2<T>& x) SG_INL { x.a = jtf[nfd + e]; x.b = qs()[nfd + e]; },
                      [&](int e, const V2<T>& x) SG_INL { cost += x.a * (x.b + T(0.5) * x.a * stiw(e)); });
    for (int dof = sl; dof < nfd; dof += LPW) {
      const int c = chain_of(dof), jl = dof - D.chain_dof0[c];
      T s = 0;
      for (int jj = 0; jj < D.ncd[c]; jj++) s += hot[L.minv + 16 * c + 4 * jl + jj] * jtf[D.chain_dof0[c] + jj];
      cost += jtf[dof] * (qs()[dof] + T(0.5) * s);
    }
    cost = gsum(cost);
    const bool keep = !(cost > T(0));
    // (aref, R) -> (u, n):  u = R f - aref is -(J.qacc_warm) when the warm start is kept and -aref when it is dropped;
    // n = -1 / (1/m1 + 1/m2 + R) is what the sweep multiplies the residual with
    if (K.tm_cols) rows_to_tm(keep);
    else
    for (int p = sl; p < D.nrow; p += LPW) {
      const int d12 = rd[p], d1 = d12 & 0xffff, d2 = (d12 >> 16) & 0xffff;
      T ar, R; ld2(row2 + 2 * p, ar, R);
      T ja = a()[nfd + d1], diag = stiw(d1);
      if (d2 != 0xffff) { ja -= a()[nfd + d2]; diag += stiw(d2); }
      row2[2 * p] = keep ? -ja : -ar;
      row2[2 * p + 1] = T(-1) / (diag + R);
    }
    tn.u = keep ? -tja : -tn.aref;
    if (!keep) {
      if (sl < D.nchain) {
#pragma unroll
        for (int jl = 0; jl < MAXCD; jl++) if (jl < D.ncd[sl]) lf(D.chain_dof0[sl] + jl) = 0;
      }
      for (int i = sl; i < ncon; i += LPW) { T* r = rec0 + CR_STRIDE * i; r[CR_F] = 0; r[CR_F + 1] = 0; r[CR_F + 2] = 0; }
    }
    __syncwarp();
    // a = qacc_smooth + M^-1 jtf (or qacc_smooth alone)
    batched<8, V2<T>>(sl, ns, LPW, [&](int e, V2<T>& x) SG_INL { x.a = qs()[nfd + e]; x.b = jtf[nfd + e]; },
                      [&](int e, const V2<T>& x) SG_INL { a()[nfd + e] = x.a + (keep ? x.b * stiw(e) : T(0)); });
    for (int dof = sl; dof < nfd; dof += LPW) {
      const int c = chain_of(dof), jl = dof - D.chain_dof0[c];
      T s = 0;
      if (keep) for (int jj = 0; jj < D.ncd[c]; jj++) s += hot[L.minv + 16 * c + 4 * jl + jj] * jtf[D.chain_dof0[c] + jj];
      a()[dof] = qs()[dof] + s;
    }
    __syncwarp();
  }

  // friction forces with the normal force fixed: mju_QCQP2 + rescaling onto the cone (mj_solPGS); the fp32 fast path
  // solves the same problem with friction_fast
  __device__ __forceinline__ void friction(T& f1, T& f2, T& la, T A11, T A12, T A22, T a11n, T a12n, T kb, const T* bc, T frc, T f0) {
    if (sizeof(T) == 4) {
      float g1, g2, gl = (float)la;
      friction_fast(g1, g2, gl, (float)a11n, (float)a12n, (float)kb, (float)bc[0], (float)bc[1], (float)frc, (float)f0);
      f1 = T(g1); f2 = T(g2); la = T(gl); return;
    }
    T vv[2];
    const int active = qcqp2_fast<T>(vv, A11, A12, A22, bc, frc, frc, f0);
    if (active) {
      const T ifr2 = tdiv(T(1), frc * frc);
      T s = vv[0] * vv[0] * ifr2 + vv[1] * vv[1] * ifr2;
      s = tsqrt(tdiv(f0 * f0, tmax(T(SG_MINVAL), s)));
      vv[0] *= s; vv[1] *= s;
    }
    f1 = vv[0]; f2 = vv[1];
  }
  // One elliptic contact block (mj_solPGS inner body, dim 3) on the lane that owns its finger chain, or on one of the other
  // lanes for a contact against a static collider.  No data-dependent branch outside the friction solve (selects instead),
  // and one code path for both kinds of lane: a static contact has a zero finger Jacobian and the lane a zero chain
  // acceleration, a contact without a slider goes through the dummy slider.  That leaves two large basic blocks around the
  // Newton loop of the friction solve for the scheduler to interleave (profiles/r02e_sweep.txt: 1.193e7 -> 1.223e7).
  struct Rec { T jg[12], w1[4], w2[4], Aw[8], w3[4]; };      // the 32 words of one contact record in registers
  __device__ __forceinline__ void load_rec(Rec& x, const T* r) const {
    ld4(r + CR_JG, x.jg); ld4(r + CR_JG + 4, x.jg + 4); ld4(r + CR_JG + 8, x.jg + 8);
    ld4(r + CR_NS, x.w1);          // ns0 ns1 ns2 a12n
    ld4(r + CR_AREF, x.w2);        // aref0 aref1 aref2 R0
    ld4(r + CR_A, x.Aw); ld4(r + CR_A + 4, x.Aw + 4);   // A00 A01 A02 A11 | A12 A22 a11n kb
    ld4(r + CR_F, x.w3);           // f0 f1 f2, friction multiplier of the previous sweep
  }
  __device__ __forceinline__ void load_rec_ring(Rec& x, ring_t a) const {
    constexpr unsigned S = sizeof(T);
    lds4(a + S * CR_JG, x.jg); lds4(a + S * (CR_JG + 4), x.jg + 4); lds4(a + S * (CR_JG + 8), x.jg + 8);
    lds4(a + S * CR_NS, x.w1); lds4(a + S * CR_AREF, x.w2);
    lds4(a + S * CR_A, x.Aw); lds4(a + S * (CR_A + 4), x.Aw + 4);
    lds4(a + S * CR_F, x.w3);
  }
  // r: the record in the scratch, which takes the new force; RING: the record is read from its copy in the lane's
  // shared-memory ring (rl) instead
  template <bool RING>
  __device__ __forceinline__ T contact_block(T* r, ring_t rl, int e, T* ag, const T* mv, T* asl, T frc, T iwu) {
    Rec x;
    if (RING) load_rec_ring(x, rl); else load_rec(x, r);
    // a contact without a slider (centre sphere) reads and writes the dummy slider: its ns and 1/m words are zero
    T* const pae = asl + (e >= 0 ? e : D.ns);
    const T ae = *pae;
    const T* jg = x.jg; const T* w1 = x.w1; const T* w2 = x.w2; const T* Aw = x.Aw; const T* w3 = x.w3;
    const T A00 = Aw[0], A01 = Aw[1], A02 = Aw[2], A11 = Aw[3], A12 = Aw[4], A22 = Aw[5];
    const T R0 = w2[3], R1 = R0 * C.inv_impratio;
    const T iwe = e >= 0 ? iwu : T(0);                   // 1 / m of the contact's slider: one value for the whole shell
    const T old0 = w3[0], old1 = w3[1], old2 = w3[2];
    T la = w3[3];
    T res[3];
    const T Rr[3] = {R0, R1, R1};
    const T fo[3] = {old0, old1, old2};
#pragma unroll
    for (int k = 0; k < 3; k++) {
      T s = Rr[k] * fo[k] - w2[k];
#pragma unroll
      for (int jj = 0; jj < MAXCD; jj++) s += jg[4 * k + jj] * ag[jj];
      res[k] = s + w1[k] * ae;
    }
    // normal force: plain update of an inactive contact, ray update of an active one (mj_solPGS)
    const bool active = !(old0 < T(SG_MINVAL));
    const T x0 = A00 * old0 + A01 * old1 + A02 * old2, x1 = A01 * old0 + A11 * old1 + A12 * old2, x2 = A02 * old0 + A12 * old1 + A22 * old2;
    const T denom = old0 * x0 + old1 * x1 + old2 * x2;
    const bool okden = denom >= T(SG_MINVAL);
    T xr = -tdiv(old0 * res[0] + old1 * res[1] + old2 * res[2], okden ? denom : T(1));
    if (old0 + xr * old0 < T(0)) xr = T(-1);
    xr = okden ? xr : T(0);
    T f0n = old0 - tdiv(res[0], A00);
    f0n = f0n < T(0) ? T(0) : f0n;
    T f0 = active ? old0 + xr * old0 : f0n;
    T f1 = active ? old1 + xr * old1 : T(0);
    T f2 = active ? old2 + xr * old2 : T(0);
    // friction update with the normal force fixed
    {
      T bc[2];
      bc[0] = res[1] - (A11 * old1 + A12 * old2) + A01 * (f0 - old0);
      bc[1] = res[2] - (A12 * old1 + A22 * old2) + A02 * (f0 - old0);
      if (f0 < T(SG_MINVAL)) { f1 = 0; f2 = 0; la = 0; }
      else friction(f1, f2, la, A11, A12, A22, Aw[6], w1[3], Aw[7], bc, frc, f0);
    }
    // the chain's M^-1 block on its way (shared memory) while the cost test runs: 1.447e7 -> 1.474e7 world-steps/s against
    // loading it after the test (profiles/r02zc_sweep.log)
    T m16[16];
#pragma unroll
    for (int ii = 0; ii < MAXCD; ii++) ld4(mv + 4 * ii, m16 + 4 * ii);
#if defined(SG_FRIC_STATS) && !defined(__CUDA_ARCH__)
    {
      // development statistics under the emulator: how many blocks are no-ops (an inactive contact that stays inactive)
      static long nblk = 0, nstay = 0, nactive = 0;
      nblk++;
      if (!active && !(f0 > T(0))) nstay++;
      if (active) nactive++;
      if ((nblk & 0xfffff) == 0) fprintf(stderr, "contact_block: %ld blocks, %.3f inactive and staying inactive, %.3f active on entry\n", nblk, (double)nstay / nblk, (double)nactive / nblk);
    }
#endif
    // cost change, revert if positive
    T d0f = f0 - old0, d1f = f1 - old1, d2f = f2 - old2;
    T change = T(0.5) * (d0f * (A00 * d0f + A01 * d1f + A02 * d2f) + d1f * (A01 * d0f + A11 * d1f + A12 * d2f) + d2f * (A02 * d0f + A12 * d1f + A22 * d2f))
             + d0f * res[0] + d1f * res[1] + d2f * res[2];
    const bool revert = change > T(1e-10);
    f0 = revert ? old0 : f0; f1 = revert ? old1 : f1; f2 = revert ? old2 : f2;
    d0f = revert ? T(0) : d0f; d1f = revert ? T(0) : d1f; d2f = revert ? T(0) : d2f;
    change = revert ? T(0) : change;
    st4(r + CR_F, f0, f1, f2, la);
    // qacc += M^-1 J^T delta: unconditionally (a zero change adds exact zeros)
    *pae = ae + (w1[0] * d0f + w1[1] * d1f + w1[2] * d2f) * iwe;
    T gv[MAXCD];
#pragma unroll
    for (int jj = 0; jj < MAXCD; jj++) gv[jj] = jg[jj] * d0f + jg[4 + jj] * d1f + jg[8 + jj] * d2f;
#pragma unroll
    for (int ii = 0; ii < MAXCD; ii++) {
      const T* m4 = m16 + 4 * ii;
      ag[ii] += m4[0] * gv[0] + m4[1] * gv[1] + m4[2] * gv[2] + m4[3] * gv[3];
    }
    return change;
  }

  // ---- limit / contact rows: swept by the lane that owns the finger chain (plus a share of the static contacts) ----
  struct ChainState {
    T ag[MAXCD];            // running qacc of the chain dofs, in registers for the whole solve
    const T* mv;            // the chain's M^-1 block (shared memory)
    T* asl;                 // the world's slider accelerations (shared memory): a() + nfd
    T frc;                  // contact friction coefficient
    T iwu;                  // 1 / slider mass (uniform shell)
    int lmask, mystart, mycnt;
    bool chain_lane;
    bool primed;            // ring mode: the first record of the next sweep is already on its way
  };
  // this lane's slice of the contact schedule (contacts in their sequential order) and the chain's qacc
  __device__ void chain_prologue(ChainState& cs) {
    cs.chain_lane = sl < D.nchain;
    cs.mv = reinterpret_cast<const T*>(smem_base + keep_off((int)(reinterpret_cast<unsigned char*>(hot + L.minv + 16 * (cs.chain_lane ? sl : 0)) - smem_base)));
    cs.asl = reinterpret_cast<T*>(smem_base + keep_off((int)(reinterpret_cast<unsigned char*>(a() + D.nfd) - smem_base)));
    cs.frc = keep_val(C.con_fr);
    cs.iwu = keep_val(stim[0]);
    cs.lmask = cs.chain_lane ? misc(M2_LMASK + sl) : 0;
    cs.mystart = 0; cs.mycnt = 0; cs.primed = false;
    const int ncon = misc(M2_NCON);
    const int* const itl = pin_g(auxi + L.i_tl);
    const int* const icon = pin_g(auxi + L.i_con);
    for (int i0 = 0; i0 < ncon; i0 += 4) {
      int tl4[4]; ldi4(itl + i0, tl4);
#pragma unroll
      for (int j = 0; j < 4; j++) {
        const int ln = tl4[j] >> 16;
        if (i0 + j < ncon) { if (ln < sl) cs.mystart++; else if (ln == sl) cs.mycnt++; }
      }
    }
    int k = 0;
    int* const iord = pin_g(auxi + L.i_order + cs.mystart);
    for (int i0 = 0; i0 < ncon; i0 += 4) {
      int tl4[4]; ldi4(itl + i0, tl4);
#pragma unroll
      for (int j = 0; j < 4; j++) {
        const int i = i0 + j, tl = tl4[j];
        if (i < ncon && (tl >> 16) == sl) { iord[k] = i | ((tl & 0xff) << 8) | ((icon[i] >> 4) << 16); k++; }
      }
    }
#pragma unroll
    for (int jj = 0; jj < MAXCD; jj++) cs.ag[jj] = (cs.chain_lane && jj < D.ncd[sl]) ? a()[D.chain_dof0[sl] + jj] : T(0);
  }
  // one sweep over this lane's limit rows and contact blocks (time slots 1..tmaxw, a warp barrier after each);
  // returns the lane's cost improvement.  The contact records live in the L2-resident scratch: the lane's schedule
  // entries are fetched three blocks ahead (registers); without the ring (!RING) the 128-byte record of a later block is
  // prefetched into L1 when the current block starts.  (Measured neutral
  // or worse and removed again: records staged in registers one block ahead -- 1.1 KB of spills, -12 %; helper lanes
  // handing records over by shuffles, round 1; a reordered friction solve and a speculative M^-1 J' update -- the chain
  // phase sits where issue slots (4 warps x ~120 000 instructions per step) and single-warp latency (~540 000 cycles) meet.)
  // RING: the record of the lane's next block is copied asynchronously (cp.async, L2 -> shared memory) into the other
  // entry of a two-entry ring while the current block is computed, and the block reads its record from shared memory.
  // The ring of lane sl sits in the world's (aref, R) region, which is dead once rows_to_tm has moved the equality rows
  // to tensor memory: entry stride RB, lane stride 2 RB + 16 (the two chain lanes of a world land in different banks).
  // The contact-only profile (profiles/r02y_k2_ncu_contact_summary.txt) had 26 % of all stall samples on the first uses
  // of the record words: the L1 prefetch does not hold -- 64 worlds x ~2 blocks per slot x 128 B x (current + two ahead)
  // is twice the 27 KB of L1 that 228 KB of shared memory leave.
  template <bool RING>
  __device__ T chain_phase(ChainState& cs, int tmaxw, bool done) {
    T impr = 0;
    constexpr unsigned RB = CR_STRIDE * sizeof(T);
    const ring_t ring = ring_of(reinterpret_cast<unsigned char*>(hot) + sl * (int)(2 * RB + 16));
    const int* order = reinterpret_cast<const int*>(K.scratch + keep_off((long long)(reinterpret_cast<unsigned char*>(auxi + L.i_order + cs.mystart) - K.scratch)));
    const int cnt = done ? 0 : cs.mycnt;
    int entA = 0, entB = 0, entC = 0;
    if (cnt > 0) entA = order[0];
    if (cnt > 1) entB = order[1];
    if (cnt > 2) entC = order[2];
    const int ent0 = entA;
    if (RING) {
      if (cnt > 0 && !cs.primed) { cp_rec<RB>(ring, reinterpret_cast<const unsigned char*>(crec(ent0 & 0xff))); cs.primed = true; }
    } else if (cnt > 1) prefetch_l1(crec(entB & 0xff));
    if (cs.chain_lane && !done) {
#pragma unroll
      for (int jl = 0; jl < MAXCD; jl++) {
        if (!(cs.lmask & (1 << jl))) continue;
        const int dof = D.chain_dof0[sl] + jl;
        const T sgn = lsgn(dof), f = lf(dof), R = lR(dof);
        const T A = cs.mv[4 * jl + jl] + R;
        const T res = sgn * cs.ag[jl] - laref(dof) + R * f;
        T fn = f - tdiv(res, A);
        if (fn < T(0)) fn = 0;
        T dl = fn - f;
        T change = T(0.5) * dl * dl * A + dl * res;
        if (change > T(1e-10)) { fn = f; dl = 0; change = 0; }
        impr -= change;
        lf(dof) = fn;
        if (dl != T(0)) {
#pragma unroll
          for (int ii = 0; ii < MAXCD; ii++) cs.ag[ii] += cs.mv[4 * ii + jl] * sgn * dl;
        }
      }
    }
    int k = 0;
    {
      // one byte base for the records of this world; an entry's record is base + index * 128 (CR_STRIDE reals)
      unsigned char* const recb = K.scratch + keep_off((long long)(reinterpret_cast<unsigned char*>(aux + L.crec) - K.scratch));
      for (int t = 1; t <= tmaxw; t++) {
        if (k < cnt && ((entA >> 8) & 0xff) == t) {
          T* r = reinterpret_cast<T*>(recb + (size_t)((unsigned)(entA & 0xff) * RB));
          const int e = (entA >> 16) - 1;
          ring_t rl = ring;
          if (RING) {
            cp_wait();                                                // this block's record has landed in its ring entry
            rl = ring + (k & 1) * RB;
            if (k + 1 < cnt) cp_rec<RB>(ring + ((k + 1) & 1) * RB, recb + (size_t)((unsigned)(entB & 0xff) * RB));
          }
          k++;
          // two blocks ahead, as the entries (one block ahead measures the same, profiles/r02o_sweep.log: 1.216e7 / 1.223e7)
          if (!RING && k + 1 < cnt) prefetch_l1(recb + (size_t)((unsigned)(entC & 0xff) * RB));
          const int entD = (k + 2 < cnt) ? order[k + 2] : 0;
          impr -= contact_block<RING>(r, rl, e, cs.ag, cs.mv, cs.asl, cs.frc, cs.iwu);
          entA = entB; entB = entC; entC = entD;
        }
        __syncwarp();
      }
    }
    // next sweep's first entries and record: on their way while the equality block is swept
    if (cnt > 0) {
      prefetch_l1(order);
      if (RING) cp_rec<RB>(ring, reinterpret_cast<const unsigned char*>(crec(ent0 & 0xff)));
      else prefetch_l1(crec(ent0 & 0xff));
    }
    return impr;
  }
  __device__ void chain_epilogue(const ChainState& cs) {
    if (cs.chain_lane) {
#pragma unroll
      for (int jj = 0; jj < MAXCD; jj++) if (jj < D.ncd[sl]) a()[D.chain_dof0[sl] + jj] = cs.ag[jj];
    }
  }

  // one sweep over the equality block and the volume-tendon row; returns this lane's cost improvement.
  // Step slots (built per lanes-per-world by the host, staged in shared memory by the kernel prologue and shared by all
  // worlds of the CTA): slot = step * LPW + lane.  Slots that pad a step, and the second slider of fix rows, are
  // predicated off, so they cost no shared-memory wavefronts (the sweep is bound by those, see sg_plan.hpp).
  // Per row the sweep keeps (u, n) with u = R f - aref and n = -1 / (1/m1 + 1/m2 + R): the residual is a1 - a2 + u, the
  // force change dl = res * n, and since an (unclamped) equality row has zero residual right after its own update, the
  // new u is simply a2' - a1' -- neither R nor f is needed, and there is no division in the sweep.
  // TM: the (u, n) pair of this lane's slot of step `st` is in the lane's tensor memory at column st * TmPair<T>::cols
  // (written by rows_to_tm at the end of the warm start); the pair of the next step is requested before this step's
  // arithmetic, so the sweep never waits for it.  Padding slots hold (0, 0) and go through the arithmetic as zeros.
  template <bool GATED, bool TM = false>
  __device__ __forceinline__ T equality_rows(bool done) {
    const int nstep = D.nstep;
    char* avb = reinterpret_cast<char*>(a() + D.nfd);
    char* rwb = reinterpret_cast<char*>(hot);     // Layout2::row2 == 0 (make_layout2)
    T acc = 0;                                   // sum of res * dl = -2 * cost improvement
    constexpr unsigned CW = TmPair<T>::cols;
    unsigned tcol = tm;
    T un_ = 0, nn_ = 0;
    if (TM) tm_ld2(tcol, un_, nn_);
    const T iwu = stim[0];                       // 1 / element mass, the same for every slider
    // one row per lane per step, a warp barrier where the schedule asks for one.  The next step's slot is fetched
    // before the barrier so that its latency overlaps this step's arithmetic.
    Slot<T> sn = ld_slot<T>(slots);
    // unrolled by four: 1.202e7 / 1.200e7 / 1.227e7 world-steps/s at 1 / 2 / 4 (profiles/r02j_sweep.log)
#pragma unroll 4
    for (int st = 0; st < nstep; st++) {
      const Slot<T> sc = sn;
      sn = ld_slot<T>(slots + (st + 1) * LPW);   // the table carries one empty step past the end
      const unsigned o2 = sc.x >> 16;
      const bool valid = (sc.y & 0x40000000u) != 0u, has2 = o2 != 0xffffu;     // padding slot / fix row: predicated off
      T* pa1 = reinterpret_cast<T*>(avb + (sc.x & 0xffffu));
      T* pa2 = reinterpret_cast<T*>(avb + o2);
      T* pr = reinterpret_cast<T*>(rwb + (sc.y & 0x3fffffffu));
      T a1 = 0, a2 = 0, u = 0, n = 0;
      if (TM) {
        tm_wait_ld(un_, nn_);
        u = un_; n = nn_;
        tm_ld2(tcol + CW, un_, nn_);              // next step's pair (the window carries one empty step past the end)
        if (valid) a1 = *pa1;
      } else if (valid) { a1 = *pa1; ld2(pr, u, n); }
      if (has2) a2 = *pa2;
      const T res = (a1 - a2) + u;
      if (GATED) n = done ? T(0) : n;
      const T dl = res * n;
      acc += dl * res;
      a1 += iwu * dl; a2 -= (has2 ? iwu : T(0)) * dl;        // fix rows have no second slider
      T un = a2 - a1;
      if (GATED) un = done ? u : un;
      if (TM) { tm_st1(tcol, un); tcol += CW; if (valid) *pa1 = a1; }
      else if (valid) { *pr = un; *pa1 = a1; }
      if (has2) *pa2 = a2;
      // nearly every step of the 8-lane schedules ends a dependency level: an unconditional barrier is cheaper than
      // testing the flag; narrower worlds have runs of independent steps that are allowed to overlap
      if (LPW >= 8 || (int)sc.y < 0) __syncwarp();
    }
    if (TM) { tm_wait_ld(un_, nn_); tm_wait_st(); }     // the look-ahead load has landed; the stores are visible to the next sweep
    return T(-0.5) * acc;
  }
  // (aref, R) of the warm start -> (u, n) of the sweep, from the compact shared-memory pairs into the slot order of the
  // lane's tensor memory (see warmstart for the formulas); padding slots and the step past the end become (0, 0)
  __device__ void rows_to_tm(bool keep) {
    const int nstep = D.nstep;
    const char* avb = reinterpret_cast<const char*>(a() + D.nfd);
    const char* rwb = reinterpret_cast<const char*>(hot);
    constexpr unsigned CW = TmPair<T>::cols;
    unsigned tcol = tm;
    const T iwu = stim[0];
    for (int st = 0; st <= nstep; st++, tcol += CW) {
      const Slot<T> sc = ld_slot<T>(slots + st * LPW);
      const unsigned o2 = sc.x >> 16;
      const bool valid = st < nstep && (sc.y & 0x40000000u) != 0u, has2 = st < nstep && o2 != 0xffffu;
      T u = 0, n = 0;
      if (valid) {
        T ar, R; ld2(reinterpret_cast<const T*>(rwb + (sc.y & 0x3fffffffu)), ar, R);
        T ja = *reinterpret_cast<const T*>(avb + (sc.x & 0xffffu));
        T diag = iwu;
        if (has2) { ja -= *reinterpret_cast<const T*>(avb + o2); diag += iwu; }
        u = keep ? -ja : -ar;
        n = T(-1) / (diag + R);
      }
      tm_st2(tcol, u, n);
    }
    tm_wait_st();
  }
  // the u's back into the compact shared-memory pairs (debug dump only; every lane of the warp takes part)
  __device__ void rows_from_tm() {
    char* rwb = reinterpret_cast<char*>(hot);
    constexpr unsigned CW = TmPair<T>::cols;
    for (int st = 0; st < D.nstep; st++) {
      const Slot<T> sc = ld_slot<T>(slots + st * LPW);
      T u, n; tm_ld2(tm + (unsigned)st * CW, u, n); tm_wait_ld(u, n);
      if (sc.y & 0x40000000u) *reinterpret_cast<T*>(rwb + (sc.y & 0x3fffffffu)) = u;
    }
    __syncwarp();
  }
  __device__ __forceinline__ T equality_sweep(Tendon& tn, bool done) {
    const int ns = D.ns;
    T* av = a() + D.nfd;
    // worlds stop sweeping one by one (rarely before the last sweep): the gated loop is only taken by a warp that
    // holds a finished world
    T impr;
    if (K.tm_cols) impr = __any_sync(FULLMASK, done) ? equality_rows<true, true>(done) : equality_rows<false, true>(false);
    else impr = __any_sync(FULLMASK, done) ? equality_rows<true>(done) : equality_rows<false>(false);
    // volume-tendon row: dense over the shell, sub-warp shuffle reduction
    {
      T s = 0;
#pragma unroll 4
      for (int e = sl; e < ns; e += LPW) s += av[e];            // tendon coefficients are all 1
      s = gsum(s);
      const T res = s + tn.u;
      const T dl = done ? T(0) : res * tn.nA;
      if (sl == 0) impr -= T(0.5) * dl * res;
      tn.u += tn.R * dl;
      const T da = stim[0] * dl;
#pragma unroll 4
      for (int e = sl; e < ns; e += LPW) av[e] += da;
      __syncwarp();
    }
    return impr;
  }

  // projected Gauss-Seidel (mj_solPGS) in MuJoCo's row order.
  // (A "team mode" in which one warp swept the limit/contact rows of 16 worlds through a 2-lane view between named
  // barriers was measured slower twice and removed; see DESIGN.md and the history.)
  __device__ void pgs(Tendon& tn, unsigned char* smem) {
    int iter = 0;
    bool done = false;
    {
      ChainState cs;
      chain_prologue(cs);
      const int tmaxw = wmax(misc(M2_TMAX));
      __syncwarp();
      tick(PH_PGS_SETUP);
      for (int it = 0; it < D.iters; it++) {
        if (!__any_sync(FULLMASK, !done)) break;
        T impr = equality_sweep(tn, done);
        tick(PH_PGS_EQUALITY);
        impr += K.rec_ring ? chain_phase<true>(cs, tmaxw, done) : chain_phase<false>(cs, tmaxw, done);
        tick(PH_PGS_CHAIN);
        impr = gsum(impr) * C.impr_scale;
        if (!done) { iter++; if (impr < C.tol) done = true; }
      }
      chain_epilogue(cs);
    }
    if (K.rec_ring) cp_wait();     // (a record requested for a sweep that did not happen)
    if (sl == 0) misc(M2_ITERS) = iter;
    __syncwarp();
  }

  // ------------------------------------------------------------------------------------------
  // mj_forward for this world; returns true if qacc is bad
  // ------------------------------------------------------------------------------------------
  __device__ bool forward() {
    Tendon tn; ChainRows cr; T Ft;
    tick(PH_OTHER);
    if (sl < D.nchain) gripper(sl);
    __syncwarp();
    tick(PH_GRIPPER);
    collide();
    tick(PH_COLLIDE);
    rows_and_smooth(tn, Ft);
    if (sl < D.nchain) chain_limits(sl, cr); else cr.lmask = 0;
    tick(PH_ROWS);
    warmstart(tn, cr);
    tick(PH_WARMSTART);
    pgs(tn, smem_base);
    // accelerometers (mj_sensorAcc): R_site^T (Jv qacc + bias - g)
    for (int s = sl; s < D.nsens; s += LPW) {
      const T* se = tab(D.o_sens + s * SE_STRIDE);
      if ((int)se[SE_TYPE] == SENS_ACCEL) {
        const int c = (int)se[SE_CHAIN], d0 = D.chain_dof0[c], adr = (int)se[SE_ADR];
        T acc[3] = {aux[L.s_ab + 3 * s], aux[L.s_ab + 3 * s + 1], aux[L.s_ab + 3 * s + 2]};
        for (int jj = 0; jj < D.ncd[c]; jj++) {
          const T aj = a()[d0 + jj];
#pragma unroll
          for (int k = 0; k < 3; k++) acc[k] += aux[L.s_jv + 12 * s + 3 * jj + k] * aj;
        }
        T o[3]; matTvec3(o, aux + L.s_rot + 9 * s, acc);
#pragma unroll
        for (int k = 0; k < 3; k++) aux[L.sens + adr + k] = o[k];
      }
    }
    {
      int s = (sl < D.nchain) ? __popc((unsigned)misc(M2_LMASK + sl)) : 0;
#pragma unroll
      for (int o = LPW / 2; o > 0; o >>= 1) s += __shfl_xor_sync(FULLMASK, s, o);
      if (sl == 0) misc(M2_NLIM) = s;
    }
    __syncwarp();
    tick(PH_SENSORS);
    if (K.tm_cols && K.debug_out && __any_sync(FULLMASK, valid && w == K.debug_world)) rows_from_tm();
    if (valid && w == K.debug_world) debug_dump(tn);
    bool badacc = false;
    for (int i = sl; i < D.nv; i += LPW) if (!(tabs(a()[i]) <= T(SG_MAXVAL))) badacc = true;
    __syncwarp();
    return gballot(badacc) != 0u;
  }

  // mj_Euler with implicit joint damping: (M + h diag(d)) qacc' = qfrc_smooth + J^T f = M qacc
  __device__ void euler() {
    const int nfd = D.nfd; const T h = C.h;
    {
      T* __restrict__ qp = pin_g(q() + nfd); T* __restrict__ vp = pin_g(v() + nfd);
      const T* __restrict__ ap = pin_s(a() + nfd);
      struct EuV { T m, d, v, q; };
      batched<8, EuV>(sl, D.ns, LPW,
        [&](int e, EuV& x) SG_INL { x.m = tab(D.o_sl_m)[e]; x.d = damping(e); x.v = vp[e]; x.q = qp[e]; },
        [&](int e, const EuV& x) SG_INL {
          const T qa = x.m * ap[e] / (x.m + h * x.d);
          const T vn = x.v + h * qa;
          vp[e] = vn; qp[e] = x.q + h * vn;
        });
    }
    for (int i = sl; i < nfd; i += LPW) { const T vn = v()[i] + h * a()[i]; v()[i] = vn; q()[i] += h * vn; }
    if (sl < D.nu) aux[L.act + sl] += h * aux[L.actdot + sl];
    __syncwarp();
  }

  // mj_step (integrate) or mj_forward (!integrate).  forward() is inlined exactly once: the kernel is one loop over
  // physics steps around this function, so the whole step stays a few thousand instructions (instruction cache).
  __device__ void step(bool integrate) {
    if (integrate) {
      bool badpv = false;
      batched<8, V2<T>>(sl, D.nv, LPW, [&](int i, V2<T>& x) SG_INL { x.a = q()[i]; x.b = v()[i]; },
                        [&](int, const V2<T>& x) SG_INL { if (!(tabs(x.a) <= T(SG_MAXVAL)) || !(tabs(x.b) <= T(SG_MAXVAL))) badpv = true; });
      const bool gbad = gballot(badpv) != 0u;
      if (gbad && sl == 0) misc(M2_STATUS) |= 1;
      // reset_if contains a warp collective: every group goes through it, only the bad ones write
      reset_if(gbad);
      T* a0 = aux + L.a0;
      for (int i = sl; i < D.nv; i += LPW) a0[i] = a()[i];
    }
    for (int pass = 0; pass < 2; pass++) {
      const bool bad = forward();
      // CTA-uniform decision when the warps step together (per-step barrier)
      if (!integrate || !cta_any(bad)) break;
      // mj_step re-runs mj_forward after mj_resetData.  forward() is full of warp collectives, so the other
      // groups of the warp re-run it too, from their saved warm start: they recompute identical values.
      if (bad && sl == 0) misc(M2_STATUS) |= 1;
      if (pass == 0 && !bad) { const T* a0 = aux + L.a0; for (int i = sl; i < D.nv; i += LPW) a()[i] = a0[i]; }
      reset_if(bad);
    }
    if (integrate) { tick(PH_OTHER); euler(); tick(PH_EULER); }
  }
  __device__ __forceinline__ bool cta_any(bool p) const {
    // without the per-step barrier the warps of a CTA never wait for each other: the decision
    // only has to be uniform over the warp (forward() is full of warp collectives)
    if (blockDim.x > 32 && K.step_barrier) return __syncthreads_or(p ? 1 : 0) != 0;
    return __any_sync(FULLMASK, p) != 0;
  }
  __device__ void reset_if(bool doit) {
    if (doit) {
      for (int i = sl; i < D.nv; i += LPW) { q()[i] = 0; v()[i] = 0; a()[i] = 0; }
      if (sl == 0) a()[D.nv] = 0;      // dummy slider of the level sweep
      if (sl < D.nu) { aux[L.act + sl] = 0; aux[L.ctrl + sl] = 0; }
    }
    __syncwarp();
  }

  __device__ void debug_dump(const Tendon& tn) {
    // header: [0]=ncon_total [1]=nefc [2]=iters [3]=ncon(rows) [4]=nlim [5]=tmax [6]=ncand ; contacts at 64+16*i ;
    // then at 64+16*maxcon*2: qacc[nv], efc_force / aref / R (equality block in schedule order, then MuJoCo order);
    // the last nrow+1 doubles of the buffer hold the equality arefs written by rows_and_smooth, the nrow+1 before them the R's
    double* o = K.debug_out;
    if (!o) return;
    const int ncon = misc(M2_NCON), nlim = misc(M2_NLIM);
    const int nefc = D.nrow + 1 + nlim + 3 * ncon;
    if (sl == 0) { o[0] = misc(M2_NCONTOT); o[1] = nefc; o[2] = misc(M2_ITERS); o[3] = ncon; o[4] = nlim; o[5] = misc(M2_TMAX); o[6] = misc(M2_NCAND); }
    const int base = 64 + 16 * 2 * D.maxcon;
    for (int i = sl; i < D.nv; i += LPW) if (base + i < K.debug_cap) o[base + i] = (double)a()[i];
    const int eb = base + D.nv;
    const int tail = K.debug_cap - (D.nrow + 1), tailR = tail - (D.nrow + 1);
    if (eb + 3 * nefc > tailR) return;
    const T* row2 = hot + L.row2;
    for (int p = sl; p < D.nrow; p += LPW) {
      const double ar = o[tail + p], R = o[tailR + p];
      o[eb + p] = ((double)row2[2 * p] + ar) / R; o[eb + nefc + p] = ar; o[eb + 2 * nefc + p] = R;
    }
    if (sl == 0) {
      int r = D.nrow;
      o[eb + r] = ((double)tn.u + (double)tn.aref) / (double)tn.R; o[eb + nefc + r] = (double)tn.aref; o[eb + 2 * nefc + r] = (double)tn.R; r++;
      for (int c = 0; c < D.nchain; c++)
        for (int jl = 0; jl < D.ncd[c]; jl++)
          if (misc(M2_LMASK + c) & (1 << jl)) {
            const int dof = D.chain_dof0[c] + jl;
            o[eb + r] = (double)lf(dof); o[eb + nefc + r] = (double)laref(dof); o[eb + 2 * nefc + r] = (double)lR(dof); r++;
          }
      for (int i = 0; i < ncon; i++)
        for (int k = 0; k < 3; k++, r++) {
          const T* cr = crec(i);
          o[eb + r] = (double)cr[CR_F + k]; o[eb + nefc + r] = (double)cr[CR_AREF + k];
          o[eb + 2 * nefc + r] = (double)(k ? cr[CR_R0] * C.inv_impratio : cr[CR_R0]);
        }
    }
  }
};

// ---------------------------------------------------------------------------------------------
// kernel
// ---------------------------------------------------------------------------------------------
#ifndef SG_SHARED_BYTES
#define SG_SHARED_BYTES(name) extern __shared__ __align__(16) unsigned char name[]
#endif

// A CTA holds 1..SG_MAX_WARPS warps (blockDim.x / 32, chosen by the host).  Warps never exchange data: the CTA exists so
// that (i) the level-sweep step tables are staged in shared memory once and shared by all its worlds and (ii) its
// warps start every physics step together (one __syncthreads per step), which keeps them in the same region of the
// large straight-line set-up code and therefore in the same instruction-cache lines.
#ifndef SG_MAX_WARPS
#define SG_MAX_WARPS 16
#endif
#ifndef SG_MIN_CTAS
#define SG_MIN_CTAS 1
#endif
template <typename T, int LPW>
__global__ void __launch_bounds__(32 * SG_MAX_WARPS, SG_MIN_CTAS) sg_step_kernel2(const __grid_constant__ KArgs2<T> K) {
  SG_SHARED_BYTES(smem_raw);
  constexpr int WPW = 32 / LPW;
  const PlanDims& D = K.D;
  const Layout2& L = K.L;
  const int lane = threadIdx.x & 31, grp = lane / LPW, sl = lane % LPW;
  const int warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
  // tensor memory for the (u, n) rows of the equality sweep (see tm_ld2): warp 0 allocates K.tm_cols columns for the CTA
  unsigned tm_window = 0;
#if defined(__CUDA_ARCH__)
  __shared__ unsigned tm_base_s;
  if (K.tm_cols && warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(&tm_base_s)), "r"(K.tm_cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  }
#endif
  {
    // stage the step tables: one descriptor slot per (step, lane)
    Slot<T>* ss = reinterpret_cast<Slot<T>*>(smem_raw);
    const int nslot = (D.nstep + 1) * LPW;
    for (int i = threadIdx.x; i < nslot; i += blockDim.x) {
      Slot<T> t; t.x = (unsigned)K.itab[D.io_step_d + 2 * i]; t.y = (unsigned)K.itab[D.io_step_d + 2 * i + 1];
      ss[i] = t;
    }
    T* tc = reinterpret_cast<T*>(smem_raw + (size_t)nslot * sizeof(Slot<T>));
    for (int i = threadIdx.x; i < D.ns; i += blockDim.x) { tc[i] = K.tab[D.o_sl_tc + i]; tc[D.ns + i] = K.tab[D.o_sl_tciw + i]; tc[2 * D.ns + i] = T(1) / K.tab[D.o_sl_m + i]; }
    T* ax = tc + 3 * D.ns;
    for (int i = threadIdx.x; i < 3 * D.ns; i += blockDim.x) ax[i] = K.tab[D.o_sl_axis + i];
    T* cl = ax + 3 * D.ns;
    for (int i = threadIdx.x; i < MAXCOLL * CO_STRIDE; i += blockDim.x) cl[i] = K.tab[D.o_coll + i];
    int* rn = reinterpret_cast<int*>(cl + MAXCOLL * CO_STRIDE);
    for (int i = threadIdx.x; i < 4 * D.nrun; i += blockDim.x) rn[i] = K.itab[D.io_run + i];
    for (int i = threadIdx.x; i < D.nrow; i += blockDim.x) rn[4 * D.nrun + i] = K.itab[D.io_row_d12 + i];
    __syncthreads();
  }
  if (K.tm_cols) {
#if defined(__CUDA_ARCH__)
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    tm_window = tm_base_s;
#endif
    tm_window += ((unsigned)((warp & 3) * 32) << 16) + (unsigned)((warp >> 2) * K.tm_stride);
  }
#if defined(__CUDA_ARCH__)
  if (K.prof && lane == 0) K.prof[PH_COUNT + (size_t)blockIdx.x * nwarp + warp] = clock64();
#endif
  const int cta_worlds = nwarp * WPW;
  // Persistent CTAs.  Episodes differ in length of their contact phase, so the batches are handed out dynamically: a CTA
  // that finishes early takes the next batch instead of idling behind a fixed share (65 536 worlds are 6.9 batches per
  // CTA).  Which CTA simulates a world does not enter its arithmetic: results are identical to the static order.
#if defined(__CUDA_ARCH__)
  __shared__ int next_batch_s;
#else
  static int next_batch_s;
#endif
  for (int it = 0;; it++) {
    if (K.batch_counter) {
      if (threadIdx.x == 0) next_batch_s = atomicAdd(K.batch_counter, 1);
      __syncthreads();
    }
    const int b0 = (K.batch_counter ? next_batch_s : it * (int)gridDim.x + (int)blockIdx.x) * cta_worlds;
    if (K.batch_counter) __syncthreads();          // everybody has read the batch before thread 0 fetches the next one
    if (b0 >= K.nworlds) break;
    const int wi = b0 + warp * WPW + grp;
    const bool valid = wi < K.nworlds;
    World2<T, LPW> W(K, smem_raw, valid ? wi : K.nworlds - 1, valid);
    W.tm = tm_window;
    W.load_params();
    if (sl == 0) { W.misc(M2_STATUS) = 0; W.a()[D.nv] = 0; W.hot[L.row2 + 2 * D.nrow] = 0; W.hot[L.row2 + 2 * D.nrow + 1] = -1; }
    const int w = W.w;
    const size_t sb = (size_t)w * D.nv;
    T* aux = W.aux;
    if (sl < D.nu) { aux[L.act + sl] = K.act[(size_t)w * D.nu + sl]; aux[L.ctrl + sl] = K.ctrl[(size_t)w * D.nu + sl]; }
    if (!K.rollout) {
      for (int i = sl; i < D.nv; i += LPW) { W.q()[i] = K.qpos[sb + i]; W.v()[i] = K.qvel[sb + i]; W.a()[i] = K.warm[sb + i]; }
      __syncwarp();
    } else W.reset_if(true);     // whole episode on-chip (create_dataset.log_into_file, ref: create_dataset.py:33-60)
    const int total = K.rollout ? K.sim_start + K.nrows * K.sim_step : (K.integrate ? K.nsub : 1);
    // rollout: pass s = -1 is the mj_forward of ManEnv.reset (ref: manenv.py:57-58 sim.reset(); sim.forward()).  It moves no
    // state but, like every mj_forward, leaves its qacc as the warm start of the first step (mj_fwdConstraint saves it).
    for (int s = K.rollout ? -1 : 0; s < total; s++) {
      if (nwarp > 1 && K.step_barrier) __syncthreads();     // warps start each step together (instruction-cache locality, see above)
      int t = -1, phase = 0;
      if (K.rollout && s >= K.sim_start) {
        const int r = s - K.sim_start;
        t = r / K.sim_step; phase = r - t * K.sim_step;
        if (phase == 0) {
          if (K.ctrl_event[t] && sl < D.nu) aux[L.ctrl + sl] = T(K.ctrl_value[t * D.nu + sl]);
          __syncwarp();
        }
      }
      W.step(s >= 0 && (K.rollout || K.integrate));
      if (t >= 0 && phase == K.sim_step - 1 && valid) {
        // sensor row of this env-step (ref: manenv.py:85 np.copy(sensordata)).  World-major: one world's row is 12
        // consecutive values, written as 128-bit vectors by the first lanes of the world; SoA: channel-major planes with
        // the world index fastest, the worlds of a warp / CTA land in the same 32-byte sectors.
        if (K.traj_soa) {
          for (int i = sl; i < D.nsd; i += LPW) K.sens_out[((size_t)t * D.nsd + i) * K.nworlds + w] = aux[L.sens + i];
        } else if ((D.nsd & 3) == 0) {
          T* row = K.sens_out + ((size_t)w * K.nrows + t) * D.nsd;
          for (int i = 4 * sl; i < D.nsd; i += 4 * LPW) { T x[4]; ld4(aux + L.sens + i, x); st4(row + i, x[0], x[1], x[2], x[3]); }
        } else {
          for (int i = sl; i < D.nsd; i += LPW) K.sens_out[((size_t)w * K.nrows + t) * D.nsd + i] = aux[L.sens + i];
        }
        if (K.touch_out && sl == 0) K.touch_out[(size_t)w * K.nrows + t] = W.misc(M2_TOUCH);
      }
    }
    // (a forward-only launch stores its qacc as the next warm start as well: mj_fwdConstraint saves it on every mj_forward)
    if (valid) {
      for (int i = sl; i < D.nv; i += LPW) { K.qpos[sb + i] = W.q()[i]; K.qvel[sb + i] = W.v()[i]; K.warm[sb + i] = W.a()[i]; }
      if (!K.rollout) {
        if (K.sens_out) for (int i = sl; i < D.nsd; i += LPW) K.sens_out[(size_t)w * D.nsd + i] = aux[L.sens + i];
        if (K.touch_out && sl == 0) K.touch_out[w] = W.misc(M2_TOUCH);
      }
    }
    __syncwarp();
    if (valid) {
      if (sl < D.nu) { K.act[(size_t)w * D.nu + sl] = aux[L.act + sl]; K.ctrl[(size_t)w * D.nu + sl] = aux[L.ctrl + sl]; }
      if (sl == 0 && W.misc(M2_STATUS)) atomicOr(&K.status[w], W.misc(M2_STATUS));
    }
    __syncwarp();
  }
#if defined(__CUDA_ARCH__)
  if (K.tm_cols) {
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tm_base_s), "r"(K.tm_cols) : "memory");
  }
#endif
}

}  // namespace sg
