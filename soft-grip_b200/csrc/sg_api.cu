// sg_api.cu -- C-ABI of libsoftgrip.so (include/softgrip.h): model/plan upload, batch state in HBM,
// kernel launches.  Host logic only; all physics is in sg_kernels2.cuh.  There is no CPU fallback: every
// entry point that would compute needs a CUDA device and fails with an error otherwise.
#include "sg_rt.hpp"

#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/softgrip.h"
#include "sg_plan.hpp"
#include "sg_launch.hpp"
#include "sg_traj.cuh"

using namespace sg;

static thread_local std::string g_err;
static int fail(const std::string& msg) { g_err = msg; return -1; }
#define CUDA_OK(expr) do { cudaError_t e_ = (expr); if (e_ != cudaSuccess) return fail(std::string(#expr) + ": " + cudaGetErrorString(e_)); } while (0)

struct sg_model {
  Plan plan;
  int maxcon_default, maxcand_default;
};

struct sg_batch {
  const sg_model* model;
  PlanDims D;                 // with per-batch capacities and masks folded in
  int W, device, precision;
  size_t esize;
  int lpw = 8;                // lanes per world
  int nwarp = 16;             // warps per CTA
  int tm_cols = 0, tm_stride = 0;   // tensor-memory window of the equality rows (KArgs2::tm_cols, tm_stride); 0: shared memory
  int rec_ring = 0;                 // contact records through a shared-memory ring in the freed row region (KArgs2::rec_ring)
  size_t smem2 = 0;           // dynamic shared memory per CTA
  Layout2 L2;
  unsigned char* scratch = nullptr;   // global aux slots of the worlds (KArgs2::scratch)
  std::vector<int> step_d;            // level-sweep step tables for this batch's lanes per world
  std::vector<int> row_perm;          // plan schedule position -> storage position of the row in this batch's kernel tables
  void* tab = nullptr;        // device table in batch precision
  int* itab = nullptr;
  void *qpos = nullptr, *qvel = nullptr, *warm = nullptr, *act = nullptr, *ctrl = nullptr;
  double *p_stiff = nullptr, *p_damp = nullptr, *p_tdamp = nullptr, *p_objoff = nullptr;   // owned copies
  bool has_stiff = false, has_damp = false, has_tdamp = false, has_objoff = false;
  int* status = nullptr;
  int* d_ctrl_event = nullptr; double* d_ctrl_value = nullptr; int sched_cap = 0;
  double* debug_out = nullptr; int debug_cap = 0, debug_world = -1;
  void* stage_traj = nullptr; size_t stage_traj_bytes = 0;   // device staging for rollout_host
  int* stage_touch = nullptr; size_t stage_touch_bytes = 0;
  long long launches = 0;
  int traj_soa = 0;           // trajectory layout of sg_batch_rollout: 0 = [W][T][C], 1 = [T][C][W]
  unsigned long long* prof = nullptr; size_t prof_n = 0;   // SOFTGRIP_PROF=1: phase clocks of the step kernel (development aid)
  int* batch_counter = nullptr;     // KArgs2::batch_counter (dynamic hand-out of world batches to the persistent CTAs)
  int max_ctas = 0, per_sm = 0;
};

extern "C" const char* sg_last_error(void) { return g_err.c_str(); }
extern "C" int sg_version(void) { return 1; }

extern "C" int sg_model_load(const void* blob, size_t nbytes, sg_model** out) {
  if (!blob || !out) return fail("sg_model_load: null argument");
  try {
    sg_model* m = new sg_model();
    m->plan = build_plan(blob, nbytes);
    const int ns = m->plan.d.ns;
    int mc = ((ns * 3 / 4 + 15) / 16) * 16;
    if (mc < 32) mc = 32;
    if (mc > 128) mc = 128;
    if (const char* e = std::getenv("SOFTGRIP_MAXCON")) mc = std::atoi(e);
    if (mc > 255) mc = 255;             // contact index and time slot are 8-bit fields of the schedule entries
    if (mc < 1) mc = 1;
    m->maxcon_default = mc;
    m->maxcand_default = 256;
    if (const char* e = std::getenv("SOFTGRIP_MAXCAND")) m->maxcand_default = std::atoi(e);
    *out = m;
    return 0;
  } catch (const std::exception& e) { return fail(e.what()); }
}

extern "C" void sg_model_destroy(sg_model* m) { delete m; }

extern "C" int sg_model_info(const sg_model* m, sg_info* out) {
  if (!m || !out) return fail("sg_model_info: null argument");
  std::memset(out, 0, sizeof(*out));
  PlanDims D = m->plan.d;
  D.maxcon = m->maxcon_default; D.maxcand = m->maxcand_default;
  out->nv = D.nv; out->nfinger = D.nfd; out->nshell = D.ns; out->neq = m->plan.neq; out->nu = D.nu; out->nsensordata = D.nsd;
  out->nlevels = D.nlev; out->maxcon = D.maxcon; out->ngeom = m->plan.ngeom;
  out->smem_bytes32 = make_layout2<float>(D, 4, 8).smem_stride; out->smem_bytes64 = make_layout2<double>(D, 4, 8).smem_stride;
  return 0;
}

extern "C" int sg_model_set_stiffness_targets(sg_model* m, const int* joint_mask, int tendon0) {
  if (!m || !joint_mask) return fail("sg_model_set_stiffness_targets: null argument");
  PlanDims& D = m->plan.d;
  for (int i = 0; i < D.nfd; i++) if (joint_mask[i]) return fail("stiffness targets must be shell joints");
  for (int e = 0; e < D.ns; e++) m->plan.itab[D.io_kmask + e] = joint_mask[D.nfd + e] ? 1 : 0;
  D.stiff_tendon0 = tendon0 ? 1 : 0;
  return 0;
}

extern "C" int sg_model_set_geom_mask(sg_model* m, const int* mask) {
  if (!m || !mask) return fail("sg_model_set_geom_mask: null argument");
  Plan& P = m->plan;
  P.geom_mask.assign(mask, mask + P.ngeom);
  for (size_t c = 0; c < P.coll_geom.size(); c++) P.tab[P.d.o_coll + c * CO_STRIDE + CO_MASK] = mask[P.coll_geom[c]];
  P.d.cap_mask = 0;
  for (int e = 0; e < P.d.ns; e++) P.d.cap_mask = (double)((int)P.d.cap_mask | mask[P.first_capsule_geom + e]);
  for (int e = 0; e < P.d.ns; e++) if (mask[P.first_capsule_geom + e] != (int)P.d.cap_mask) return fail("shell geoms must share one name mask");
  P.d.sph_mask = P.center_geom >= 0 ? mask[P.center_geom] : 0;
  return 0;
}

// device tables = the model's plan tables + this batch's level-sweep step tables (which depend on lanes per world)
static void host_tables(const sg_batch* b, std::vector<double>& tab, std::vector<int>& itab) {
  const Plan& P = b->model->plan;
  tab = P.tab; itab = P.itab;
  // the kernel stores the equality rows at the positions its step schedule chose (bank-conflict-free steps)
  const PlanDims& D = P.d;
  const std::vector<int>& perm = b->row_perm;
  for (int p = 0; p < D.nrow; p++) {
    const int q = perm[p];
    itab[D.io_row_d1 + q] = P.itab[D.io_row_d1 + p]; itab[D.io_row_d2 + q] = P.itab[D.io_row_d2 + p];
    itab[D.io_row_d12 + q] = P.itab[D.io_row_d12 + p];
    tab[D.o_row_iw + 2 * q] = P.tab[D.o_row_iw + 2 * p]; tab[D.o_row_iw + 2 * q + 1] = P.tab[D.o_row_iw + 2 * p + 1];
  }
  // rows of each slider for the warm start: row position | other slider << 12 (0xfff: none) | "second slider" << 24
  for (int i = 0; i < D.ns * MAXDOFROWS; i++) {
    const int code = P.itab[D.io_dof_rows + i];
    if (code < 0) continue;
    const int p = code >> 1, second = code & 1;
    const int d1 = P.itab[D.io_row_d1 + p], d2 = P.itab[D.io_row_d2 + p];
    const int other = second ? d1 : (d2 >= 0 ? d2 : 0xfff);
    itab[D.io_dof_rows + i] = perm[p] | (other << 12) | (second << 24);
  }
  while (itab.size() % 4) itab.push_back(0);
  itab.insert(itab.end(), b->step_d.begin(), b->step_d.end());
}

static int upload_tables(sg_batch* b, bool allocate) {
  std::vector<double> tab; std::vector<int> itab;
  host_tables(b, tab, itab);
  if (allocate) {
    CUDA_OK(cudaMalloc(&b->tab, b->esize * (tab.size() ? tab.size() : 1)));
    CUDA_OK(cudaMalloc((void**)&b->itab, sizeof(int) * (itab.size() ? itab.size() : 1)));
  }
  if (b->precision == 32) {
    std::vector<float> t(tab.size());
    for (size_t i = 0; i < t.size(); i++) t[i] = (float)tab[i];
    CUDA_OK(cudaMemcpy(b->tab, t.data(), sizeof(float) * t.size(), cudaMemcpyHostToDevice));
  } else CUDA_OK(cudaMemcpy(b->tab, tab.data(), sizeof(double) * tab.size(), cudaMemcpyHostToDevice));
  CUDA_OK(cudaMemcpy(b->itab, itab.data(), sizeof(int) * itab.size(), cudaMemcpyHostToDevice));
  return 0;
}

// (precision, lanes-per-world) -> instantiation; the list must match the Makefile's SG_INSTANCES
#ifdef SG_SMALL_BUILD
#define SG_K2_CASES(X) X(float, 8) X(double, 8)
#else
#define SG_K2_CASES(X) X(float, 4) X(float, 8) X(float, 16) X(float, 32) X(double, 4) X(double, 8) X(double, 16) X(double, 32)
#endif
static int k2_dispatch_configure(int precision, int lpw, int block, size_t smem, int* per_sm) {
#define X(T, N) if ((precision == 32) == (sizeof(T) == 4) && lpw == N) return k2_configure<T, N>(block, smem, per_sm);
  SG_K2_CASES(X)
#undef X
  return -12345;
}
template <typename T>
static int k2_dispatch_launch(int lpw, const KArgs2<T>& K, int grid, int block, size_t smem, void* stream) {
#define X(TT, N) if (sizeof(TT) == sizeof(T) && lpw == N) return k2_launch<T, N>(K, grid, block, smem, stream);
  SG_K2_CASES(X)
#undef X
  return -12345;
}

extern "C" void sg_batch_destroy(sg_batch* b);
static int batch_create_body(const sg_model* m, int nworlds, int device, int precision, sg_batch*& b);
extern "C" int sg_batch_create(const sg_model* m, int nworlds, int device, int precision, sg_batch** out) {
  if (!m || !out) return fail("sg_batch_create: null argument");
  *out = nullptr;
  sg_batch* b = nullptr;
  const int rc = batch_create_body(m, nworlds, device, precision, b);
  if (rc) { if (b) sg_batch_destroy(b); return rc; }      // every failure path frees the handle and what it already owns
  *out = b;
  return 0;
}
static int batch_create_body(const sg_model* m, int nworlds, int device, int precision, sg_batch*& b) {
  if (nworlds < 1) return fail("sg_batch_create: nworlds must be >= 1");
  if (precision != 32 && precision != 64) return fail("sg_batch_create: precision must be 32 or 64");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) return fail("sg_batch_create: no CUDA device available (libsoftgrip has no CPU path)");
  if (device < 0 || device >= ndev) return fail("sg_batch_create: bad device index");
  CUDA_OK(cudaSetDevice(device));
  b = new sg_batch();
  b->model = m; b->W = nworlds; b->device = device; b->precision = precision;
  b->esize = precision == 32 ? 4 : 8;
  b->D = m->plan.d;
  b->D.maxcon = m->maxcon_default; b->D.maxcand = m->maxcand_default;
  cudaDeviceProp prop;
  CUDA_OK(cudaGetDeviceProperties(&prop, device));
  // launch configuration (environment overrides are development knobs; the defaults are the measured best)
  // lanes per world: 8 for the committed models (measured best for softbox, softball; within 9 % for softcylinder), 32 for
  // shells beyond 256 elements, where shared memory leaves few worlds per SM and the equality sweep is twice as long at 8
  // lanes (softbox_refined, 434 elements: 1.11e6 / 1.48e6 / 1.72e6 world-steps/s at 8 / 16 / 32 lanes, profiles/r02a_*)
  b->lpw = b->D.ns > 256 ? 32 : 8; b->nwarp = 16;
  if (const char* e = std::getenv("SOFTGRIP_LPW")) b->lpw = std::atoi(e);
  if (const char* e = std::getenv("SOFTGRIP_NW")) b->nwarp = std::atoi(e);
  int aux_in_smem = 0, qv_in_smem = 0;
  if (const char* e = std::getenv("SOFTGRIP_QV_SMEM")) qv_in_smem = std::atoi(e);
  if (const char* e = std::getenv("SOFTGRIP_AUX_SMEM")) aux_in_smem = std::atoi(e);
  if (aux_in_smem || qv_in_smem) {
    return fail("SOFTGRIP_AUX_SMEM / SOFTGRIP_QV_SMEM: the shared-memory placement of the once-per-step data was removed from the step kernel (measured slower; a single address space lets the compiler emit global loads)");
  }
  if (b->nwarp < 1 || b->nwarp > SG_MAX_WARPS) { return fail("SOFTGRIP_NW must be 1..16"); }
  if (b->lpw != 4 && b->lpw != 8 && b->lpw != 16 && b->lpw != 32) { return fail("SOFTGRIP_LPW must be 4, 8, 16 or 32"); }
  const Plan& P = m->plan;
  build_step_tables(b->D, P.itab, b->lpw, (int)b->esize, b->step_d, b->row_perm, std::getenv("SOFTGRIP_NO_BANK_SCHEDULE") == nullptr);
  b->D.nstep = (int)(b->step_d.size() / (2 * (size_t)b->lpw)) - 1;   // without the trailing dummy step
  b->D.io_step_d = (int)((P.itab.size() + 3) / 4 * 4);
  int rc = upload_tables(b, true);
  if (rc) { return rc; }
  const size_t nv = b->D.nv, nu = b->D.nu > 0 ? b->D.nu : 1;
  CUDA_OK(cudaMalloc(&b->qpos, b->esize * nv * nworlds));
  CUDA_OK(cudaMalloc(&b->qvel, b->esize * nv * nworlds));
  CUDA_OK(cudaMalloc(&b->warm, b->esize * nv * nworlds));
  CUDA_OK(cudaMalloc(&b->act, b->esize * nu * nworlds));
  CUDA_OK(cudaMalloc(&b->ctrl, b->esize * nu * nworlds));
  CUDA_OK(cudaMalloc((void**)&b->status, sizeof(int) * nworlds));
  CUDA_OK(cudaMalloc((void**)&b->p_stiff, sizeof(double) * nworlds));
  CUDA_OK(cudaMalloc((void**)&b->p_damp, sizeof(double) * nworlds));
  CUDA_OK(cudaMalloc((void**)&b->p_tdamp, sizeof(double) * nworlds));
  CUDA_OK(cudaMalloc((void**)&b->p_objoff, sizeof(double) * 3 * nworlds));
  b->debug_cap = 64 + 16 * 2 * b->D.maxcon + b->D.nv + 3 * (b->D.nrow + 1 + MAXFD + 3 * b->D.maxcon) + 64 + 2 * (b->D.nrow + 1);
  CUDA_OK(cudaMalloc((void**)&b->debug_out, sizeof(double) * b->debug_cap));
  CUDA_OK(cudaMemset(b->debug_out, 0, sizeof(double) * b->debug_cap));
  const int wpw = 32 / b->lpw;
  // Launch geometry.  Warps never exchange data, and the kernel is bound by the dependent-issue latency of each warp
  // (profiles/r02c_phase_scan.txt: 1.05e6 cycles per warp-step with one warp per SM, 1.58e6 with sixteen), so what
  // counts is (i) every SM busy and (ii) as few passes over the batch list as possible.  Among the CTA sizes that fit,
  // take the one with the smallest modelled time  passes * (1 + 0.035 (resident warps - 1));  several small CTAs per SM
  // are penalised: their warps do not share the per-step barrier, which costs instruction-cache locality
  // (profiles/r01s_*).  E.g. 8 192 worlds (BASELINE configs[2] on 8 GPUs) run as 147 CTAs of 56 worlds instead of
  // 128 CTAs of 64 on 148 SMs.
  const bool nw_forced = std::getenv("SOFTGRIP_NW") != nullptr;
  int best_nw = 0; double best_cost = 0;
  for (int nw = nw_forced ? b->nwarp : SG_MAX_WARPS; nw >= (nw_forced ? b->nwarp : 1); nw--) {
    const Layout2 L = precision == 32 ? make_layout2<float>(b->D, wpw, b->lpw) : make_layout2<double>(b->D, wpw, b->lpw);
    const size_t smem = (size_t)L.smem_tables + (size_t)L.smem_stride * wpw * nw;
    if (smem > prop.sharedMemPerBlockOptin) continue;
    int ps = 0;
    const int e = k2_dispatch_configure(precision, b->lpw, 32 * nw, smem, &ps);
    if (e == -12345) { return fail("SOFTGRIP_LPW: this lanes-per-world value is not compiled in"); }
    if (e) { return fail(std::string("kernel configuration failed: ") + cudaGetErrorString((cudaError_t)e)); }
    if (ps < 1) continue;
    const long ctas = ((long)nworlds + nw * wpw - 1) / (nw * wpw);
    const long resident = (long)ps * prop.multiProcessorCount;
    const long passes = (ctas + resident - 1) / resident;
    const long per_sm_used = ctas < resident ? (ctas + prop.multiProcessorCount - 1) / prop.multiProcessorCount : ps;
    double cost = (double)passes * (1.0 + 0.035 * (double)(per_sm_used * nw - 1));
    if (per_sm_used > 1) cost *= 1.3;
    if (!best_nw || cost < best_cost * (1.0 - 1e-9)) { best_nw = nw; best_cost = cost; }
  }
  if (!best_nw) { return fail("sg_batch_create: worlds of one warp do not fit in shared memory (use more lanes per world)"); }
  b->nwarp = best_nw;
  b->L2 = precision == 32 ? make_layout2<float>(b->D, wpw, b->lpw) : make_layout2<double>(b->D, wpw, b->lpw);
  b->smem2 = (size_t)b->L2.smem_tables + (size_t)b->L2.smem_stride * wpw * b->nwarp;
  {
    // the 8-byte step slots and the unit-coefficient tendon row assume what every MuJoCo composite has: one element mass
    // and coefficient 1 for every slider of the volume tendon
    bool uniform = true;
    for (int e = 0; e < b->D.ns; e++)
      if (P.tab[b->D.o_sl_m + e] != P.tab[b->D.o_sl_m] || P.tab[b->D.o_sl_tc + e] != 1.0) uniform = false;
    if (!uniform) { return fail("sg_batch_create: shell elements with different masses or tendon coefficients are not supported"); }
  }
  if (b->D.nrow >= 0xfff || b->D.ns >= 0xfff) { return fail("sg_batch_create: too many equality rows or shell joints for the packed warm-start table"); }
  if (b->L2.cand_cap < 16) { return fail("sg_batch_create: the collision scratch (the equality-row pairs of one world) is too small for this model"); }
  if (const char* e = std::getenv("SOFTGRIP_TEAM")) { if (std::atoi(e) != 0) { return fail("SOFTGRIP_TEAM: team mode was removed from the step kernel (measured slower, profiles/r01b_*, r01g_*)"); } }
  if (b->smem2 > prop.sharedMemPerBlockOptin) { return fail("sg_batch_create: worlds of one warp do not fit in shared memory (use more lanes per world)"); }
  int per_sm = 0;
  const int cfg = k2_dispatch_configure(precision, b->lpw, 32 * b->nwarp, b->smem2, &per_sm);
  if (cfg == -12345) { return fail("SOFTGRIP_LPW: this lanes-per-world value is not compiled in"); }
  if (cfg) { return fail(std::string("kernel configuration failed: ") + cudaGetErrorString((cudaError_t)cfg)); }
  if (per_sm < 1) per_sm = 1;
  b->max_ctas = per_sm * prop.multiProcessorCount; b->per_sm = per_sm;
  {
    // The (u, n) pairs of the equality sweep go to tensor memory when every resident CTA of an SM gets its window:
    // 2 (fp32) or 4 (fp64) columns per step and one empty step past the end for each warp, four warps (one per lane
    // quarter) share a column block, 512 columns per SM.  SOFTGRIP_TMEM=0 keeps them in shared memory, =1 takes
    // tensor memory whenever one CTA fits (further CTAs of the SM then wait for the allocation).
    const int stride = (b->D.nstep + 1) * (precision == 32 ? 2 : 4);
    int need = 32;
    while (need < ((b->nwarp + 3) / 4) * stride) need *= 2;
    int mode = -1;
    if (const char* te = std::getenv("SOFTGRIP_TMEM")) mode = std::atoi(te);
    if (need <= 512 && mode != 0 && (mode == 1 || need * per_sm <= 512)) { b->tm_cols = need; b->tm_stride = stride; }
    // With the rows in tensor memory their shared-memory region is free during the solve: a two-entry ring of contact
    // records per lane goes there if it fits (SOFTGRIP_RING=0: records are read from the scratch as before).
    const size_t esz = precision == 32 ? 4 : 8;
    const size_t ring_bytes = (size_t)b->lpw * (2 * CR_STRIDE * esz + 16);
    int ring_mode = 1;
    if (const char* re = std::getenv("SOFTGRIP_RING")) ring_mode = std::atoi(re);
    if (b->tm_cols && ring_mode != 0 && ring_bytes <= 2 * (size_t)b->D.nrow * esz) b->rec_ring = 1;
  }
  const int cta_worlds = wpw * b->nwarp;
  int need = (nworlds + cta_worlds - 1) / cta_worlds;
  int slots = need < b->max_ctas ? need : b->max_ctas;
  if (const char* pe = std::getenv("SOFTGRIP_PROF")) {
    if (std::atoi(pe) != 0) {
      b->prof_n = PH_COUNT + (size_t)b->max_ctas * b->nwarp;
      CUDA_OK(cudaMalloc((void**)&b->prof, sizeof(unsigned long long) * b->prof_n));
      CUDA_OK(cudaMemset(b->prof, 0, sizeof(unsigned long long) * b->prof_n));
    }
  }
  CUDA_OK(cudaMalloc((void**)&b->batch_counter, sizeof(int)));
  CUDA_OK(cudaMalloc((void**)&b->scratch, (size_t)slots * cta_worlds * (size_t)b->L2.gs_stride));
  CUDA_OK(cudaMemset(b->scratch, 0, (size_t)slots * cta_worlds * (size_t)b->L2.gs_stride));
  return sg_batch_reset(b, nullptr);
}

extern "C" void sg_batch_destroy(sg_batch* b) {
  if (!b) return;
  cudaSetDevice(b->device);
  void* ptrs[] = {b->tab, b->itab, b->qpos, b->qvel, b->warm, b->act, b->ctrl, b->status, b->p_stiff, b->p_damp, b->p_tdamp,
                  b->p_objoff, b->d_ctrl_event, b->d_ctrl_value, b->debug_out, b->stage_traj, b->stage_touch, b->scratch, b->prof, b->batch_counter};
  for (void* p : ptrs) if (p) cudaFree(p);
  delete b;
}

extern "C" int sg_batch_nworlds(const sg_batch* b) { return b ? b->W : -1; }
extern "C" int sg_batch_precision(const sg_batch* b) { return b ? b->precision : -1; }
extern "C" long long sg_batch_launch_count(const sg_batch* b) { return b ? b->launches : -1; }
extern "C" int sg_batch_config(const sg_batch* b, int* out) {
  if (!b || !out) return fail("sg_batch_config: null argument");
  const int wpw = 32 / b->lpw;
  out[0] = b->lpw; out[1] = b->nwarp; out[2] = wpw * b->nwarp;
  out[3] = b->per_sm; out[4] = (int)b->smem2; out[5] = b->L2.smem_stride;
  out[6] = 0; out[7] = 2;
  return 0;
}

extern "C" int sg_batch_prof_get(sg_batch* b, unsigned long long* out, int n) {
  if (!b || !out) return fail("sg_batch_prof_get: null argument");
  if (!b->prof) return fail("sg_batch_prof_get: phase clocks are off (create the batch with SOFTGRIP_PROF=1)");
  CUDA_OK(cudaSetDevice(b->device));
  CUDA_OK(cudaDeviceSynchronize());
  std::vector<unsigned long long> h(PH_COUNT);
  CUDA_OK(cudaMemcpy(h.data(), b->prof, sizeof(unsigned long long) * PH_COUNT, cudaMemcpyDeviceToHost));
  for (int i = 0; i < n && i < PH_COUNT; i++) out[i] = h[i];
  CUDA_OK(cudaMemset(b->prof, 0, sizeof(unsigned long long) * PH_COUNT));
  return PH_COUNT;
}

extern "C" int sg_batch_set_params(sg_batch* b, const double* stiffness, const double* damping, const double* tdamping,
                                   const double* objoff, void* stream) {
  if (!b) return fail("sg_batch_set_params: null batch");
  CUDA_OK(cudaSetDevice(b->device));
  cudaStream_t s = (cudaStream_t)stream;
  b->has_stiff = stiffness != nullptr; b->has_damp = damping != nullptr; b->has_tdamp = tdamping != nullptr; b->has_objoff = objoff != nullptr;
  if (stiffness && stiffness != b->p_stiff) CUDA_OK(cudaMemcpyAsync(b->p_stiff, stiffness, sizeof(double) * b->W, cudaMemcpyDefault, s));
  if (damping && damping != b->p_damp) CUDA_OK(cudaMemcpyAsync(b->p_damp, damping, sizeof(double) * b->W, cudaMemcpyDefault, s));
  if (tdamping && tdamping != b->p_tdamp) CUDA_OK(cudaMemcpyAsync(b->p_tdamp, tdamping, sizeof(double) * b->W, cudaMemcpyDefault, s));
  if (objoff && objoff != b->p_objoff) CUDA_OK(cudaMemcpyAsync(b->p_objoff, objoff, sizeof(double) * 3 * b->W, cudaMemcpyDefault, s));
  return 0;
}

extern "C" int sg_batch_reset(sg_batch* b, void* stream) {
  if (!b) return fail("sg_batch_reset: null batch");
  CUDA_OK(cudaSetDevice(b->device));
  cudaStream_t s = (cudaStream_t)stream;
  const size_t nv = b->D.nv, nu = b->D.nu > 0 ? b->D.nu : 1;
  CUDA_OK(cudaMemsetAsync(b->qpos, 0, b->esize * nv * b->W, s));   // qpos0 == 0 is validated by the plan
  CUDA_OK(cudaMemsetAsync(b->qvel, 0, b->esize * nv * b->W, s));
  CUDA_OK(cudaMemsetAsync(b->warm, 0, b->esize * nv * b->W, s));
  CUDA_OK(cudaMemsetAsync(b->act, 0, b->esize * nu * b->W, s));
  CUDA_OK(cudaMemsetAsync(b->ctrl, 0, b->esize * nu * b->W, s));
  CUDA_OK(cudaMemsetAsync(b->status, 0, sizeof(int) * b->W, s));
  return 0;
}

#ifdef SG_SIMT_EMU
template <typename T> static void run_cvt(const double* in, T* out, size_t n, cudaStream_t) { for (size_t i = 0; i < n; i++) out[i] = (T)in[i]; }
template <typename T> static void run_bcast(const double* in, T* out, int nu, size_t n, cudaStream_t) { for (size_t i = 0; i < n; i++) out[i] = (T)in[i % nu]; }
#else
template <typename T> __global__ void cvt_kernel(const double* in, T* out, size_t n) {
  size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (i < n) out[i] = (T)in[i];
}
template <typename T> __global__ void bcast_kernel(const double* in, T* out, int nu, size_t n) {
  size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (i < n) out[i] = (T)in[i % nu];
}
template <typename T> static void run_cvt(const double* in, T* out, size_t n, cudaStream_t s) { cvt_kernel<T><<<(unsigned)((n + 255) / 256), 256, 0, s>>>(in, out, n); }
template <typename T> static void run_bcast(const double* in, T* out, int nu, size_t n, cudaStream_t s) { bcast_kernel<T><<<(unsigned)((n + 255) / 256), 256, 0, s>>>(in, out, nu, n); }
#endif

extern "C" int sg_batch_set_ctrl(sg_batch* b, const double* ctrl, void* stream) {
  if (!b || !ctrl) return fail("sg_batch_set_ctrl: null argument");
  CUDA_OK(cudaSetDevice(b->device));
  const size_t n = (size_t)b->D.nu * b->W;
  if (n == 0) return 0;
  cudaStream_t s = (cudaStream_t)stream;
  if (b->precision == 32) run_cvt<float>(ctrl, (float*)b->ctrl, n, s);
  else run_cvt<double>(ctrl, (double*)b->ctrl, n, s);
  b->launches++;
  CUDA_OK(cudaGetLastError());
  return 0;
}

extern "C" int sg_batch_set_ctrl_all(sg_batch* b, const double* ctrl_host, void* stream) {
  if (!b || !ctrl_host) return fail("sg_batch_set_ctrl_all: null argument");
  CUDA_OK(cudaSetDevice(b->device));
  const int nu = b->D.nu;
  if (nu == 0) return 0;
  cudaStream_t s = (cudaStream_t)stream;
  if (b->sched_cap < 1) {
    if (b->d_ctrl_event) cudaFree(b->d_ctrl_event);
    if (b->d_ctrl_value) cudaFree(b->d_ctrl_value);
    b->sched_cap = 256;
    CUDA_OK(cudaMalloc((void**)&b->d_ctrl_event, sizeof(int) * b->sched_cap));
    CUDA_OK(cudaMalloc((void**)&b->d_ctrl_value, sizeof(double) * b->sched_cap * nu));
  }
  CUDA_OK(cudaMemcpyAsync(b->d_ctrl_value, ctrl_host, sizeof(double) * nu, cudaMemcpyHostToDevice, s));
  const size_t n = (size_t)nu * b->W;
  if (b->precision == 32) run_bcast<float>(b->d_ctrl_value, (float*)b->ctrl, nu, n, s);
  else run_bcast<double>(b->d_ctrl_value, (double*)b->ctrl, nu, n, s);
  b->launches++;
  CUDA_OK(cudaGetLastError());
  return 0;
}

struct LaunchSpec {
  int nsub = 1, integrate = 1;
  int rollout = 0, sim_start = 0, sim_step = 0, nrows = 0;
  void* sens_out = nullptr;
  int* touch_out = nullptr;
};


template <typename T>
static int launch_v2(sg_batch* b, const LaunchSpec& sp, cudaStream_t s) {
  KArgs2<T> K{};
  K.D = b->D; K.L = b->L2;
  // fold the (possibly updated) model-level masks / stiffness targets into this launch
  K.D.stiff_tendon0 = b->model->plan.d.stiff_tendon0;
  K.D.cap_mask = b->model->plan.d.cap_mask; K.D.sph_mask = b->model->plan.d.sph_mask;
  K.C = make_cst<T>(K.D);
  K.tab = (const T*)b->tab; K.itab = b->itab; K.nworlds = b->W;
  K.step_barrier = 1;
  if (const char* sb = std::getenv("SOFTGRIP_STEP_BARRIER")) K.step_barrier = std::atoi(sb) != 0;
  K.scratch = b->scratch;
  K.tm_cols = b->tm_cols; K.tm_stride = b->tm_stride; K.rec_ring = b->rec_ring;
  K.qpos = (T*)b->qpos; K.qvel = (T*)b->qvel; K.warm = (T*)b->warm; K.act = (T*)b->act; K.ctrl = (T*)b->ctrl;
  K.p_stiff = b->has_stiff ? b->p_stiff : nullptr; K.p_damp = b->has_damp ? b->p_damp : nullptr;
  K.p_tdamp = b->has_tdamp ? b->p_tdamp : nullptr; K.p_objoff = b->has_objoff ? b->p_objoff : nullptr;
  K.status = b->status;
  K.debug_world = b->debug_world; K.debug_out = b->debug_out; K.debug_cap = b->debug_cap;
  K.prof = b->prof;
  K.nsub = sp.nsub; K.integrate = sp.integrate; K.sens_out = (T*)sp.sens_out; K.touch_out = sp.touch_out;
  K.rollout = sp.rollout; K.sim_start = sp.sim_start; K.sim_step = sp.sim_step; K.nrows = sp.nrows;
  K.traj_soa = sp.rollout ? b->traj_soa : 0;
  K.ctrl_event = b->d_ctrl_event; K.ctrl_value = b->d_ctrl_value;
  const int cta_worlds = (32 / b->lpw) * b->nwarp;
  int grid = (b->W + cta_worlds - 1) / cta_worlds;
  K.batch_counter = nullptr;
  if (grid > b->max_ctas) {
    grid = b->max_ctas;   // persistent: each CTA walks batches of worlds, handed out by a counter (SOFTGRIP_DYNAMIC=0: fixed shares)
    bool dyn = true;
    if (const char* de = std::getenv("SOFTGRIP_DYNAMIC")) dyn = std::atoi(de) != 0;
    if (dyn && b->batch_counter) {
      CUDA_OK(cudaMemsetAsync(b->batch_counter, 0, sizeof(int), s));
      K.batch_counter = b->batch_counter;
    }
  }
  int e = k2_dispatch_launch<T>(b->lpw, K, grid, 32 * b->nwarp, b->smem2, (void*)s);
  if (e) return fail(std::string("kernel launch failed: ") + cudaGetErrorString((cudaError_t)e));
  return 0;
}

static int launch_any(sg_batch* b, const LaunchSpec& sp, void* stream) {
  CUDA_OK(cudaSetDevice(b->device));
  cudaStream_t s = (cudaStream_t)stream;
  b->launches++;
  return b->precision == 32 ? launch_v2<float>(b, sp, s) : launch_v2<double>(b, sp, s);
}

// tables are uploaded at batch creation; model-level edits made later (masks, stiffness targets) are
// re-synchronised lazily here
static int sync_tables(sg_batch* b) { return upload_tables(b, false); }

extern "C" int sg_batch_step(sg_batch* b, int nsub, void* sens_out, int* touch_out, void* stream) {
  if (!b) return fail("sg_batch_step: null batch");
  if (nsub < 1) return fail("sg_batch_step: nsub must be >= 1");
  LaunchSpec sp; sp.nsub = nsub; sp.integrate = 1; sp.sens_out = sens_out; sp.touch_out = touch_out;
  return launch_any(b, sp, stream);
}

extern "C" int sg_batch_forward(sg_batch* b, void* sens_out, int* touch_out, void* stream) {
  if (!b) return fail("sg_batch_forward: null batch");
  LaunchSpec sp; sp.nsub = 1; sp.integrate = 0; sp.sens_out = sens_out; sp.touch_out = touch_out;
  return launch_any(b, sp, stream);
}

static int upload_schedule(sg_batch* b, const sg_schedule* sc, cudaStream_t s) {
  const int nu = b->D.nu > 0 ? b->D.nu : 1;
  if (sc->nrows > b->sched_cap) {
    if (b->d_ctrl_event) cudaFree(b->d_ctrl_event);
    if (b->d_ctrl_value) cudaFree(b->d_ctrl_value);
    b->sched_cap = sc->nrows > 256 ? sc->nrows : 256;
    CUDA_OK(cudaMalloc((void**)&b->d_ctrl_event, sizeof(int) * b->sched_cap));
    CUDA_OK(cudaMalloc((void**)&b->d_ctrl_value, sizeof(double) * b->sched_cap * nu));
  }
  CUDA_OK(cudaMemcpyAsync(b->d_ctrl_event, sc->ctrl_event, sizeof(int) * sc->nrows, cudaMemcpyHostToDevice, s));
  CUDA_OK(cudaMemcpyAsync(b->d_ctrl_value, sc->ctrl_value, sizeof(double) * sc->nrows * b->D.nu, cudaMemcpyHostToDevice, s));
  return 0;
}

extern "C" int sg_batch_rollout(sg_batch* b, const sg_schedule* sc, void* traj_out, int* touch_out, void* stream) {
  if (!b || !sc || !traj_out) return fail("sg_batch_rollout: null argument");
  if (sc->nrows < 1 || sc->sim_step < 1 || sc->sim_start < 0 || !sc->ctrl_event || !sc->ctrl_value) return fail("sg_batch_rollout: bad schedule");
  CUDA_OK(cudaSetDevice(b->device));
  cudaStream_t s = (cudaStream_t)stream;
  int rc = upload_schedule(b, sc, s);
  if (rc) return rc;
  const size_t nu = b->D.nu > 0 ? b->D.nu : 1;
  CUDA_OK(cudaMemsetAsync(b->act, 0, b->esize * nu * b->W, s));
  CUDA_OK(cudaMemsetAsync(b->ctrl, 0, b->esize * nu * b->W, s));
  LaunchSpec sp; sp.rollout = 1; sp.sim_start = sc->sim_start; sp.sim_step = sc->sim_step; sp.nrows = sc->nrows;
  sp.sens_out = traj_out; sp.touch_out = touch_out;
  return launch_any(b, sp, stream);
}

extern "C" int sg_batch_set_traj_layout(sg_batch* b, int layout) {
  if (!b) return fail("sg_batch_set_traj_layout: null batch");
  if (layout != SG_TRAJ_WORLD_MAJOR && layout != SG_TRAJ_SOA) return fail("sg_batch_set_traj_layout: layout must be SG_TRAJ_WORLD_MAJOR or SG_TRAJ_SOA");
  b->traj_soa = layout == SG_TRAJ_SOA;
  return 0;
}

extern "C" int sg_batch_rollout_host(sg_batch* b, const sg_schedule* sc, const double* stiffness_host, void* traj_host,
                                     int* touch_host, int* status_host) {
  return sg_batch_rollout_host_params(b, sc, stiffness_host, nullptr, nullptr, nullptr, traj_host, touch_host, status_host);
}

extern "C" int sg_batch_rollout_host_params(sg_batch* b, const sg_schedule* sc, const double* stiffness_host, const double* damping_host,
                                            const double* tdamping_host, const double* objoff_host, void* traj_host,
                                            int* touch_host, int* status_host) {
  if (!b || !sc || !traj_host) return fail("sg_batch_rollout_host: null argument");
  CUDA_OK(cudaSetDevice(b->device));
  const size_t tb = b->esize * (size_t)b->W * sc->nrows * b->D.nsd, ub = sizeof(int) * (size_t)b->W * sc->nrows;
  if (tb > b->stage_traj_bytes) { if (b->stage_traj) cudaFree(b->stage_traj); CUDA_OK(cudaMalloc(&b->stage_traj, tb)); b->stage_traj_bytes = tb; }
  if (touch_host && ub > b->stage_touch_bytes) { if (b->stage_touch) cudaFree(b->stage_touch); CUDA_OK(cudaMalloc((void**)&b->stage_touch, ub)); b->stage_touch_bytes = ub; }
  if (stiffness_host || damping_host || tdamping_host || objoff_host) {
    // host -> device copies of the per-world parameters (parameters that are not given keep what the batch already holds)
    int rc = sg_batch_set_params(b, stiffness_host ? stiffness_host : (b->has_stiff ? b->p_stiff : nullptr),
                                 damping_host ? damping_host : (b->has_damp ? b->p_damp : nullptr),
                                 tdamping_host ? tdamping_host : (b->has_tdamp ? b->p_tdamp : nullptr),
                                 objoff_host ? objoff_host : (b->has_objoff ? b->p_objoff : nullptr), nullptr);
    if (rc) return rc;
  }
  CUDA_OK(cudaMemsetAsync(b->status, 0, sizeof(int) * b->W, 0));
  int rc = sg_batch_rollout(b, sc, b->stage_traj, touch_host ? b->stage_touch : nullptr, nullptr);
  if (rc) return rc;
  CUDA_OK(cudaMemcpyAsync(traj_host, b->stage_traj, tb, cudaMemcpyDeviceToHost, 0));
  if (touch_host) CUDA_OK(cudaMemcpyAsync(touch_host, b->stage_touch, ub, cudaMemcpyDeviceToHost, 0));
  if (status_host) CUDA_OK(cudaMemcpyAsync(status_host, b->status, sizeof(int) * b->W, cudaMemcpyDeviceToHost, 0));
  CUDA_OK(cudaStreamSynchronize(0));
  return 0;
}

template <typename T>
static int get_arr(const void* dev, double* host, size_t n) {
  if (!host) return 0;
  std::vector<T> tmp(n);
  CUDA_OK(cudaMemcpy(tmp.data(), dev, sizeof(T) * n, cudaMemcpyDeviceToHost));
  for (size_t i = 0; i < n; i++) host[i] = (double)tmp[i];
  return 0;
}
template <typename T>
static int set_arr(void* dev, const double* host, size_t n) {
  if (!host) return 0;
  std::vector<T> tmp(n);
  for (size_t i = 0; i < n; i++) tmp[i] = (T)host[i];
  CUDA_OK(cudaMemcpy(dev, tmp.data(), sizeof(T) * n, cudaMemcpyHostToDevice));
  return 0;
}

extern "C" int sg_batch_get_state(sg_batch* b, double* qpos, double* qvel, double* act, double* warm) {
  if (!b) return fail("sg_batch_get_state: null batch");
  CUDA_OK(cudaSetDevice(b->device));
  CUDA_OK(cudaDeviceSynchronize());
  const size_t n = (size_t)b->D.nv * b->W, na = (size_t)b->D.nu * b->W;
  int rc = 0;
  if (b->precision == 32) { rc |= get_arr<float>(b->qpos, qpos, n); rc |= get_arr<float>(b->qvel, qvel, n); rc |= get_arr<float>(b->act, act, na); rc |= get_arr<float>(b->warm, warm, n); }
  else { rc |= get_arr<double>(b->qpos, qpos, n); rc |= get_arr<double>(b->qvel, qvel, n); rc |= get_arr<double>(b->act, act, na); rc |= get_arr<double>(b->warm, warm, n); }
  return rc;
}

extern "C" int sg_batch_set_state(sg_batch* b, const double* qpos, const double* qvel, const double* act, const double* warm) {
  if (!b) return fail("sg_batch_set_state: null batch");
  CUDA_OK(cudaSetDevice(b->device));
  CUDA_OK(cudaDeviceSynchronize());
  const size_t n = (size_t)b->D.nv * b->W, na = (size_t)b->D.nu * b->W;
  int rc = 0;
  if (b->precision == 32) { rc |= set_arr<float>(b->qpos, qpos, n); rc |= set_arr<float>(b->qvel, qvel, n); rc |= set_arr<float>(b->act, act, na); rc |= set_arr<float>(b->warm, warm, n); }
  else { rc |= set_arr<double>(b->qpos, qpos, n); rc |= set_arr<double>(b->qvel, qvel, n); rc |= set_arr<double>(b->act, act, na); rc |= set_arr<double>(b->warm, warm, n); }
  return rc;
}

extern "C" int sg_batch_status(sg_batch* b, int* status_host, int clear) {
  if (!b || !status_host) return fail("sg_batch_status: null argument");
  CUDA_OK(cudaSetDevice(b->device));
  CUDA_OK(cudaDeviceSynchronize());
  CUDA_OK(cudaMemcpy(status_host, b->status, sizeof(int) * b->W, cudaMemcpyDeviceToHost));
  if (clear) CUDA_OK(cudaMemset(b->status, 0, sizeof(int) * b->W));
  return 0;
}

extern "C" int sg_batch_sync(sg_batch* b, void* stream) {
  if (!b) return fail("sg_batch_sync: null batch");
  CUDA_OK(cudaSetDevice(b->device));
  CUDA_OK(cudaStreamSynchronize((cudaStream_t)stream));
  return 0;
}

extern "C" int sg_batch_set_debug_world(sg_batch* b, int world) {
  if (!b) return fail("sg_batch_set_debug_world: null batch");
  if (world >= b->W) return fail("sg_batch_set_debug_world: world out of range");
  b->debug_world = world;
  // model-level edits (geom masks, stiffness targets) may have happened since creation
  return sync_tables(b);
}

extern "C" int sg_batch_debug_get(sg_batch* b, const char* key, double* out, int cap) {
  if (!b || !key) return fail("sg_batch_debug_get: null argument");
  CUDA_OK(cudaSetDevice(b->device));
  CUDA_OK(cudaDeviceSynchronize());
  std::vector<double> h(b->debug_cap);
  CUDA_OK(cudaMemcpy(h.data(), b->debug_out, sizeof(double) * b->debug_cap, cudaMemcpyDeviceToHost));
  const int ncontot = (int)h[0], nefc = (int)h[1], ncon = (int)h[3], nlim = (int)h[4];
  const std::string k(key);
  auto put = [&](const double* src, int n) { if (out) for (int i = 0; i < n && i < cap; i++) out[i] = src[i]; return n; };
  if (k == "pair_runs") {
    // host-side collision tables (no device data): [npair, nrun], the candidate pair list in MuJoCo's contact order as
    // (type, collider a, second geom b) triples, then the run-length blocks {type, a0 | na << 8, b0, nb} the device
    // broadphase walks
    const Plan& P = b->model->plan;
    std::vector<double> t = {(double)P.d.npair, (double)P.d.nrun};
    for (int p = 0; p < P.d.npair; p++) { t.push_back(P.itab[P.d.io_pair_t + p]); t.push_back(P.itab[P.d.io_pair_a + p]); t.push_back(P.itab[P.d.io_pair_b + p]); }
    for (int i = 0; i < 4 * P.d.nrun; i++) t.push_back(P.itab[P.d.io_run + i]);
    return put(t.data(), (int)t.size());
  }
  if (k == "sweep_schedule") {
    // host-side tables of the equality sweep (no device data): [nstep, lanes per world, bytes per real, nrow, estimated
    // shared-memory wavefronts per sweep], the slot descriptors (2 ints per slot, nstep + 1 steps), then the storage
    // position of every row (plan schedule order)
    // (the rows per slot, always 1, ride in the upper digits of the wavefront figure: 1e9 * rows per slot + wavefronts)
    const int rows_per_slot = 1;
    const long wf = sweep_wavefronts(b->step_d, b->lpw, (int)b->esize);
    std::vector<double> t = {(double)b->D.nstep, (double)b->lpw, (double)b->esize, (double)b->D.nrow, (double)wf + 1e9 * rows_per_slot};
    for (int v : b->step_d) t.push_back((double)(unsigned)v);
    for (int v : b->row_perm) t.push_back((double)v);
    return put(t.data(), (int)t.size());
  }
  auto scalar = [&](double v) { if (out && cap > 0) out[0] = v; return 1; };
  if (k == "tensor_memory") {
    // [columns the CTA allocates (0: the equality rows stay in shared memory), columns per warp, record ring in use]
    const double t[3] = {(double)b->tm_cols, (double)b->tm_stride, (double)b->rec_ring};
    return put(t, 3);
  }
  if (k == "ncon") return scalar(ncontot);
  if (k == "nefc") return scalar(nefc);
  if (k == "solver_iter") return scalar(h[2]);
  if (k == "ncon_rows") return scalar(ncon);
  if (k == "nlim") return scalar(nlim);
  if (k == "maxlev") return scalar(h[5]);
  if (k == "ncand") return scalar(h[6]);
  const int base = 64 + 16 * 2 * b->D.maxcon, eb = base + b->D.nv;
  if (k == "qacc") return put(&h[base], b->D.nv);
  if (k == "con_dist" || k == "con_pos" || k == "con_frame") {
    const int per = k == "con_dist" ? 1 : (k == "con_pos" ? 3 : 9), offs = k == "con_dist" ? 0 : (k == "con_pos" ? 1 : 4);
    std::vector<double> t((size_t)per * ncontot);
    for (int i = 0; i < ncontot && i < 2 * b->D.maxcon; i++) for (int j = 0; j < per; j++) t[(size_t)i * per + j] = h[64 + 16 * i + offs + j];
    return put(t.data(), per * ncontot);
  }
  if (k == "efc_force" || k == "efc_aref" || k == "efc_R") {
    // device rows are in schedule order; map the equality block back to MuJoCo row ids
    const int which = k == "efc_force" ? 0 : (k == "efc_aref" ? 1 : 2);
    std::vector<double> t(nefc);
    const std::vector<int>& sched = b->model->plan.sched_eq;
    for (int p = 0; p < b->D.nrow; p++) t[sched[p]] = h[eb + which * nefc + (b->row_perm.empty() ? p : b->row_perm[p])];
    for (int r = b->D.nrow; r < nefc; r++) t[r] = h[eb + which * nefc + r];
    return put(t.data(), nefc);
  }
  return fail("sg_batch_debug_get: unknown key " + k);
}

// ---- trajectory post-processing (sg_traj.cuh): noise augmentation, channel statistics, --mask-contact ----------------
static int traj_sm_count(int device, int* out) {
  static std::atomic<int> cached[64];                // SM count per device; racing first calls store the same value
  if (device < 0 || device >= 64) return fail("bad device index");
  if (!cached[device].load(std::memory_order_relaxed)) {
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) return fail("no CUDA device available (libsoftgrip has no CPU path)");
    if (device >= ndev) return fail("bad device index");
    cudaDeviceProp prop;
    CUDA_OK(cudaGetDeviceProperties(&prop, device));
    cached[device].store(prop.multiProcessorCount, std::memory_order_relaxed);
  }
  *out = cached[device].load(std::memory_order_relaxed);
  return 0;
}

static int traj_check(const char* fn, const void* p, long long nrows, int nchan, int precision) {
  if (!p) return fail(std::string(fn) + ": null trajectory");
  if (precision != 32 && precision != 64) return fail(std::string(fn) + ": precision must be 32 or 64");
  if (nrows < 0) return fail(std::string(fn) + ": negative row count");
  if (nchan < 4 || nchan % 4 != 0 || nchan > TRAJ_STATS_MAX_CHAN) return fail(std::string(fn) + ": nchan must be a multiple of 4 in [4, 64]");
  if (((uintptr_t)p & 15) != 0) return fail(std::string(fn) + ": trajectory must be 16-byte aligned");
  return 0;
}

template <typename T>
static int traj_noise_launch(const void* in, void* out, long long nrows, long long first_row, int nchan, int nacc, double sa, double sg_,
                             unsigned long long seed, const double* mean, const double* stdev, int sms, void* stream) {
  TrajNoiseArgs<T> A;
  A.in = (const T*)in; A.out = (T*)out; A.nelem = nrows * nchan; A.nchan = nchan; A.nacc = nacc;
  A.sigma_acc = (float)sa; A.sigma_gyro = (float)sg_;
  A.k0 = (uint32_t)seed; A.k1 = (uint32_t)(seed >> 32);
  A.first_quad = (unsigned long long)first_row * (unsigned long long)(nchan / 4);
  A.mean = mean; A.stdev = stdev;
  const int block = 256;
  const long long nquad = A.nelem / 4;
  long long grid = (nquad + block - 1) / block;
  auto kp = sg_traj_noise_kernel<T>;
  static std::atomic<int> occ{0};                     // resident CTAs per SM of this instantiation (asked once)
  int per_sm = occ.load(std::memory_order_relaxed);
  if (!per_sm) {
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kp, block, 3 * 64 * sizeof(T)) != cudaSuccess || per_sm < 1) per_sm = 1;
    occ.store(per_sm, std::memory_order_relaxed);
  }
  if (grid > (long long)sms * per_sm) grid = (long long)sms * per_sm;   // exactly one resident wave, grid-stride beyond that
  SG_LAUNCH(kp, (int)grid, block, (size_t)3 * nchan * sizeof(T), (cudaStream_t)stream, A);
  CUDA_OK(cudaGetLastError());
  return 0;
}

extern "C" int sg_traj_add_noise(const void* traj_in, void* traj_out, long long nrows, long long first_row, int nchan, int nacc,
                                 double sigma_acc, double sigma_gyro, unsigned long long seed, const double* mean, const double* stdev,
                                 int precision, int device, void* stream) {
  if (int rc = traj_check("sg_traj_add_noise", traj_in, nrows, nchan, precision)) return rc;
  if (int rc = traj_check("sg_traj_add_noise", traj_out, nrows, nchan, precision)) return rc;
  if (nacc < 0 || nacc > nchan) return fail("sg_traj_add_noise: nacc out of range");
  if (first_row < 0) return fail("sg_traj_add_noise: negative first_row");
  if (!(sigma_acc >= 0) || !(sigma_gyro >= 0)) return fail("sg_traj_add_noise: negative or NaN sigma");
  if ((mean == nullptr) != (stdev == nullptr)) return fail("sg_traj_add_noise: mean and std must be given together");
  int sms = 0;
  if (int rc = traj_sm_count(device, &sms)) return rc;
  if (nrows == 0) return 0;
  CUDA_OK(cudaSetDevice(device));
  return precision == 32 ? traj_noise_launch<float>(traj_in, traj_out, nrows, first_row, nchan, nacc, sigma_acc, sigma_gyro, seed, mean, stdev, sms, stream)
                         : traj_noise_launch<double>(traj_in, traj_out, nrows, first_row, nchan, nacc, sigma_acc, sigma_gyro, seed, mean, stdev, sms, stream);
}

static int traj_stats_block(int nchan) {           // a multiple of 32 and of nchan / 4: 384 threads for 12 or 24 channels
  const int qpr = nchan / 4;
  int l = 32;
  while (l % qpr) l += 32;                         // lcm(32, qpr) <= 480 for qpr <= 16
  int block = l;
  while (block + l <= 384) block += l;
  return block;
}

// one resident wave of pass-1 CTAs (the occupancy the hardware reports for this instantiation), never more CTAs than quads
static int traj_stats_grid(int nchan, long long nrows, int sms, int precision) {
  const int block = traj_stats_block(nchan);
  const long long nquad = nrows * (nchan / 4);
  long long grid = (nquad + block - 1) / block;
  static std::atomic<int> occ[2][17];                // [precision][block / 32]: asked once per instantiation and block size
  std::atomic<int>& slot = occ[precision == 32 ? 0 : 1][(block / 32) & 15];
  int per_sm = slot.load(std::memory_order_relaxed);
  if (!per_sm) {
    const size_t smem = (size_t)block * 8 * sizeof(double);
    const cudaError_t e = precision == 32 ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, sg_traj_stats_partial_kernel<float>, block, smem)
                                          : cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, sg_traj_stats_partial_kernel<double>, block, smem);
    if (e != cudaSuccess || per_sm < 1) per_sm = 1;
    slot.store(per_sm, std::memory_order_relaxed);
  }
  const long long cap = (long long)sms * per_sm;
  if (grid > cap) grid = cap;
  return (int)(grid < 1 ? 1 : grid);
}

extern "C" long long sg_traj_stats_workspace_bytes(long long nrows, int nchan, int device) {
  if (nrows < 0 || nchan < 4 || nchan % 4 != 0 || nchan > TRAJ_STATS_MAX_CHAN) return fail("sg_traj_stats_workspace_bytes: bad shape");
  int sms = 0;
  if (int rc = traj_sm_count(device, &sms)) return rc;
  if (cudaSetDevice(device) != cudaSuccess) return fail("sg_traj_stats_workspace_bytes: cudaSetDevice failed");
  // (sized for either precision: the larger of the two grids)
  const int g32 = traj_stats_grid(nchan, nrows, sms, 32), g64 = traj_stats_grid(nchan, nrows, sms, 64);
  return (long long)(g32 > g64 ? g32 : g64) * 2 * nchan * (long long)sizeof(double);
}

template <typename T>
static int traj_stats_launch(const void* in, long long nrows, int nchan, double* mean, double* stdev, void* ws, int sms, void* stream) {
  TrajStatsArgs<T> A;
  A.in = (const T*)in; A.nrows = nrows; A.nchan = nchan; A.partial = (double*)ws; A.mean = mean; A.stdev = stdev;
  const int block = traj_stats_block(nchan);
  A.nblocks = traj_stats_grid(nchan, nrows, sms, sizeof(T) == 4 ? 32 : 64);
  auto k1 = sg_traj_stats_partial_kernel<T>;
  SG_LAUNCH(k1, A.nblocks, block, (size_t)block * 8 * sizeof(double), (cudaStream_t)stream, A);
  CUDA_OK(cudaGetLastError());
  auto k2 = sg_traj_stats_final_kernel<T>;
  SG_LAUNCH(k2, 1, TRAJ_STATS_FINAL_THREADS, (size_t)(TRAJ_STATS_FINAL_THREADS / (2 * nchan)) * 2 * nchan * sizeof(double), (cudaStream_t)stream, A);
  CUDA_OK(cudaGetLastError());
  return 0;
}

extern "C" int sg_traj_channel_stats(const void* traj, long long nrows, int nchan, int precision, int device, double* mean_out,
                                     double* std_out, void* workspace, long long workspace_bytes, void* stream) {
  if (int rc = traj_check("sg_traj_channel_stats", traj, nrows, nchan, precision)) return rc;
  if (!mean_out || !std_out || !workspace) return fail("sg_traj_channel_stats: null output or workspace");
  if (nrows < 1) return fail("sg_traj_channel_stats: needs at least one row");
  const long long need = sg_traj_stats_workspace_bytes(nrows, nchan, device);
  if (need < 0) return (int)need;
  if (workspace_bytes < need) return fail("sg_traj_channel_stats: workspace too small (see sg_traj_stats_workspace_bytes)");
  int sms = 0;
  if (int rc = traj_sm_count(device, &sms)) return rc;
  CUDA_OK(cudaSetDevice(device));
  return precision == 32 ? traj_stats_launch<float>(traj, nrows, nchan, mean_out, std_out, workspace, sms, stream)
                         : traj_stats_launch<double>(traj, nrows, nchan, mean_out, std_out, workspace, sms, stream);
}

template <typename T>
static int traj_mask_launch(void* traj, const int* touch, int nworlds, int T_, int nchan, int allf, int anybit, int mode, int* fleft,
                            int sms, void* stream) {
  TrajMaskArgs<T> A;
  A.traj = (T*)traj; A.touch = touch; A.nworlds = nworlds; A.T_ = T_; A.nchan = nchan; A.allf = allf; A.anybit = anybit; A.mode = mode;
  A.fleft = fleft;
  const int block = 256, wpb = block / 32;
  long long grid = ((long long)nworlds + wpb - 1) / wpb;
  if (grid > (long long)sms * 8) grid = (long long)sms * 8;
  auto kp = sg_traj_mask_kernel<T>;
  SG_LAUNCH(kp, (int)grid, block, 0, (cudaStream_t)stream, A);
  CUDA_OK(cudaGetLastError());
  return 0;
}

extern "C" int sg_traj_mask_contact(void* traj, const int* touch, int nworlds, int nrows_per_world, int nchan, int all_fingers,
                                    int any_bit, int mode, int* fingers_left, int precision, int device, void* stream) {
  if (int rc = traj_check("sg_traj_mask_contact", traj, (long long)nworlds * nrows_per_world, nchan, precision)) return rc;
  if (!touch) return fail("sg_traj_mask_contact: null touch");
  if (nworlds < 0 || nrows_per_world < 0) return fail("sg_traj_mask_contact: negative shape");
  if (mode != 0 && mode != 1) return fail("sg_traj_mask_contact: mode must be 0 (intended) or 1 (reference-literal)");
  if (all_fingers & any_bit) return fail("sg_traj_mask_contact: any_bit overlaps the finger bits");
  int sms = 0;
  if (int rc = traj_sm_count(device, &sms)) return rc;
  if (nworlds == 0 || nrows_per_world == 0) return 0;
  CUDA_OK(cudaSetDevice(device));
  return precision == 32 ? traj_mask_launch<float>(traj, touch, nworlds, nrows_per_world, nchan, all_fingers, any_bit, mode, fingers_left, sms, stream)
                         : traj_mask_launch<double>(traj, touch, nworlds, nrows_per_world, nchan, all_fingers, any_bit, mode, fingers_left, sms, stream);
}
