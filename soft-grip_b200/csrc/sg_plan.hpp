// sg_plan.hpp -- host side of libsoftgrip: parses the model blob written by mjcf.py and builds the
// device "plan": flat constant tables specialised for the reference's model family
//   (static world) + finger chains of hinge joints + a composite shell of slide joints on a static body,
// plus the Gauss-Seidel dependency-level schedule of the composite's equality rows.
//
// It replaces what mj_loadXML/mj_makeData hand to mj_step in the reference (ref: environment/manenv.py:27-28).
// Anything outside that model family is rejected with an error -- there is no generic/CPU fallback.
#pragma once
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <map>
#include <stdexcept>
#include <string>
#include <vector>

namespace sg {

constexpr int MAXCHAIN = 2;   // finger chains (dof trees of hinge joints)
constexpr int MAXCD = 4;      // dofs per chain
constexpr int MAXCB = 2;      // moving bodies per chain
constexpr int MAXFD = MAXCHAIN * MAXCD;
constexpr int MAXCOLL = 12;   // plane + boxes
constexpr int MAXSENS = 8;
constexpr int MAXDOFROWS = 7; // fix + 3 neighbour rows as first joint + 3 as second joint

enum { GEOM_PLANE = 0, GEOM_SPHERE = 2, GEOM_CAPSULE = 3, GEOM_BOX = 6 };
enum { JNT_SLIDE = 2, JNT_HINGE = 3 };
enum { EQ_JOINT = 2, EQ_TENDON = 3 };
enum { TEN_FIXED = 0, TEN_SPATIAL = 1 };
enum { SENS_ACCEL = 0, SENS_GYRO = 1 };
// pair types of the device pair list
enum { PAIR_PLANE_CAPSULE = 0, PAIR_BOX_CAPSULE = 1, PAIR_SPHERE_BOX = 2, PAIR_BOX_BOX = 3, PAIR_PLANE_BOX = 4 };

// chain descriptor layout inside the double table (per chain, stride CH_STRIDE)
constexpr int CH_BASEPOS = 0;               // 3  world position of the static parent frame
constexpr int CH_BASEROT = 3;               // 9  its rotation
constexpr int CH_BODY = 12;                 // MAXCB x CB_STRIDE
constexpr int CB_POS = 0, CB_ROT = 3, CB_IPOS = 12, CB_IROT = 15, CB_MASS = 24, CB_INERTIA = 25,
              CB_GPOS = 28, CB_GROT = 31, CB_GSIZE = 40, CB_BIW = 43, CB_STRIDE = 44;
constexpr int CH_DOF = CH_BODY + MAXCB * CB_STRIDE;   // MAXCD x CD_STRIDE
constexpr int CD_BODY = 0, CD_AXIS = 1, CD_JPOS = 4, CD_LO = 7, CD_HI = 8, CD_LIMITED = 9, CD_IW = 10, CD_STRIDE = 11;
constexpr int CH_TEN = CH_DOF + MAXCD * CD_STRIDE;    // tendon/actuator of this chain
constexpr int CT_HAS = 0, CT_S0 = 1 /*3 static site world pos*/, CT_BODY = 4, CT_S1 = 5 /*3 local*/, CT_GEAR = 8,
              CT_GAIN = 9, CT_TIMECONST = 10, CT_ACT = 11, CT_STRIDE = 12;
constexpr int CH_STRIDE = CH_TEN + CT_STRIDE;
// collider table (per collider, stride CO_STRIDE)
constexpr int CO_TYPE = 0, CO_CHAIN = 1 /*-1 static*/, CO_BODY = 2, CO_POS = 3, CO_ROT = 6, CO_SIZE = 15, CO_RBOUND = 18,
              CO_BIW = 19, CO_MASK = 20, CO_STRIDE = 21;
// sensor table
constexpr int SE_TYPE = 0, SE_CHAIN = 1, SE_BODY = 2, SE_POS = 3, SE_ROT = 6, SE_ADR = 15, SE_STRIDE = 16;

// POD handed to the kernels by value
struct PlanDims {
  int nv, nfd, ns, nrow, nlev, nchain, nu, nsd, ncoll, npair, nsens, maxcon, maxcand, iters, stiff_tendon0, has_sphere;
  int ncd[MAXCHAIN], ncb[MAXCHAIN], chain_dof0[MAXCHAIN];
  double h, g[3], tol, impratio, impr_scale;
  double eqj_K, eqj_B, eqj_solimp[5];
  double eqt_K, eqt_B, eqt_solimp[5], ten_iw, ten_k0, ten_d0, ten_lspring, ten_l0;
  double lim_K, lim_B, lim_solimp[5];
  double con_K, con_B, con_solimp[5], con_fr;
  double cap_r, cap_hl, sph_r, sph_pos[3], sph_mask, cap_mask;
  double obj_pos[3];
  // offsets into the double table
  int o_sl_axis, o_sl_cap0, o_sl_k0, o_sl_d0, o_sl_m, o_sl_tc, o_sl_biw, o_sl_iw, o_chain, o_coll, o_sens;
  int o_row_iw;     // 2*nrow: 1/m of the row's first and second slider (0 when the row has one dof), schedule order
  int o_sl_tciw;    // ns: tendon coefficient / slider mass
  // offsets into the int table
  int io_kmask, io_row_d1, io_row_d2, io_lev_start, io_dof_rows, io_pair_t, io_pair_a, io_pair_b;
  int io_row_d12;   // nrow: first slider | second slider << 16 (0xffff: none), schedule order
  int io_run, nrun; // broadphase runs of the pair list: {pair type, first collider | colliders << 8, first second geom, count}
  // per-batch step tables of the level sweep (depend on the lanes per world; appended by sg_api.cu)
  int io_step_d;    // 2*(nstep+1)*lpw ints: {byte offset of d1 | of d2 << 16, byte offset of the row pair | barrier << 31} per slot
  int o_step_iw;    // unused: the slots carry no masses (every shell slider has the same one)
  int nstep;
};

struct Blob {
  const unsigned char* p = nullptr;
  size_t n = 0;
  bool find(const char* name, int& dtype, unsigned& count, const void*& data) const {
    if (n < 12 || std::memcmp(p, "SGM1", 4) != 0) return false;
    unsigned nsec;
    std::memcpy(&nsec, p + 8, 4);
    const unsigned char* e = p + 12;
    for (unsigned i = 0; i < nsec; i++, e += 48) {
      if (std::strncmp((const char*)e, name, 32) == 0) {
        unsigned dt, cnt;
        unsigned long long off;
        std::memcpy(&dt, e + 32, 4);
        std::memcpy(&cnt, e + 36, 4);
        std::memcpy(&off, e + 40, 8);
        if (off + (size_t)cnt * (dt == 0 ? 8 : 4) > n) return false;
        dtype = (int)dt; count = cnt; data = p + off;
        return true;
      }
    }
    return false;
  }
  std::vector<double> d(const char* name) const {
    int dt; unsigned c; const void* q;
    if (!find(name, dt, c, q) || dt != 0) throw std::runtime_error(std::string("model blob: missing float section ") + name);
    std::vector<double> v(c);
    if (c) std::memcpy(v.data(), q, c * 8);
    return v;
  }
  std::vector<int> i(const char* name) const {
    int dt; unsigned c; const void* q;
    if (!find(name, dt, c, q) || dt != 1) throw std::runtime_error(std::string("model blob: missing int section ") + name);
    std::vector<int> v(c);
    if (c) std::memcpy(v.data(), q, c * 4);
    return v;
  }
};

inline void h_quat2mat(const double* q, double* R) {
  double w = q[0], x = q[1], y = q[2], z = q[3];
  R[0] = w * w + x * x - y * y - z * z; R[1] = 2 * (x * y - w * z); R[2] = 2 * (x * z + w * y);
  R[3] = 2 * (x * y + w * z); R[4] = w * w - x * x + y * y - z * z; R[5] = 2 * (y * z - w * x);
  R[6] = 2 * (x * z - w * y); R[7] = 2 * (y * z + w * x); R[8] = w * w - x * x - y * y + z * z;
}
inline void h_matmul3(const double* A, const double* B, double* C) {
  double t[9];
  for (int i = 0; i < 3; i++) for (int j = 0; j < 3; j++) t[3 * i + j] = A[3 * i] * B[j] + A[3 * i + 1] * B[3 + j] + A[3 * i + 2] * B[6 + j];
  std::memcpy(C, t, sizeof(t));
}
inline void h_matvec3(const double* A, const double* v, double* r) {
  double t[3] = {A[0] * v[0] + A[1] * v[1] + A[2] * v[2], A[3] * v[0] + A[4] * v[1] + A[5] * v[2], A[6] * v[0] + A[7] * v[1] + A[8] * v[2]};
  std::memcpy(r, t, sizeof(t));
}

struct Plan {
  PlanDims d{};
  std::vector<double> tab;
  std::vector<int> itab;
  std::vector<int> geom_mask;      // per geom (host); folded into collider masks on upload
  std::vector<int> coll_geom;      // collider -> geom id
  int ngeom = 0, neq = 0, center_geom = -1, first_capsule_geom = -1;
  std::vector<int> sched_eq;       // schedule position -> equality id (diagnostics)
  std::vector<int> stiff_mask;     // per dof
};

#define SG_REQUIRE(cond, msg) do { if (!(cond)) throw std::runtime_error(std::string("unsupported model: ") + msg); } while (0)

// Level sweep tables for `lpw` lanes per world.  The rows are list-scheduled onto steps of `lpw` slots: a row is ready
// once every earlier row (in MuJoCo's sequential order) that shares one of its sliders has run in an earlier step; among
// the ready rows the ones with the longest chain of dependants go first.  A step carries the "barrier" flag when a row of
// a later step, up to the next flagged step, depends on one of its rows or of an earlier unflagged step.  The result
// equals the sequential sweep (rows that share a slider keep their order, rows that do not commute).
// The sweep is bound by shared-memory wavefronts, so the schedule also avoids bank conflicts: the worlds of a warp sit
// `lpw` banks apart, hence the accesses of a step are conflict-free when the slider indices (first sliders among each
// other, second sliders among each other) and the storage positions of the rows are distinct modulo `lpw`.  A row with
// slack waits for a step where it fits (`target` = schedule length the slack is measured against; the caller searches
// it); the storage position of every row (`perm`: schedule position of the plan -> position in the kernel's row
// arrays) is chosen so that the rows of a step get distinct residues.  Padding slots and the missing second slider of
// fix rows are predicated off by the kernel (second-slider offset 0xffff, valid bit clear).
// Slot encoding (esize = bytes per real of the kernel precision): {first slider * esize | second slider * esize << 16,
// row position * 2 * esize | valid << 30 | barrier << 31}.
// (A second scheduler that gave every lane two rows per step -- 31 steps instead of 58 for softbox, bit-identical results --
// measured 2 % slower, profiles/r02l_sweep.log: at 16 warps per SM the sweep is bound by shared-memory wavefronts, which
// fusing does not reduce, not by the latency of a step.  It was removed.)
inline int build_step_tables_for(const PlanDims& D, const std::vector<int>& itab, int lpw, int esize, int target,
                                 std::vector<int>& step_d, std::vector<int>& perm) {
  step_d.clear();
  const int nrow = D.nrow;
  const bool avoid = target > 0;
  const int R = lpw < 32 ? lpw : 32;                 // residue modulus: bank distance of the worlds of a warp
  SG_REQUIRE((size_t)(D.ns + 1) * esize < 0xffff && (size_t)(nrow + 1) * 2 * esize < (1u << 30), "too many shell joints for the packed step descriptors");
  // dependency chains per slider, in schedule order (which respects MuJoCo's row order along every slider)
  std::vector<int> last(D.ns, -1), npred(nrow, 0), height(nrow, 1), step_of(nrow, -1);
  std::vector<std::vector<int>> pred(nrow), succ(nrow);
  for (int p = 0; p < nrow; p++) {
    const int ds[2] = {itab[D.io_row_d1 + p], itab[D.io_row_d2 + p]};
    for (int k = 0; k < 2; k++) {
      const int d = ds[k];
      if (d < 0) continue;
      const int q = last[d];
      if (q >= 0 && (pred[p].empty() || pred[p].back() != q)) { pred[p].push_back(q); succ[q].push_back(p); }
      last[d] = p;
    }
    npred[p] = (int)pred[p].size();
  }
  for (int p = nrow - 1; p >= 0; p--) for (int s : succ[p]) if (height[s] + 1 > height[p]) height[p] = height[s] + 1;
  std::vector<std::vector<int>> steps;
  std::vector<int> ready;
  for (int p = 0; p < nrow; p++) if (npred[p] == 0) ready.push_back(p);
  int done = 0;
  while (done < nrow) {
    SG_REQUIRE(!ready.empty(), "cyclic equality schedule");
    std::stable_sort(ready.begin(), ready.end(), [&](int a, int b) { return height[a] != height[b] ? height[a] > height[b] : a < b; });
    const int now = (int)steps.size();
    std::vector<int> cur, rest;
    std::vector<char> use1(R, 0), use2(R, 0);
    for (int p : ready) {
      const int d1 = itab[D.io_row_d1 + p], d2 = itab[D.io_row_d2 + p];
      const bool clash = avoid && (use1[d1 % R] || (d2 >= 0 && use2[d2 % R]));
      const bool must = now + height[p] >= target;   // no slack left: waiting would lengthen the schedule
      if ((int)cur.size() < lpw && (!clash || must)) {
        cur.push_back(p); use1[d1 % R] = 1; if (d2 >= 0) use2[d2 % R] = 1;
      } else rest.push_back(p);
    }
    ready.swap(rest);
    for (int p : cur) step_of[p] = now;
    for (int p : cur) for (int s : succ[p]) if (--npred[s] == 0) ready.push_back(s);
    done += (int)cur.size();
    steps.push_back(cur);
  }
  const int nstep = (int)steps.size();
  std::vector<int> flag(nstep, 0);
  int synced = -1;                                   // every step <= synced is followed by a barrier somewhere before the current one
  for (int s = 0; s < nstep; s++) {
    bool need = false;
    for (int p : steps[s]) for (int q : pred[p]) if (step_of[q] > synced) need = true;
    if (need) { flag[s - 1] = 1; synced = s - 1; }
  }
  if (nstep > 0) flag[nstep - 1] = 1;                // the tendon row reads every slider
  // storage positions: the rows of a step get distinct residues, classes filled evenly
  perm.assign(nrow, -1);
  if (avoid) {
    std::vector<int> cap(R, 0), used(R, 0);
    for (int q = 0; q < nrow; q++) cap[q % R]++;
    for (int s = 0; s < nstep; s++) {
      std::vector<char> taken(R, 0);
      for (int p : steps[s]) {
        int best = -1;
        for (int pass = 0; pass < 2 && best < 0; pass++)
          for (int r = 0; r < R; r++) {
            if (used[r] >= cap[r] || (pass == 0 && taken[r])) continue;
            if (best < 0 || cap[r] - used[r] > cap[best] - used[best]) best = r;
          }
        SG_REQUIRE(best >= 0, "row storage assignment");
        taken[best] = 1;
        perm[p] = best + R * used[best]++;
      }
    }
  } else for (int p = 0; p < nrow; p++) perm[p] = p;
  auto emit = [&](int p, int fl) {
    unsigned x = 0xffffffffu, y = (unsigned)fl << 31;
    if (p >= 0) {
      const int d1 = itab[D.io_row_d1 + p], d2 = itab[D.io_row_d2 + p];
      const unsigned o2 = d2 >= 0 ? (unsigned)(d2 * esize) : 0xffffu;
      x = (unsigned)(d1 * esize) | (o2 << 16);
      y = ((unsigned)fl << 31) | (unsigned)(perm[p] * 2 * esize) | (1u << 30);
    }
    step_d.push_back((int)x); step_d.push_back((int)y);
  };
  for (int s = 0; s < nstep; s++) for (int k = 0; k < lpw; k++) emit(k < (int)steps[s].size() ? steps[s][k] : -1, flag[s]);
  // one empty step past the end: the sweep prefetches the next step's descriptors unconditionally
  for (int k = 0; k < lpw; k++) emit(-1, 0);
  return nstep;
}

// shared-memory wavefronts of one equality sweep for the tables above (the model the schedule is tuned with): 32-bit
// accesses to the sliders (load + store each), 64-bit load and 32-bit store of the row pair.  The two worlds of a
// half-warp sit 16 banks apart (World2's slot permutation), all worlds of a warp `lpw` banks apart.
inline long sweep_wavefronts(const std::vector<int>& step_d, int lpw, int esize) {
  const int wpw = 32 / lpw, nslot = (int)step_d.size() / 2, nstep = nslot / lpw - 1;
  long total = 0;
  auto worst_bank = [&](const std::vector<long>& word, int lo, int hi, int nbank, int unit) {
    int worst = 0;
    for (int b = 0; b < nbank; b++) {
      std::vector<long> seen;
      for (int i = lo; i < hi; i++) { if (word[i] < 0) continue; const long w = word[i] / unit; if (w % nbank == b && std::find(seen.begin(), seen.end(), w) == seen.end()) seen.push_back(w); }
      worst = std::max(worst, (int)seen.size());
    }
    return worst;
  };
  for (int s = 0; s < nstep; s++) {
    std::vector<long> a1, a2, rw;
    for (int g = 0; g < wpw; g++) {
      const int slot = wpw > 1 ? (g % (wpw / 2)) * 2 + g / (wpw / 2) : 0;
      for (int k = 0; k < lpw; k++) {
        const unsigned x = (unsigned)step_d[2 * (s * lpw + k)], y = (unsigned)step_d[2 * (s * lpw + k) + 1];
        const long goff = (long)slot * lpw + 4096L * slot;   // worlds sit lpw banks apart (plus whole multiples of 32 words)
        const bool valid = (y >> 30) & 1, has2 = (x >> 16) != 0xffffu;   // (the unpredicated variant also touches the dummies: not modelled)
        a1.push_back(valid ? goff + (x & 0xffff) / 4 : -1); a2.push_back(valid && has2 ? goff + (x >> 16) / 4 : -1);
        rw.push_back(valid ? goff + (y & 0x3fffffffu) / 4 : -1);
      }
    }
    total += 2 * worst_bank(a1, 0, 32, 32, 1) + 2 * worst_bank(a2, 0, 32, 32, 1) + worst_bank(rw, 0, 32, 32, 1);
    if (esize == 4) total += worst_bank(rw, 0, 16, 16, 2) + worst_bank(rw, 16, 32, 16, 2);      // 64-bit load: two half-warps
    else total += worst_bank(rw, 0, 32, 32, 1);
  }
  return total;
}

// the schedule the kernel runs: the target length (critical path + slack) with the least estimated cost
inline void build_step_tables(const PlanDims& D, const std::vector<int>& itab, int lpw, int esize, std::vector<int>& step_d,
                              std::vector<int>& perm, bool avoid_conflicts = true) {
  const int base = build_step_tables_for(D, itab, lpw, esize, 0, step_d, perm);
  if (!avoid_conflicts) return;
  const double per_step = 6.0;                       // fixed cost of a step (issue, barrier) in wavefront units
  double best_cost = 1e300; int best_target = 0;
  for (int target = base; target <= base + base / 4 + 4; target++) {
    std::vector<int> sd, pm;
    const int n = build_step_tables_for(D, itab, lpw, esize, target, sd, pm);
    const double cost = (double)sweep_wavefronts(sd, lpw, esize) + per_step * n;
    if (cost < best_cost) { best_cost = cost; best_target = target; }
  }
  build_step_tables_for(D, itab, lpw, esize, best_target, step_d, perm);
}

inline bool same(const double* a, const double* b, int n) { for (int i = 0; i < n; i++) if (a[i] != b[i]) return false; return true; }

inline Plan build_plan(const void* blob, size_t nbytes) {
  Blob B{(const unsigned char*)blob, nbytes};
  Plan P;
  PlanDims& D = P.d;
  auto opt = B.d("opt");
  SG_REQUIRE(opt.size() >= 12, "opt section");
  D.h = opt[0]; D.g[0] = opt[1]; D.g[1] = opt[2]; D.g[2] = opt[3]; D.iters = (int)opt[4]; D.tol = opt[5];
  D.impratio = opt[6];
  double meaninertia = opt[7];
  auto body_parent = B.i("body_parentid"), body_jntadr = B.i("body_jntadr"), body_jntnum = B.i("body_jntnum"),
       body_weld = B.i("body_weldid"), body_geomadr = B.i("body_geomadr"), body_geomnum = B.i("body_geomnum");
  auto body_pos = B.d("body_pos"), body_quat = B.d("body_quat"), body_ipos = B.d("body_ipos"), body_iquat = B.d("body_iquat"),
       body_mass = B.d("body_mass"), body_inertia = B.d("body_inertia"), body_biw = B.d("body_invweight0");
  auto jnt_type = B.i("jnt_type"), jnt_body = B.i("jnt_bodyid"), jnt_limited = B.i("jnt_limited");
  auto jnt_pos = B.d("jnt_pos"), jnt_axis = B.d("jnt_axis"), jnt_range = B.d("jnt_range"), jnt_stiff = B.d("jnt_stiffness"),
       jnt_margin = B.d("jnt_margin"), jnt_solref = B.d("jnt_solref"), jnt_solimp = B.d("jnt_solimp"), qpos0 = B.d("qpos0"),
       qpos_spring = B.d("qpos_spring");
  auto dof_parent = B.i("dof_parentid");
  auto dof_damping = B.d("dof_damping"), dof_iw = B.d("dof_invweight0");
  auto geom_type = B.i("geom_type"), geom_body = B.i("geom_bodyid"), geom_contype = B.i("geom_contype"),
       geom_conaff = B.i("geom_conaffinity"), geom_condim = B.i("geom_condim");
  auto geom_pos = B.d("geom_pos"), geom_quat = B.d("geom_quat"), geom_size = B.d("geom_size"), geom_friction = B.d("geom_friction"),
       geom_solref = B.d("geom_solref"), geom_solimp = B.d("geom_solimp"), geom_margin = B.d("geom_margin"), geom_gap = B.d("geom_gap"),
       geom_solmix = B.d("geom_solmix"), geom_rbound = B.d("geom_rbound");
  auto site_body = B.i("site_bodyid");
  auto site_pos = B.d("site_pos"), site_quat = B.d("site_quat");
  auto ten_type = B.i("tendon_type"), ten_adr = B.i("tendon_adr"), ten_num = B.i("tendon_num"), wrap_obj = B.i("wrap_objid");
  auto ten_stiff = B.d("tendon_stiffness"), ten_damp = B.d("tendon_damping"), ten_l0 = B.d("tendon_length0"),
       ten_lspring = B.d("tendon_lengthspring"), ten_iw = B.d("tendon_invweight0"), wrap_prm = B.d("wrap_prm");
  auto eq_type = B.i("eq_type"), eq_o1 = B.i("eq_obj1id"), eq_o2 = B.i("eq_obj2id");
  auto eq_data = B.d("eq_data"), eq_solref = B.d("eq_solref"), eq_solimp = B.d("eq_solimp");
  auto act_trn = B.i("actuator_trnid");
  auto act_gear = B.d("actuator_gear"), act_tc = B.d("actuator_timeconst"), act_gain = B.d("actuator_gain"), act_bias = B.d("actuator_bias");
  auto sens_type = B.i("sensor_type"), sens_obj = B.i("sensor_objid"), sens_adr = B.i("sensor_adr");

  const int nbody = (int)body_parent.size(), nv = (int)jnt_type.size(), ngeom = (int)geom_type.size();
  const int ntendon = (int)ten_type.size(), neq = (int)eq_type.size(), nu = (int)act_trn.size(), nsens = (int)sens_type.size();
  P.ngeom = ngeom; P.neq = neq;
  D.nv = nv; D.nu = nu; D.nsd = 3 * nsens; D.nsens = nsens;
  SG_REQUIRE(nsens <= MAXSENS, "too many sensors");
  for (int i = 0; i < nv; i++) SG_REQUIRE(qpos0[i] == 0 && qpos_spring[i] == 0, "non-zero qpos0/springref");

  // static world transforms of bodies welded to the world
  std::vector<double> wpos(3 * nbody, 0.0), wrot(9 * nbody, 0.0);
  wrot[0] = wrot[4] = wrot[8] = 1;
  auto compose_static = [&](int b) {
    int p = body_parent[b];
    double R[9], t[3];
    h_quat2mat(&body_quat[4 * b], R);
    h_matvec3(&wrot[9 * p], &body_pos[3 * b], t);
    for (int k = 0; k < 3; k++) wpos[3 * b + k] = wpos[3 * p + k] + t[k];
    h_matmul3(&wrot[9 * p], R, &wrot[9 * b]);
  };
  for (int b = 1; b < nbody; b++) if (body_weld[b] == 0) compose_static(b);

  // ---- dofs: hinges (finger chains) first, then sliders (shell) ----
  int nfd = 0;
  while (nfd < nv && jnt_type[nfd] == JNT_HINGE) nfd++;
  for (int i = nfd; i < nv; i++) SG_REQUIRE(jnt_type[i] == JNT_SLIDE, "hinge dofs must precede slide dofs");
  const int ns = nv - nfd;
  SG_REQUIRE(ns > 0, "no composite shell (slide joints) found");
  SG_REQUIRE(nfd <= MAXFD, "too many finger dofs");
  D.nfd = nfd; D.ns = ns;

  // chains = dof trees among the hinge dofs; must be serial
  int nchain = 0;
  std::vector<int> dof_chain(nfd, -1), dof_local(nfd, -1);
  for (int i = 0; i < nfd; i++) {
    SG_REQUIRE(dof_damping[i] == 0 && jnt_stiff[i] == 0, "finger joints with stiffness/damping");
    if (dof_parent[i] < 0) {
      SG_REQUIRE(nchain < MAXCHAIN, "too many finger chains");
      D.chain_dof0[nchain] = i; D.ncd[nchain] = 1; dof_chain[i] = nchain; dof_local[i] = 0; nchain++;
    } else {
      SG_REQUIRE(dof_parent[i] == i - 1, "finger dof tree is not a serial chain");
      int c = dof_chain[i - 1];
      dof_chain[i] = c; dof_local[i] = D.ncd[c]++;
      SG_REQUIRE(D.ncd[c] <= MAXCD, "finger chain too long");
    }
  }
  D.nchain = nchain;

  auto alloc_d = [&](size_t n) { size_t r = P.tab.size(); P.tab.resize(r + n, 0.0); return (int)r; };
  auto alloc_i = [&](size_t n) { size_t r = P.itab.size(); P.itab.resize(r + n, 0); return (int)r; };

  // ---- chain descriptors ----
  D.o_chain = alloc_d((size_t)MAXCHAIN * CH_STRIDE);
  std::map<int, std::pair<int, int>> body_to_chain;  // body id -> (chain, k)
  for (int c = 0; c < nchain; c++) {
    double* ch = &P.tab[D.o_chain + c * CH_STRIDE];
    int nb = 0, lastbody = -1;
    for (int j = 0; j < D.ncd[c]; j++) {
      int dof = D.chain_dof0[c] + j, b = jnt_body[dof];
      if (b != lastbody) {
        SG_REQUIRE(nb < MAXCB, "too many bodies in a finger chain");
        if (nb == 0) {
          int p = body_parent[b];
          SG_REQUIRE(body_weld[p] == 0, "finger chain must hang off a static body");
          for (int k = 0; k < 3; k++) ch[CH_BASEPOS + k] = wpos[3 * p + k];
          for (int k = 0; k < 9; k++) ch[CH_BASEROT + k] = wrot[9 * p + k];
        } else SG_REQUIRE(body_parent[b] == lastbody, "finger chain bodies must be parent-child");
        double* cb = ch + CH_BODY + nb * CB_STRIDE;
        for (int k = 0; k < 3; k++) cb[CB_POS + k] = body_pos[3 * b + k];
        h_quat2mat(&body_quat[4 * b], cb + CB_ROT);
        for (int k = 0; k < 3; k++) cb[CB_IPOS + k] = body_ipos[3 * b + k];
        h_quat2mat(&body_iquat[4 * b], cb + CB_IROT);
        cb[CB_MASS] = body_mass[b];
        for (int k = 0; k < 3; k++) cb[CB_INERTIA + k] = body_inertia[3 * b + k];
        SG_REQUIRE(body_geomnum[b] == 1 && geom_type[body_geomadr[b]] == GEOM_BOX, "finger bodies must carry exactly one box geom");
        int g = body_geomadr[b];
        for (int k = 0; k < 3; k++) cb[CB_GPOS + k] = geom_pos[3 * g + k];
        h_quat2mat(&geom_quat[4 * g], cb + CB_GROT);
        for (int k = 0; k < 3; k++) cb[CB_GSIZE + k] = geom_size[3 * g + k];
        cb[CB_BIW] = body_biw[2 * b];
        body_to_chain[b] = {c, nb};
        lastbody = b; nb++;
      }
      double* cd = ch + CH_DOF + j * CD_STRIDE;
      cd[CD_BODY] = nb - 1;
      for (int k = 0; k < 3; k++) { cd[CD_AXIS + k] = jnt_axis[3 * dof + k]; cd[CD_JPOS + k] = jnt_pos[3 * dof + k]; }
      cd[CD_LO] = jnt_range[2 * dof]; cd[CD_HI] = jnt_range[2 * dof + 1]; cd[CD_LIMITED] = jnt_limited[dof];
      cd[CD_IW] = dof_iw[dof];
      SG_REQUIRE(jnt_margin[dof] == 0, "joint limit margin");
      SG_REQUIRE(same(&jnt_solref[2 * dof], &jnt_solref[0], 2) && same(&jnt_solimp[5 * dof], &jnt_solimp[0], 5), "per-joint limit solref/solimp");
    }
    D.ncb[c] = nb;
  }
  // bodies with joints must all be chain bodies or shell bodies
  auto solparams = [&](const double* solref, const double* solimp, double& K, double& Bd, double* si) {
    for (int k = 0; k < 5; k++) si[k] = solimp[k];
    si[0] = std::fmin(0.9999, std::fmax(0.0001, si[0])); si[1] = std::fmin(0.9999, std::fmax(0.0001, si[1]));
    si[2] = std::fmax(0.0, si[2]); si[3] = std::fmin(0.9999, std::fmax(0.0001, si[3])); si[4] = std::fmax(1.0, si[4]);
    double dmax = si[1];
    if (solref[0] > 0) {
      double tc = std::fmax(solref[0], 2 * D.h);
      K = 1 / std::fmax(1e-15, dmax * dmax * tc * tc * solref[1] * solref[1]);
      Bd = 2 / std::fmax(1e-15, dmax * tc);
    } else { K = -solref[0] / std::fmax(1e-15, dmax * dmax); Bd = -solref[1] / std::fmax(1e-15, dmax); }
  };
  if (nfd > 0) solparams(&jnt_solref[0], &jnt_solimp[0], D.lim_K, D.lim_B, D.lim_solimp);

  // ---- shell sliders ----
  const int objroot = body_parent[jnt_body[nfd]];
  SG_REQUIRE(body_weld[objroot] == 0, "composite centre body must be static (freejoint variant is not restated yet)");
  for (int k = 0; k < 3; k++) D.obj_pos[k] = wpos[3 * objroot + k];
  D.o_sl_axis = alloc_d(3 * ns); D.o_sl_cap0 = alloc_d(3 * ns); D.o_sl_k0 = alloc_d(ns); D.o_sl_d0 = alloc_d(ns);
  D.o_sl_m = alloc_d(ns); D.o_sl_tc = alloc_d(ns); D.o_sl_biw = alloc_d(ns); D.o_sl_iw = alloc_d(ns);
  D.io_kmask = alloc_i(ns);
  P.stiff_mask.assign(nv, 0);
  int capg0 = -1;
  for (int e = 0; e < ns; e++) {
    int dof = nfd + e, b = jnt_body[dof];
    SG_REQUIRE(body_parent[b] == objroot && body_jntnum[b] == 1 && dof_parent[dof] < 0, "shell bodies must be single-slider children of the centre body");
    SG_REQUIRE(!jnt_limited[dof], "limited shell joints");
    SG_REQUIRE(body_geomnum[b] == 1 && geom_type[body_geomadr[b]] == GEOM_CAPSULE, "shell bodies must carry exactly one capsule");
    int g = body_geomadr[b];
    if (capg0 < 0) capg0 = g;
    SG_REQUIRE(g == capg0 + e, "shell capsule geoms must be consecutive");
    SG_REQUIRE(geom_size[3 * g] == geom_size[3 * capg0] && geom_size[3 * g + 1] == geom_size[3 * capg0 + 1], "shell capsules must share one size");
    // body frame in the frame of the centre body, then world (centre body is static)
    double Rb[9], Rw[9], t[3], ax[3], gp[3];
    h_quat2mat(&body_quat[4 * b], Rb);
    h_matmul3(&wrot[9 * objroot], Rb, Rw);
    h_matvec3(Rw, &jnt_axis[3 * dof], ax);
    SG_REQUIRE(jnt_pos[3 * dof] == 0 && jnt_pos[3 * dof + 1] == 0 && jnt_pos[3 * dof + 2] == 0, "shell joint anchors must be at the body origin");
    // capsule axis must be the slide axis direction (composite: both local z)
    double Rg[9], Rgw[9];
    h_quat2mat(&geom_quat[4 * g], Rg);
    h_matmul3(Rw, Rg, Rgw);
    SG_REQUIRE(std::fabs(Rgw[2] - ax[0]) < 1e-12 && std::fabs(Rgw[5] - ax[1]) < 1e-12 && std::fabs(Rgw[8] - ax[2]) < 1e-12, "capsule axis must equal the slide axis");
    h_matvec3(&wrot[9 * objroot], &body_pos[3 * b], t);     // body origin relative to the centre body origin (world axes)
    h_matvec3(Rw, &geom_pos[3 * g], gp);
    for (int k = 0; k < 3; k++) { P.tab[D.o_sl_axis + 3 * e + k] = ax[k]; P.tab[D.o_sl_cap0 + 3 * e + k] = t[k] + gp[k]; }
    P.tab[D.o_sl_k0 + e] = jnt_stiff[dof]; P.tab[D.o_sl_d0 + e] = dof_damping[dof];
    P.tab[D.o_sl_m + e] = body_mass[b]; P.tab[D.o_sl_biw + e] = body_biw[2 * b]; P.tab[D.o_sl_iw + e] = dof_iw[dof];
  }
  P.first_capsule_geom = capg0;
  D.cap_r = geom_size[3 * capg0]; D.cap_hl = geom_size[3 * capg0 + 1];

  // ---- tendons: tendon 0 = fixed volume tendon over the shell; spatial tendons drive the chains ----
  SG_REQUIRE(ntendon >= 1 && ten_type[0] == TEN_FIXED, "tendon 0 must be the composite's fixed tendon");
  for (int w = ten_adr[0]; w < ten_adr[0] + ten_num[0]; w++) {
    SG_REQUIRE(wrap_obj[w] >= nfd, "fixed tendon must only wrap shell joints");
    P.tab[D.o_sl_tc + wrap_obj[w] - nfd] = wrap_prm[w];
  }
  D.ten_iw = ten_iw[0]; D.ten_k0 = ten_stiff[0]; D.ten_d0 = ten_damp[0]; D.ten_lspring = ten_lspring[0]; D.ten_l0 = ten_l0[0];
  for (int t = 1; t < ntendon; t++) {
    SG_REQUIRE(ten_type[t] == TEN_SPATIAL && ten_num[t] == 2, "only two-site spatial tendons besides the composite tendon");
    SG_REQUIRE(ten_stiff[t] == 0 && ten_damp[t] == 0, "spatial tendon stiffness/damping");
    int s0 = wrap_obj[ten_adr[t]], s1 = wrap_obj[ten_adr[t] + 1];
    SG_REQUIRE(body_weld[site_body[s0]] == 0, "spatial tendon must start on a static body");
    auto it = body_to_chain.find(site_body[s1]);
    SG_REQUIRE(it != body_to_chain.end(), "spatial tendon must end on a finger body");
    double* ct = &P.tab[D.o_chain + it->second.first * CH_STRIDE + CH_TEN];
    SG_REQUIRE(ct[CT_HAS] == 0, "more than one tendon per finger chain");
    ct[CT_HAS] = 1;
    double tp[3];
    h_matvec3(&wrot[9 * site_body[s0]], &site_pos[3 * s0], tp);
    for (int k = 0; k < 3; k++) { ct[CT_S0 + k] = wpos[3 * site_body[s0] + k] + tp[k]; ct[CT_S1 + k] = site_pos[3 * s1 + k]; }
    ct[CT_BODY] = it->second.second;
    ct[CT_ACT] = -1;
    for (int u = 0; u < nu; u++) if (act_trn[u] == t) {
      SG_REQUIRE(ct[CT_ACT] < 0, "more than one actuator per tendon");
      SG_REQUIRE(act_bias[3 * u] == 0 && act_bias[3 * u + 1] == 0 && act_bias[3 * u + 2] == 0, "actuator bias");
      ct[CT_ACT] = u; ct[CT_GEAR] = act_gear[u]; ct[CT_GAIN] = act_gain[u]; ct[CT_TIMECONST] = act_tc[u];
    }
  }
  for (int u = 0; u < nu; u++) SG_REQUIRE(act_trn[u] >= 1, "actuators must act on the spatial tendons");

  // ---- equality rows + Gauss-Seidel level schedule ----
  SG_REQUIRE(neq >= 2 && eq_type[neq - 1] == EQ_TENDON && eq_o1[neq - 1] == 0 && eq_o2[neq - 1] < 0, "last equality must be the volume-tendon equality");
  const int nrow = neq - 1;
  D.nrow = nrow;
  std::vector<int> level(nrow), lastlev(ns, 0);
  int maxlev = 0;
  for (int r = 0; r < nrow; r++) {
    SG_REQUIRE(eq_type[r] == EQ_JOINT, "equalities before the tendon row must be joint equalities");
    const double* dat = &eq_data[5 * r];
    SG_REQUIRE(dat[0] == 0 && dat[1] == 1 && dat[2] == 0 && dat[3] == 0 && dat[4] == 0, "joint equality polycoef must be 0 1 0 0 0");
    SG_REQUIRE(same(&eq_solref[2 * r], &eq_solref[0], 2) && same(&eq_solimp[5 * r], &eq_solimp[0], 5), "joint equalities must share solref/solimp");
    int d1 = eq_o1[r] - nfd, d2 = eq_o2[r] >= 0 ? eq_o2[r] - nfd : -1;
    SG_REQUIRE(d1 >= 0 && (eq_o2[r] < 0 || d2 >= 0), "joint equalities must couple shell joints");
    int lv = lastlev[d1];
    if (d2 >= 0 && lastlev[d2] > lv) lv = lastlev[d2];
    lv += 1;
    level[r] = lv; lastlev[d1] = lv;
    if (d2 >= 0) lastlev[d2] = lv;
    if (lv > maxlev) maxlev = lv;
  }
  solparams(&eq_solref[0], &eq_solimp[0], D.eqj_K, D.eqj_B, D.eqj_solimp);
  solparams(&eq_solref[2 * (neq - 1)], &eq_solimp[5 * (neq - 1)], D.eqt_K, D.eqt_B, D.eqt_solimp);
  {
    const double* dat = &eq_data[5 * (neq - 1)];
    SG_REQUIRE(dat[0] == 0, "tendon equality offset");
  }
  // schedule: rows sorted by (level, original order); levels wider than a warp are split
  std::vector<std::vector<int>> bylev(maxlev + 1);
  for (int r = 0; r < nrow; r++) bylev[level[r]].push_back(r);
  std::vector<int> lev_start;
  std::vector<int> sched;  // position -> eq row
  for (int lv = 1; lv <= maxlev; lv++) {
    for (size_t k = 0; k < bylev[lv].size(); k++) {
      if (k % 32 == 0) lev_start.push_back((int)sched.size());
      sched.push_back(bylev[lv][k]);
    }
  }
  lev_start.push_back((int)sched.size());
  D.nlev = (int)lev_start.size() - 1;
  D.io_row_d1 = alloc_i(nrow); D.io_row_d2 = alloc_i(nrow); D.io_lev_start = alloc_i(D.nlev + 1);
  D.io_dof_rows = alloc_i((size_t)ns * MAXDOFROWS);
  for (int i = 0; i < ns * MAXDOFROWS; i++) P.itab[D.io_dof_rows + i] = -1;
  std::vector<int> cnt(ns, 0);
  for (int p = 0; p < nrow; p++) {
    int r = sched[p];
    int d1 = eq_o1[r] - nfd, d2 = eq_o2[r] >= 0 ? eq_o2[r] - nfd : -1;
    P.itab[D.io_row_d1 + p] = d1; P.itab[D.io_row_d2 + p] = d2;
    SG_REQUIRE(cnt[d1] < MAXDOFROWS, "too many equality rows on one joint");
    P.itab[D.io_dof_rows + d1 * MAXDOFROWS + cnt[d1]++] = p * 2;
    if (d2 >= 0) { SG_REQUIRE(cnt[d2] < MAXDOFROWS, "too many equality rows on one joint"); P.itab[D.io_dof_rows + d2 * MAXDOFROWS + cnt[d2]++] = p * 2 + 1; }
  }
  for (int l = 0; l <= D.nlev; l++) P.itab[D.io_lev_start + l] = lev_start[l];
  P.sched_eq = sched;
  // packed per-row descriptors of the level sweep
  SG_REQUIRE(ns < 0xffff, "too many shell joints for the packed row descriptors");
  D.io_row_d12 = alloc_i(nrow);
  D.o_row_iw = alloc_d(2 * (size_t)nrow);
  D.o_sl_tciw = alloc_d(ns);
  for (int p = 0; p < nrow; p++) {
    const int d1 = P.itab[D.io_row_d1 + p], d2 = P.itab[D.io_row_d2 + p];
    P.itab[D.io_row_d12 + p] = d1 | ((d2 >= 0 ? d2 : 0xffff) << 16);
    P.tab[D.o_row_iw + 2 * p] = 1.0 / P.tab[D.o_sl_m + d1];
    P.tab[D.o_row_iw + 2 * p + 1] = d2 >= 0 ? 1.0 / P.tab[D.o_sl_m + d2] : 0.0;
  }
  for (int e = 0; e < ns; e++) P.tab[D.o_sl_tciw + e] = P.tab[D.o_sl_tc + e] / P.tab[D.o_sl_m + e];

  // ---- contact parameters must be uniform over all geoms ----
  for (int g = 0; g < ngeom; g++) {
    SG_REQUIRE(same(&geom_solref[2 * g], &geom_solref[0], 2) && same(&geom_solimp[5 * g], &geom_solimp[0], 5), "per-geom solref/solimp");
    SG_REQUIRE(same(&geom_friction[3 * g], &geom_friction[0], 3), "per-geom friction");
    SG_REQUIRE(geom_margin[g] == 0 && geom_gap[g] == 0, "geom margin/gap");
    SG_REQUIRE(geom_solmix[g] == geom_solmix[0], "per-geom solmix");
  }
  solparams(&geom_solref[0], &geom_solimp[0], D.con_K, D.con_B, D.con_solimp);
  D.con_fr = geom_friction[0];

  // ---- colliders (plane + boxes) and the candidate pair list in MuJoCo's contact order ----
  D.o_coll = alloc_d((size_t)MAXCOLL * CO_STRIDE);
  std::vector<int> geom_coll(ngeom, -1);
  int ncoll = 0;
  D.has_sphere = 0;
  for (int g = 0; g < ngeom; g++) {
    int b = geom_body[g], t = geom_type[g];
    if (t == GEOM_CAPSULE) { SG_REQUIRE(g >= capg0 && g < capg0 + ns, "capsules outside the shell"); continue; }
    if (t == GEOM_SPHERE) {
      SG_REQUIRE(!D.has_sphere && b == objroot, "only the composite's centre sphere is supported");
      D.has_sphere = 1; P.center_geom = g; D.sph_r = geom_size[3 * g];
      double tp[3]; h_matvec3(&wrot[9 * b], &geom_pos[3 * g], tp);
      for (int k = 0; k < 3; k++) D.sph_pos[k] = tp[k];
      continue;
    }
    SG_REQUIRE(t == GEOM_PLANE || t == GEOM_BOX, "geom type");
    SG_REQUIRE(ncoll < MAXCOLL, "too many plane/box geoms");
    double* co = &P.tab[D.o_coll + ncoll * CO_STRIDE];
    co[CO_TYPE] = t; co[CO_RBOUND] = geom_rbound[g]; co[CO_BIW] = body_biw[2 * b];
    for (int k = 0; k < 3; k++) co[CO_SIZE + k] = geom_size[3 * g + k];
    auto it = body_to_chain.find(b);
    if (it != body_to_chain.end()) { co[CO_CHAIN] = it->second.first; co[CO_BODY] = it->second.second; }
    else {
      SG_REQUIRE(body_weld[b] == 0, "box on a moving body that is not a finger body");
      co[CO_CHAIN] = -1; co[CO_BODY] = -1;
      double R[9], tp[3];
      h_quat2mat(&geom_quat[4 * g], R); h_matmul3(&wrot[9 * b], R, co + CO_ROT);
      h_matvec3(&wrot[9 * b], &geom_pos[3 * g], tp);
      for (int k = 0; k < 3; k++) co[CO_POS + k] = wpos[3 * b + k] + tp[k];
    }
    geom_coll[g] = ncoll; P.coll_geom.push_back(g); ncoll++;
  }
  D.ncoll = ncoll;
  std::vector<int> pt, pa, pb;
  auto weldparent = [&](int w) { return body_weld[body_parent[w]]; };
  for (int b1 = 0; b1 < nbody; b1++) {
    if (!body_geomnum[b1]) continue;
    for (int b2 = b1 + 1; b2 < nbody; b2++) {
      if (!body_geomnum[b2]) continue;
      int w1 = body_weld[b1], w2 = body_weld[b2];
      if (w1 == w2) continue;
      if (w1 != 0 && w2 != 0 && (w1 == weldparent(w2) || w2 == weldparent(w1))) continue;
      for (int a = body_geomadr[b1]; a < body_geomadr[b1] + body_geomnum[b1]; a++)
        for (int b = body_geomadr[b2]; b < body_geomadr[b2] + body_geomnum[b2]; b++) {
          if (!((geom_contype[a] & geom_conaff[b]) || (geom_contype[b] & geom_conaff[a]))) continue;
          int g1 = a, g2 = b;
          if (geom_type[g1] > geom_type[g2]) std::swap(g1, g2);
          int t1 = geom_type[g1], t2 = geom_type[g2];
          SG_REQUIRE(std::max(geom_condim[g1], geom_condim[g2]) == 3, "contact condim must be 3");
          if (t1 == GEOM_PLANE && t2 == GEOM_CAPSULE) { pt.push_back(PAIR_PLANE_CAPSULE); pa.push_back(geom_coll[g1]); pb.push_back(g2 - capg0); }
          else if (t1 == GEOM_CAPSULE && t2 == GEOM_BOX) { pt.push_back(PAIR_BOX_CAPSULE); pa.push_back(geom_coll[g2]); pb.push_back(g1 - capg0); }
          else if (t1 == GEOM_SPHERE && t2 == GEOM_BOX) { pt.push_back(PAIR_SPHERE_BOX); pa.push_back(geom_coll[g2]); pb.push_back(0); }
          else if (t1 == GEOM_BOX && t2 == GEOM_BOX) { pt.push_back(PAIR_BOX_BOX); pa.push_back(geom_coll[g1]); pb.push_back(geom_coll[g2]); }
          else if (t1 == GEOM_PLANE && t2 == GEOM_BOX) { pt.push_back(PAIR_PLANE_BOX); pa.push_back(geom_coll[g1]); pb.push_back(geom_coll[g2]); }
          else SG_REQUIRE(false, "geom pair type outside the restated narrowphase set");
        }
    }
  }
  D.npair = (int)pt.size();
  D.io_pair_t = alloc_i(D.npair); D.io_pair_a = alloc_i(D.npair); D.io_pair_b = alloc_i(D.npair);
  for (int p = 0; p < D.npair; p++) { P.itab[D.io_pair_t + p] = pt[p]; P.itab[D.io_pair_a + p] = pa[p]; P.itab[D.io_pair_b + p] = pb[p]; }
  // run-length form of the same list (same order): a run is a block {type, first collider a0, na, first second geom b0,
  // nb} standing for the pairs (a0 + i, b0 + j) in the order j-major, i-minor (MuJoCo walks body pairs and, inside a body
  // pair, geom x geom: a body with two boxes against the shell gives a-minor runs).  The device broadphase walks runs, so
  // the pair tables are not touched at all.
  {
    std::vector<int> runs;
    for (int p = 0; p < D.npair;) {
      int na = 1;
      while (p + na < D.npair && pt[p + na] == pt[p] && pb[p + na] == pb[p] && pa[p + na] == pa[p] + na) na++;
      int nb = 1;
      for (;;) {
        const int q = p + nb * na;
        if (q + na > D.npair) break;
        bool ok = true;
        for (int i = 0; i < na && ok; i++) ok = pt[q + i] == pt[p] && pa[q + i] == pa[p] + i && pb[q + i] == pb[p] + nb;
        if (!ok) break;
        nb++;
      }
      runs.push_back(pt[p]); runs.push_back(pa[p] | (na << 8)); runs.push_back(pb[p]); runs.push_back(nb);
      p += na * nb;
    }
    D.nrun = (int)runs.size() / 4;
    D.io_run = alloc_i(runs.size());
    for (size_t i = 0; i < runs.size(); i++) P.itab[D.io_run + i] = runs[i];
    SG_REQUIRE(ns < (1 << 20) && ncoll < 32, "candidate encoding");
  }

  // ---- sensors ----
  D.o_sens = alloc_d((size_t)MAXSENS * SE_STRIDE);
  for (int s = 0; s < nsens; s++) {
    double* se = &P.tab[D.o_sens + s * SE_STRIDE];
    int site = sens_obj[s];
    auto it = body_to_chain.find(site_body[site]);
    SG_REQUIRE(it != body_to_chain.end(), "sensors must sit on finger bodies");
    SG_REQUIRE(sens_type[s] == SENS_ACCEL || sens_type[s] == SENS_GYRO, "sensor type");
    se[SE_TYPE] = sens_type[s]; se[SE_CHAIN] = it->second.first; se[SE_BODY] = it->second.second; se[SE_ADR] = sens_adr[s];
    for (int k = 0; k < 3; k++) se[SE_POS + k] = site_pos[3 * site + k];
    h_quat2mat(&site_quat[4 * site], se + SE_ROT);
  }

  D.impr_scale = 1.0 / (meaninertia * (nv > 1 ? nv : 1));
  D.stiff_tendon0 = 0;
  D.maxcon = 0; D.maxcand = 0;   // filled by the caller (capacity policy)
  P.geom_mask.assign(ngeom, 0);
  return P;
}

}  // namespace sg
