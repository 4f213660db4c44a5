// odg_prep.h — host-side preparation of the constants the step kernel reads: OdgModel (doubles,
// MuJoCo layout) + OdgEnvConfig -> DevConst (__constant__), per-leg constant table and hull-vertex
// table (staged into shared memory by every block). Pure host C++, no CUDA calls; shared by
// odg_sim.cu and the test-only lane emulator.
#pragma once

#include <cmath>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/odg.h"
#include "odg_core.cuh"

namespace odg {

struct Prepared {
  DevConst C;
  std::vector<float> lc;        // [njl][LC_COUNT][4]
  std::vector<float> gc;        // [nslot][GC_COUNT][4], then (DevConst::oct_off / idx_off, in floats) the support-vertex
                                // candidate table [nslot][24 cells][4 legs] of (start | count << 16) and the byte lists
  std::vector<float> vert;      // [rows][4 legs][4 floats]
};

// Support-vertex candidates of a hull for one cell of query directions.
// The collision pass looks for the hull vertex that is extreme towards the floor and towards three directions tilted
// by `tilt` off it (odg_core.cuh: collision). A vertex v can win for a direction d only if d lies in v's normal cone
// {d : d.(v - u) >= 0 for all hull vertices u}. Directions are binned into 24 cells: dominant axis of d (3) x the signs
// of its components (8), i.e. a quarter of a cube face each. All four query directions of one pass lie in the cell of
// the floor direction widened by the tilt, so per cell only the vertices whose normal cone meets the widened cell
// need to be scanned. The test is exact up to a tolerance that only adds vertices: on the plane d_axis = +-1 the
// widened cell is a square, and the normal cone clips it half-plane by half-plane (Sutherland-Hodgman); the vertex
// is a candidate iff something is left.
inline bool hull_vertex_is_candidate(const double (*verts)[3], int n, int v, int axis, const int sigma[3], double w_lo,
                                     double w_hi, double tol) {
  struct P3 { double x[3]; };
  std::vector<P3> poly, next;
  const int b = (axis + 1) % 3, c = (axis + 2) % 3;
  const double lo = -w_lo, hi = 1.0 + w_hi;
  const double cb[4] = { lo, hi, hi, lo }, cc[4] = { lo, lo, hi, hi };
  for (int i = 0; i < 4; i++) {
    P3 p; p.x[axis] = sigma[axis]; p.x[b] = sigma[b] * cb[i]; p.x[c] = sigma[c] * cc[i];
    poly.push_back(p);
  }
  for (int u = 0; u < n && !poly.empty(); u++) {
    if (u == v) continue;
    const double nx = verts[v][0] - verts[u][0], ny = verts[v][1] - verts[u][1], nz = verts[v][2] - verts[u][2];
    if (nx == 0.0 && ny == 0.0 && nz == 0.0) continue;         // duplicate vertex
    auto h = [&](const P3& p) { return nx * p.x[0] + ny * p.x[1] + nz * p.x[2] + tol; };
    next.clear();
    const size_t m = poly.size();
    for (size_t i = 0; i < m; i++) {
      const P3& a = poly[i]; const P3& bb = poly[(i + 1) % m];
      const double ha = h(a), hb = h(bb);
      if (ha >= 0.0) next.push_back(a);
      if ((ha >= 0.0) != (hb >= 0.0)) {
        const double t = ha / (ha - hb);
        P3 q; for (int j = 0; j < 3; j++) q.x[j] = a.x[j] + t * (bb.x[j] - a.x[j]);
        next.push_back(q);
      }
    }
    poly.swap(next);
  }
  return !poly.empty();
}

inline float clampf(double v, double lo, double hi) { return (float)std::fmin(hi, std::fmax(lo, v)); }

inline void solref_kb(const OdgModel& m, const double* solref, const double* solimp, double* K, double* B) {
  double dmax = std::fmin(0.9999, std::fmax(0.0001, solimp[1]));
  if (solref[0] > 0) {
    double tc = std::fmax(solref[0], 2 * m.timestep), dr = solref[1];
    *K = 1 / std::fmax(1e-15, dmax * dmax * tc * tc * dr * dr);
    *B = 2 / std::fmax(1e-15, dmax * tc);
  } else {
    *K = -solref[0] / std::fmax(1e-15, dmax * dmax);
    *B = -solref[1] / std::fmax(1e-15, dmax);
  }
}
inline void pack_imp(const double* solimp, float* out) {
  out[0] = clampf(solimp[0], 0.0001, 0.9999); out[1] = clampf(solimp[1], 0.0001, 0.9999);
  out[2] = (float)std::fmax(1e-15, solimp[2]); out[3] = clampf(solimp[3], 0.0001, 0.9999);
  out[4] = (float)std::fmax(1.0, solimp[4]);
}
inline void quat2mat(const double* q, double* M) {
  double w = q[0], x = q[1], y = q[2], z = q[3];
  M[0] = w * w + x * x - y * y - z * z; M[1] = 2 * (x * y - w * z); M[2] = 2 * (x * z + w * y);
  M[3] = 2 * (x * y + w * z); M[4] = w * w - x * x + y * y - z * z; M[5] = 2 * (y * z - w * x);
  M[6] = 2 * (x * z - w * y); M[7] = 2 * (y * z + w * x); M[8] = w * w - x * x - y * y + z * z;
}

// Returns "" on success, otherwise why the model/config is not supported by the kernel.
inline std::string prepare(const OdgModel& m, const OdgEnvConfig& cfg, uint64_t seed, Prepared* out) {
  DevConst& C = out->C;
  std::memset(&C, 0, sizeof(C));
  if (m.nleg != 4) return "kernel maps one leg per lane: nleg must be 4";
  if (m.njl < 1 || m.njl > kMaxJL) return "njl out of range";
  if (m.cone != 1) return "only cone=elliptic is supported";
  if (m.nu != m.nleg * m.njl) return "one position actuator per hinge joint is expected";
  for (int i = 0; i < 6; i++) if (m.base_damping[i] != 0) return "trunk damping is not supported";
  for (int l = 0; l < m.nleg; l++) for (int j = 0; j < m.njl; j++)
    if (m.damping[l][j] != 0) C.any_damping = 1;             // mj_Euler's implicit joint damping (Go1: go1.xml:9,12)
  if (m.base_armature[3] != m.base_armature[4] || m.base_armature[3] != m.base_armature[5])
    return "trunk rotational armature must be isotropic";
  C.nleg = m.nleg; C.njl = m.njl; C.nq = m.nq; C.nv = m.nv; C.nu = m.nu;
  C.h = (float)m.timestep; C.gx = (float)m.gravity[0]; C.gy = (float)m.gravity[1]; C.gz = (float)m.gravity[2];
  C.impratio = (float)m.impratio;
  C.base_mass = (float)m.base_mass;
  for (int i = 0; i < 3; i++) { C.base_ip[i] = (float)m.base_ipos[i]; C.base_arm_t[i] = (float)m.base_armature[i]; }
  C.base_arm_r = (float)m.base_armature[3];
  const int sidx[6] = { 0, 1, 2, 4, 5, 8 };
  for (int i = 0; i < 6; i++) C.base_I[i] = (float)m.base_inertia[sidx[i]];
  double Kf, Bf, Kl, Bl;
  solref_kb(m, m.dof_solref, m.dof_solimp, &Kf, &Bf);
  solref_kb(m, m.lim_solref, m.lim_solimp, &Kl, &Bl);
  C.B_fl = (float)Bf; C.K_lim = (float)Kl; C.B_lim = (float)Bl;
  pack_imp(m.lim_solimp, C.lim_imp);
  const double d0 = std::fmin(0.9999, std::fmax(0.0001, m.dof_solimp[0]));
  for (int i = 0; i < 6; i++) {
    C.base_fl[i] = (float)m.base_frictionloss[i];
    double R = std::fmax(1e-15, (1 - d0) / d0 * m.base_invweight0[i]);
    C.base_Rfl[i] = (float)R; C.base_Dfl[i] = (float)(1 / R);
  }
  // per-leg joint constants
  const int njl = m.njl;
  out->lc.assign((size_t)njl * LC_COUNT * 4, 0.f);
  auto LC = [&](int f, int j, int l) -> float& { return out->lc[((size_t)j * LC_COUNT + f) * 4 + l]; };
  bool ident = true;
  for (int l = 0; l < 4; l++) for (int j = 0; j < njl; j++) {
    double R[9]; quat2mat(m.body_quat[l][j], R);
    for (int k = 0; k < 9; k++) { LC(LC_BR0 + k, j, l) = (float)R[k]; ident &= (R[k] == ((k % 4 == 0) ? 1.0 : 0.0)); }
    for (int k = 0; k < 3; k++) {
      LC(LC_BP0 + k, j, l) = (float)m.body_pos[l][j][k]; LC(LC_JP0 + k, j, l) = (float)m.jnt_pos[l][j][k];
      LC(LC_JA0 + k, j, l) = (float)m.jnt_axis[l][j][k]; LC(LC_IP0 + k, j, l) = (float)m.ipos[l][j][k];
    }
    LC(LC_MASS, j, l) = (float)m.mass[l][j];
    for (int k = 0; k < 6; k++) LC(LC_IXX + k, j, l) = (float)m.inertia[l][j][sidx[k]];
    LC(LC_LO, j, l) = (float)m.jnt_range[l][j][0]; LC(LC_HI, j, l) = (float)m.jnt_range[l][j][1];
    LC(LC_LIMITED, j, l) = m.jnt_limited[l][j] ? 1.f : 0.f;
    LC(LC_ARM, j, l) = (float)m.armature[l][j]; LC(LC_FL, j, l) = (float)m.frictionloss[l][j];
    double R_ = std::fmax(1e-15, (1 - d0) / d0 * m.dof_invweight0[l][j]);
    LC(LC_RFL, j, l) = (float)R_; LC(LC_DFL, j, l) = (float)(1 / R_);
    LC(LC_DAMP, j, l) = (float)m.damping[l][j]; LC(LC_INVW, j, l) = (float)m.dof_invweight0[l][j];
    LC(LC_HOMEQ, j, l) = (float)m.key_qpos[7 + l * njl + j];
    LC(LC_UIDX, j, l) = 0.f;
  }
  C.body_rot_identity = ident ? 1 : 0;
  // ScaleActionEnvironment.py:8-17: float32 table, thigh [2.36, 2.8], knee [-1.8, -1.20] per actuator (the OpenDOG
  // model). Other models (Go1, which has no walk environment in the reference) map [-1, 1] around the home target.
  const bool opendog = (m.nu == 8 && m.njl == 2);
  const float slo[2] = { 2.36f, -1.8f }, shi[2] = { 2.8f, -1.20f };
  for (int u = 0; u < m.nu; u++) {
    int l = m.act_leg[u], j = m.act_joint[u];
    if (LC(LC_HASACT, j, l) != 0.f) return "more than one actuator per joint";
    LC(LC_HASACT, j, l) = 1.f; LC(LC_UIDX, j, l) = (float)u;
    LC(LC_KP, j, l) = (float)m.act_kp[u]; LC(LC_KV, j, l) = (float)m.act_kv[u];
    LC(LC_CLIM, j, l) = m.act_ctrllimited[u] ? 1.f : 0.f; LC(LC_FLIM, j, l) = m.act_forcelimited[u] ? 1.f : 0.f;
    LC(LC_CLO, j, l) = (float)m.act_ctrlrange[u][0]; LC(LC_CHI, j, l) = (float)m.act_ctrlrange[u][1];
    LC(LC_FLO, j, l) = (float)m.act_forcerange[u][0]; LC(LC_FHI, j, l) = (float)m.act_forcerange[u][1];
    {
      // other models: [-1, 1] -> home -+ d, d = min(0.5 rad, distance of the home target to either end of ctrlrange)
      const double home = m.key_ctrl[u], lo_ = m.act_ctrlrange[u][0], hi_ = m.act_ctrlrange[u][1];
      const double d = std::fmax(0.0, std::fmin(0.5, std::fmin(home - lo_, hi_ - home)));
      LC(LC_SLO, j, l) = opendog ? slo[u & 1] : (float)(home - d);
      LC(LC_SHI, j, l) = opendog ? shi[u & 1] : (float)(home + d);
    }
    C.key_ctrl[u] = (float)m.key_ctrl[u];
  }
  if (cfg.task == ODG_TASK_WALK)
    for (int u = 0; u < m.nu; u++)
      if (m.act_leg[u] != m.act_leg[u - u % m.njl] || m.act_joint[u] != u % m.njl)
        return "walk task expects the actuators of a leg to be consecutive, root to tip";
  for (int i = 0; i < m.nq; i++) C.key_qpos[i] = (float)m.key_qpos[i];
  C.obs_joint_offset = (float)m.key_ctrl[m.nu - 1];       // key_ctrl[0, 7:] (WalkEnvironment.py:116)
  // collision slots: every leg must carry the same sequence of (link, type)
  // per_leg[l][s] = model geom of lane l in slot s, or -1 (empty). Hull / sphere models (OpenDOG; Go1 feet only): every
  // leg carries the same sequence. Models with primitive or trunk colliders (unitree_go1/go1.xml:26-64): slots are
  // aligned link by link (a leg with fewer geoms on a link gets empty slots), and the trunk's colliders are dealt out
  // over the four lanes in further slots with link -1; type and presence then come from the per-lane GC_TYPE table.
  std::vector<int> per_leg[4];
  bool per_lane = false;
  for (int g = 0; g < m.ngeom; g++)
    if (m.geom[g].leg < 0 || m.geom[g].type >= ODG_GEOM_CAPSULE) per_lane = true;
  if (!per_lane) {
    for (int g = 0; g < m.ngeom; g++) per_leg[m.geom[g].leg].push_back(g);
  } else {
    if (m.njl != 3) return "primitive / trunk colliders are compiled into the 3-joint-leg kernel only";
    for (int g = 0; g < m.ngeom; g++) if (m.geom[g].type == ODG_GEOM_HULL) return "hulls and primitive colliders cannot be mixed";
    for (int link = 0; link < m.njl; link++) {
      std::vector<int> on[4]; size_t n = 0;
      for (int g = 0; g < m.ngeom; g++) if (m.geom[g].leg >= 0 && m.geom[g].link == link) on[m.geom[g].leg].push_back(g);
      for (int l = 0; l < 4; l++) n = on[l].size() > n ? on[l].size() : n;
      for (size_t k = 0; k < n; k++) for (int l = 0; l < 4; l++) per_leg[l].push_back(k < on[l].size() ? on[l][k] : -1);
    }
    std::vector<int> trunk;
    for (int g = 0; g < m.ngeom; g++) if (m.geom[g].leg < 0) trunk.push_back(g);
    for (size_t i = 0; i < trunk.size(); i += 4)
      for (int l = 0; l < 4; l++) per_leg[l].push_back(i + l < trunk.size() ? trunk[i + l] : -1);
  }
  C.per_lane_geoms = per_lane ? 1 : 0;
  const int nslot = (int)per_leg[0].size();
  if (nslot > kMaxSlot) return "too many collision geoms per leg";
  for (int l = 1; l < 4; l++) if ((int)per_leg[l].size() != nslot) return "legs differ in collision geoms";
  C.nslot = nslot;
  out->gc.assign((size_t)(nslot > 0 ? nslot : 1) * GC_COUNT * 4, 0.f);
  int rows = 0;
  for (int s = 0; s < nslot; s++) {
    int first = -1;
    for (int l = 0; l < 4; l++) if (first < 0 && per_leg[l][s] >= 0) first = per_leg[l][s];
    const OdgGeom& g0 = m.geom[first];
    int nv = 0;
    for (int l = 0; l < 4; l++) {
      if (per_leg[l][s] < 0) continue;                 // empty slot on this lane: GC_TYPE stays 0
      const OdgGeom& g = m.geom[per_leg[l][s]];
      if (g.link != g0.link || (!per_lane && g.type != g0.type) || g.condim != g0.condim || g.friction != g0.friction ||
          g.friction_torsion != g0.friction_torsion || g.friction_roll != g0.friction_roll || g.margin != g0.margin)
        return "legs differ in collision geom parameters";
      for (int k = 0; k < 2; k++) if (g.solref[k] != g0.solref[k]) return "legs differ in collision geom parameters";
      for (int k = 0; k < 5; k++) if (g.solimp[k] != g0.solimp[k]) return "legs differ in collision geom parameters";
      if (g.condim != 1 && g.condim != 3 && !(g.condim == 6 && m.njl == 3))
        return "contact condim must be 1 or 3 (6 in the 3-joint-leg kernel)";
      if (per_lane) {
        auto G = [&](int f) -> float& { return out->gc[((size_t)s * GC_COUNT + f) * 4 + l]; };
        G(GC_TYPE) = (float)(g.type + 1);
        for (int k = 0; k < 9; k++) G(GC_R0 + k) = (float)g.rot[k];
        for (int k = 0; k < 3; k++) G(GC_S0 + k) = (float)g.size[k];
        if (g.type == ODG_GEOM_SPHERE) G(GC_S0) = (float)g.radius;
      }
      nv = g.vert_count > nv ? g.vert_count : nv;
      out->gc[((size_t)s * GC_COUNT + GC_INVW) * 4 + l] = (float)g.invweight0;
      out->gc[((size_t)s * GC_COUNT + GC_CX) * 4 + l] = (float)g.center[0];
      out->gc[((size_t)s * GC_COUNT + GC_CY) * 4 + l] = (float)g.center[1];
      out->gc[((size_t)s * GC_COUNT + GC_CZ) * 4 + l] = (float)g.center[2];
      if (g.vert_count > 0) {                        // bounding sphere of the hull (bbox centre, max distance)
        double lo[3] = { 1e30, 1e30, 1e30 }, hi[3] = { -1e30, -1e30, -1e30 }, c[3], r2 = 0;
        for (int k = 0; k < g.vert_count; k++) for (int a = 0; a < 3; a++) {
          lo[a] = std::fmin(lo[a], m.vert[g.vert_start + k][a]); hi[a] = std::fmax(hi[a], m.vert[g.vert_start + k][a]);
        }
        for (int a = 0; a < 3; a++) c[a] = 0.5 * (lo[a] + hi[a]);
        for (int k = 0; k < g.vert_count; k++) {
          double d2 = 0; for (int a = 0; a < 3; a++) { double t = m.vert[g.vert_start + k][a] - c[a]; d2 += t * t; }
          r2 = std::fmax(r2, d2);
        }
        for (int a = 0; a < 3; a++) out->gc[((size_t)s * GC_COUNT + GC_BX + a) * 4 + l] = (float)c[a];
        out->gc[((size_t)s * GC_COUNT + GC_BR) * 4 + l] = (float)(std::sqrt(r2) * 1.0001 + 1e-6);
        for (int a = 0; a < 3; a++)             // half extents of the link-frame bounding box (slightly inflated)
          out->gc[((size_t)s * GC_COUNT + GC_HX + a) * 4 + l] = (float)(0.5 * (hi[a] - lo[a]) * 1.0001 + 1e-6);
      }
    }
    C.slot_link[s] = g0.link; C.slot_type[s] = g0.type; C.slot_nvert[s] = nv; C.slot_vstart[s] = rows;
    C.slot_condim[s] = g0.condim;
    // reward_calc:93 body_feet_indices = [4, 7, 10, 13]: the last body of each leg chain
    C.slot_isfoot[s] = (g0.leg >= 0 && g0.mj_body_id == 4 + 3 * g0.leg) ? 1 : 0;
    C.slot_margin[s] = (float)g0.margin; C.slot_radius[s] = (float)g0.radius;
    double K, B; solref_kb(m, g0.solref, g0.solimp, &K, &B);
    C.slot_K[s] = (float)K; C.slot_B[s] = (float)B; pack_imp(g0.solimp, C.slot_imp[s]);
    C.slot_fri[s] = (float)g0.friction;
    C.slot_mu[s] = (float)(g0.friction / std::sqrt(std::fmax(1e-15, m.impratio)));
    { const double mu = (double)C.slot_mu[s]; C.slot_dmk[s] = (float)(1.0 / std::fmax(1e-30, mu * mu * (1.0 + mu * mu))); }
    if (g0.condim == 6) {                            // torsional / rolling rows: R_row = R_slide * mu_slide^2 / mu_row^2
      const double f0 = std::fmax(1e-5, g0.friction), ft = std::fmax(1e-5, g0.friction_torsion), fr = std::fmax(1e-5, g0.friction_roll);
      C.slot_frt[s] = (float)ft; C.slot_frr[s] = (float)fr;
      C.slot_dt_tor[s] = (float)(m.impratio * ft * ft / (f0 * f0)); C.slot_dt_roll[s] = (float)(m.impratio * fr * fr / (f0 * f0));
    }
    rows += nv;
  }
  C.nvert_rows = rows;
  out->vert.assign((size_t)(rows > 0 ? rows : 1) * 16, 0.f);
  for (int s = 0; s < nslot; s++)
    for (int l = 0; l < 4; l++) {
      if (per_leg[l][s] < 0) continue;
      const OdgGeom& g = m.geom[per_leg[l][s]];
      for (int k = 0; k < C.slot_nvert[s]; k++) {
        int src = g.vert_count > 0 ? g.vert_start + (k < g.vert_count ? k : g.vert_count - 1) : -1;
        float* dst = &out->vert[((size_t)(C.slot_vstart[s] + k) * 4 + l) * 4];
        for (int c = 0; c < 3; c++) dst[c] = src >= 0 ? (float)m.vert[src][c] : 0.f;
      }
    }
  // support-vertex candidate lists per (slot, cell of the floor direction in the link frame, leg)
  {
    // widening of a cell in its normalised coordinates (dominant component = 1) that covers the three tilted
    // directions: a unit floor direction m has dominant component >= 1/sqrt(3); a tilted one is cos(t) m + sin(t) e
    const double a = std::sin(std::fabs(m.multicontact_tilt)), cm = std::cos(m.multicontact_tilt) / std::sqrt(3.0);
    const bool prune = cm - a > 0.2;
    const double w_lo = prune ? 1.05 * a / (cm - a) + 1e-3 : 0.0, w_hi = prune ? 1.05 * ((cm + a) / (cm - a) - 1.0) + 1e-3 : 0.0;
    std::vector<int> table((size_t)(nslot > 0 ? nslot : 1) * kSupportCells * 4, 0);
    std::vector<unsigned char> idx;
    for (int s = 0; s < nslot; s++) for (int l = 0; l < 4; l++) {
      static const OdgGeom kEmpty = OdgGeom();
      const OdgGeom& g = per_leg[l][s] >= 0 ? m.geom[per_leg[l][s]] : kEmpty;
      if (g.vert_count > 255) return "hull too large for the support-vertex candidate lists";
      double ext = 0.0;
      for (int k = 0; k < g.vert_count; k++) for (int c = 0; c < 3; c++) ext = std::fmax(ext, std::fabs(m.vert[g.vert_start + k][c]));
      const double tol = 1e-7 + 1e-5 * ext;
      for (int cell = 0; cell < kSupportCells; cell++) {
        const int axis = cell >> 3, o = cell & 7;
        const int sigma[3] = { (o & 1) ? -1 : 1, (o & 2) ? -1 : 1, (o & 4) ? -1 : 1 };
        const size_t start = idx.size();
        for (int k = 0; k < g.vert_count; k++)
          if (!prune || hull_vertex_is_candidate(&m.vert[g.vert_start], g.vert_count, k, axis, sigma, w_lo, w_hi, tol))
            idx.push_back((unsigned char)k);
        if (start > 0xFFFF) return "support-vertex candidate lists too long";
        table[((size_t)s * kSupportCells + cell) * 4 + l] = (int)start | ((int)(idx.size() - start) << 16);
      }
    }
    while (out->gc.size() % 4) out->gc.push_back(0.f);
    C.oct_off = (int)out->gc.size();
    for (int v : table) { float f; std::memcpy(&f, &v, 4); out->gc.push_back(f); }
    C.idx_off = (int)out->gc.size();
    while (idx.size() % 16) idx.push_back(0);
    for (size_t i = 0; i < idx.size(); i += 4) { float f; std::memcpy(&f, &idx[i], 4); out->gc.push_back(f); }
    while (out->gc.size() % 4) out->gc.push_back(0.f);
  }
  // three extra support directions tilted off -normal, 120 degrees apart (frame t1=+y, t2=-x)
  C.n_tilt = m.multicontact_tilt > 0 ? 3 : 0;
  for (int i = 0; i < 3; i++) {
    double ang = 2.0 * 3.14159265358979323846 * i / 3.0, t = m.multicontact_tilt;
    C.tilt_dir[i][0] = (float)(-std::sin(t) * std::sin(ang));
    C.tilt_dir[i][1] = (float)(std::sin(t) * std::cos(ang));
    C.tilt_dir[i][2] = (float)(-std::cos(t));
  }
  C.frame_skip = cfg.frame_skip; C.max_steps = cfg.max_episode_steps; C.auto_reset = cfg.auto_reset;
  C.solver_iters = cfg.solver_iterations; C.ls_iters = cfg.ls_iterations; C.scale_actions = cfg.scale_actions;
  C.obs_layout = cfg.obs_layout ? 1 : 0;
  if (cfg.task != ODG_TASK_WALK && cfg.task != ODG_TASK_JUMP) return "unknown task";
  if (cfg.task == ODG_TASK_JUMP && m.njl != 3) return "the jump task is defined on the 12-actuator (3 joints per leg) model";
  C.task = cfg.task;
  C.obs_dim = cfg.task == ODG_TASK_JUMP ? 9 + m.nu : (C.obs_layout ? 12 : 9) + 3 * m.nu;
  C.first_env_id = cfg.first_env_id; C.tol = cfg.solver_tolerance; C.ls_tol = cfg.ls_tolerance; C.noise = cfg.reset_noise_scale;
  C.seed_lo = (uint32_t)seed; C.seed_hi = (uint32_t)(seed >> 32);
  if (cfg.frame_skip < 1 || cfg.solver_iterations < 1) return "bad config";
  // one pass evaluates only {0.25, 0.5, 1, 2}: a zero of phi' below 0.25 (a stiff row switching on next to the iterate)
  // then gets the chord across the kink on every iteration and the solve reaches the iteration cap unconverged. Two
  // passes leave the ladder no pass to refine its bracket in, and states of both models still stall at the cap far from
  // the optimum. In the GPU-sized state sets of tests/test_solver_optimality.py (same indices on the B200 and in the
  // host emulator): OpenDOG rollout state 1729 at ls_tolerance 0.01 (gap 7e9 x its float32 floor), OpenDOG rest state
  // 2457 at 0.1 (1.5e9 x), Go1 rollout state 447 at 0.5 (3.9e9 x)
  if (cfg.ls_iterations < 3) return "ls_iterations must be >= 3 (fewer passes cannot resolve steps below 0.25)";
  return "";
}

inline void default_config(OdgEnvConfig* c) {
  c->task = ODG_TASK_WALK; c->frame_skip = 10; c->max_episode_steps = 750; c->auto_reset = 1;
  c->solver_iterations = 30; c->ls_iterations = 4; c->solver_tolerance = 1e-4f; c->ls_tolerance = 0.1f; c->reset_noise_scale = 0.02f;
  c->scale_actions = 1; c->launch_lanes = 0; c->first_env_id = 0; c->obs_layout = 0; c->launch_block = 0; c->launch_lockstep = -1; c->launch_fat = -1;
}

}  // namespace odg
