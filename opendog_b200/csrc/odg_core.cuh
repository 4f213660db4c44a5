// odg_core.cuh — the fused environment step, written once for a 4-lane cooperative group.
//
// One environment = 4 lanes (one per leg; 8 environments per warp). Every lane carries the trunk
// state redundantly and its own leg's joints; quantities that couple legs (composite inertia of the
// trunk, trunk wrench, the 6x6 Schur complement of the Newton system) are combined with xor-butterfly
// shuffles inside the 4-lane group, which leave bit-identical values in all 4 lanes.
//
// What it replaces (reference, per environment, on the CPU):
//   mujoco.mj_step x frame_skip           WalkEnvironment.py:58, sim2real/train.py:281-284   [3P wheel]
//   _get_obs / rewards / is_healthy       WalkEnvironment.py:59-136, reward_calc.py:117-390
//   ScaleActionWrapper.action             ScaleActionEnvironment.py:21-23
//   SubprocVecEnv worker auto-reset       train/train.py:81-86                                 [3P SB3]
//
// Formulation (differs structurally from oracle/odg_oracle.c on purpose):
//   * positions are kept relative to the trunk origin O (fp32 stays accurate far from the world origin);
//   * the trunk's rotational DoFs are handled in the WORLD frame internally (alpha_w = R0 * qacc_rot);
//   * M and the Newton Hessian H = M + J^T D J are block-arrow (6x6 trunk block + one NJLxNJL block per
//     leg + couplings), so each lane eliminates its own leg block and the group reduces one 6x6 Schur
//     complement (21+6 floats) per Newton iteration;
//   * contact Jacobians are never stored: J*x is evaluated as the acceleration of the contact point.
//
// The same source compiles for the host (ODG_HOST_EMU) where 4 std::threads emulate the lanes; that
// build exists only for tests/ (numerics debugging without a GPU) and is never shipped or loaded by
// the package.
#pragma once

#include <stdint.h>
#include <math.h>
#include <string.h>

#ifdef ODG_HOST_EMU
#define ODG_DEV inline
#define ODG_NOINLINE inline
#define ODG_RESTRICT
struct float4 { float x, y, z, w; };
float odg_emu_shfl_xor(float v, int m);     // provided by the emulator
double odg_emu_shfl_xor_d(double v, int m);
static inline float odg_rsqrt(float x) { return 1.0f / sqrtf(x); }
static inline float odg_fmul_rn(float a, float b) { volatile float r = a * b; return r; }
static inline float odg_fadd_rn(float a, float b) { volatile float r = a + b; return r; }
static inline float odg_fsub_rn(float a, float b) { volatile float r = a - b; return r; }
static inline float odg_fdiv_rn(float a, float b) { volatile float r = a / b; return r; }
static inline float odg_fdiv_fast(float a, float b) { return a / b; }
static inline float odg_fma_rn(float a, float b, float c) { return fmaf(a, b, c); }
#ifdef ODG_EMU_STATS
// solver statistics of the host emulator (tools/emu_solver_stats.py): one record per Newton iteration of lane 0
void odg_emu_stat(int it, float rel_step, float alpha, int ls_passes, int nc_leg, float d10);
#endif
#define ODG_UNROLL
#define ODG_NO_UNROLL
#else
#define ODG_DEV __device__ __forceinline__
#define ODG_NOINLINE static __device__ __noinline__
#define ODG_RESTRICT __restrict__
#define odg_fmul_rn __fmul_rn
#define odg_fadd_rn __fadd_rn
#define odg_fsub_rn __fsub_rn
#define odg_fdiv_rn __fdiv_rn
#define odg_fma_rn __fmaf_rn
#define odg_fdiv_fast __fdividef               // 2-ulp quotient without the IEEE slow-path call (step lengths, stiffnesses)
// one MUFU.RSQ: every argument in this file is clamped to a normal number first, so the denormal pre/post-scaling that
// rsqrtf() carries without -ftz (a compare and two predicated multiplies per call) is dead weight in the hot loops
__device__ __forceinline__ float odg_rsqrt(float x) { float r; asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
#define ODG_UNROLL _Pragma("unroll")
#define ODG_NO_UNROLL _Pragma("unroll 1")
#endif

#ifndef ODG_LS_WIDTH
#define ODG_LS_WIDTH 4
#endif

namespace odg {

constexpr int kMaxJL = 3;
constexpr int kMaxSlot = 12;         // collision geoms per lane (a leg's own, plus its share of the trunk's)
constexpr int kMaxConLeg = 12;       // contacts per lane (<= 4 per geom)
constexpr int kMaxNU = 12;
constexpr int kMaxNQ = 7 + 4 * kMaxJL;

// ---- per-joint, per-leg constants staged in shared memory as s_lc[(j*LC_COUNT + f)*4 + leg]
enum LegConstField {
  LC_BP0, LC_BP1, LC_BP2,                       // body_pos
  LC_BR0, LC_BR1, LC_BR2, LC_BR3, LC_BR4, LC_BR5, LC_BR6, LC_BR7, LC_BR8,   // body_quat as matrix
  LC_JP0, LC_JP1, LC_JP2,                       // jnt_pos
  LC_JA0, LC_JA1, LC_JA2,                       // jnt_axis
  LC_MASS, LC_IP0, LC_IP1, LC_IP2,
  LC_IXX, LC_IXY, LC_IXZ, LC_IYY, LC_IYZ, LC_IZZ,
  LC_LO, LC_HI, LC_LIMITED,
  LC_ARM, LC_FL, LC_RFL, LC_DFL, LC_DAMP, LC_INVW,
  LC_KP, LC_KV, LC_CLO, LC_CHI, LC_FLO, LC_FHI, LC_HASACT, LC_CLIM, LC_FLIM, LC_UIDX,
  LC_SLO, LC_SHI,                               // ScaleActionWrapper table (float32 values)
  LC_HOMEQ,                                     // key_qpos of the joint
  LC_COUNT
};
// per-slot, per-leg constants: s_gc[(slot*GC_COUNT + f)*4 + leg]
enum GeomConstField { GC_INVW, GC_CX, GC_CY, GC_CZ, GC_BX, GC_BY, GC_BZ, GC_BR, GC_HX, GC_HY, GC_HZ,
                      // primitives (capsule / cylinder / box; only the 3-joint-leg instantiation reads them): geom type of
                      // THIS lane's geom in the slot (0 = none: front legs carry one hip cylinder less than rear legs, and
                      // the trunk's colliders are dealt out over the four lanes), geom frame in the link frame, sizes
                      GC_TYPE, GC_R0, GC_R1, GC_R2, GC_R3, GC_R4, GC_R5, GC_R6, GC_R7, GC_R8, GC_S0, GC_S1, GC_S2,
                      GC_COUNT };
// geom types as the kernel numbers them (model types + 1 where the lane-level table is used; 0 = empty slot)
enum { PRIM_NONE = 0, PRIM_SPHERE = 2, PRIM_CAPSULE = 3, PRIM_CYLINDER = 4, PRIM_BOX = 5 };

struct DevConst {
  int nleg, njl, nq, nv, nu, nslot, nvert_rows;
  int oct_off, idx_off;                         // s_gc offsets (floats) of the support-vertex candidate table / byte lists
  int body_rot_identity;
  int lockstep;                                 // block-lockstep Newton iterations (batches of more than one wave)
  int any_damping;                              // some joint has damping > 0: mj_Euler integrates it implicitly
  float h, gx, gy, gz, impratio;
  // trunk
  float base_mass, base_ip[3], base_I[6];
  float base_arm_t[3], base_arm_r;
  float base_fl[6], base_Rfl[6], base_Dfl[6];
  float B_fl;                                   // friction-loss rows: aref = -B_fl * vel
  float K_lim, B_lim, lim_imp[5];
  // collision slots (identical layout on every leg)
  int slot_link[kMaxSlot], slot_type[kMaxSlot], slot_nvert[kMaxSlot], slot_vstart[kMaxSlot];
  int slot_condim[kMaxSlot], slot_isfoot[kMaxSlot];
  float slot_margin[kMaxSlot], slot_K[kMaxSlot], slot_B[kMaxSlot], slot_imp[kMaxSlot][5];
  float slot_fri[kMaxSlot], slot_mu[kMaxSlot], slot_radius[kMaxSlot];
  float slot_dmk[kMaxSlot];                     // 1 / (mu^2 (1 + mu^2)): Dm = Dn * slot_dmk (cone surface stiffness)
  // condim 6 (Go1 feet, go1.xml:61-64): torsional / rolling friction coefficients and the stiffness ratios of their rows,
  // D_row = D_normal * ratio with ratio = impratio * mu_slide^2 / mu_row^2 (mj_makeImpedance); all 0 for condim < 6
  float slot_frt[kMaxSlot], slot_frr[kMaxSlot], slot_dt_tor[kMaxSlot], slot_dt_roll[kMaxSlot];
  int per_lane_geoms;                           // slots differ between lanes (type / presence from the GC_TYPE table)
  float tilt_dir[3][3];                         // extra support directions (world)
  int n_tilt;
  // env
  int frame_skip, max_steps, auto_reset, solver_iters, ls_iters, scale_actions, first_env_id;
  int obs_layout;                               // OdgEnvConfig::obs_layout
  int task;                                     // OdgEnvConfig::task (0 walk, 1 jump: 3-joint-leg kernel only)
  int obs_dim;                                  // walk: (obs_layout ? 12 : 9) + 3 nu; jump: 9 + nu
  float tol, ls_tol, noise;
  float key_qpos[kMaxNQ], key_ctrl[kMaxNU];
  float obs_joint_offset;                       // key_ctrl[0,7:] broadcast quirk (WalkEnvironment.py:116)
  uint32_t seed_lo, seed_hi;
};

struct SimPtrs {            // SoA state in HBM: x[i*N + env]
  int N;                    // array stride = environments rounded up to a whole number of blocks (padding envs are
                            // stepped like real ones, so every warp of a block reaches every block barrier)
  int n;                    // real environments: caller-owned buffers ([n][dim]) are touched only for env < n
  float* qpos; float* qvel; float* warm;        // [nq][N], [nv][N], [nv][N]
  float* last_action;                            // [nu][N]
  float* desvel;                                 // [3][N]
  int* step; int* gait_idx; int* gait_cnt; unsigned* episode;   // [N]
  unsigned char* fresh;                          // [N] last_action is the float64 zeros of reset_model
  int* work;                                     // [N] solver work of the last env-step (Newton iterations + line-search passes)
};

// MPPI mode of the step kernel (include/odg_mppi.h: odg_mppi_rollout): T > 0 turns one launch into a whole rollout —
// every environment walks T env-steps, drawing its own action row before each one and accumulating its cost.
// Environments form groups of S samples (odg_mppi_rollout_groups): sample g * S + s reads the nominal rows of group g and
// draws the noise of sample s under the key seed + g.
struct MppiArgs {
  int T;                          // horizon; 0 = ordinary step
  int S;                          // samples per group (MPPI mode only)
  int mean_stride;                // floats between the nominal sequences of consecutive groups
  float sigma, term_cost;
  uint32_t seed_lo, seed_hi, iteration;
  const uint32_t* iteration_dev;  // nullable: device-side plan counter (CUDA-graph replays draw fresh noise)
  const float* mean;              // [G][T][A]
  float* actions;                 // [T][n][A]
  float* cost;                    // [n]
};

struct StepArgs {
  const float* action;      // [N][nu]
  float* obs;               // [N][obs_dim]
  float* reward;            // [N]
  unsigned char* terminated; unsigned char* truncated;
  int mode;                 // 0 = step, 1 = evaluate (one forward pass, no integration, no auto-reset)
  int want_info;
  // info (nullable)
  float* x_position; float* y_position; float* distance; float* paw_forces; float* patterns_matches;
  float* lin_vel_reward; float* reward_ctrl; float* terminal_obs; unsigned char* paws_in_ground;
  int* gait_reward; float* qacc; int* ncon; float* fn_sum; int* solver_iters; int* ls_evals;
  float* reward_raw;        // rewards - costs before the max(0, .) of WalkEnvironment.py:84
  float* cfrc_ext;          // [N][1 + 4*njl][6] data.cfrc_ext of the robot's bodies (3-joint-leg kernel)
  float* task_terms;        // [N][10] weighted reward / cost terms of the jump task (compute_rewards' reward_info)
};

// ---------------------------------------------------------------------------------------------
struct V3 { float x, y, z; };
ODG_DEV V3 mk3(float x, float y, float z) { V3 r; r.x = x; r.y = y; r.z = z; return r; }
ODG_DEV V3 operator+(V3 a, V3 b) { return mk3(a.x + b.x, a.y + b.y, a.z + b.z); }
ODG_DEV V3 operator-(V3 a, V3 b) { return mk3(a.x - b.x, a.y - b.y, a.z - b.z); }
ODG_DEV V3 operator*(float s, V3 a) { return mk3(s * a.x, s * a.y, s * a.z); }
ODG_DEV V3 operator-(V3 a) { return mk3(-a.x, -a.y, -a.z); }
// (sums of products in one fixed fused order — see cross(): the order must not depend on the code around the call)
ODG_DEV float dot3(float ax, float ay, float az, float bx, float by, float bz) {
  return odg_fma_rn(az, bz, odg_fma_rn(ay, by, odg_fmul_rn(ax, bx)));
}
ODG_DEV float dot(V3 a, V3 b) { return dot3(a.x, a.y, a.z, b.x, b.y, b.z); }
// (explicit fused form: `a.y * b.z - a.z * b.y` may be contracted either way round, and the two instantiations of the step
//  kernel — one stores a contact's Jacobian columns, one recomputes them — must produce the same bits at every site)
ODG_DEV float cross1(float a, float b, float c, float d) { return odg_fma_rn(a, b, -odg_fmul_rn(c, d)); }      // a*b - c*d
ODG_DEV V3 cross(V3 a, V3 b) { return mk3(cross1(a.y, b.z, a.z, b.y), cross1(a.z, b.x, a.x, b.z), cross1(a.x, b.y, a.y, b.x)); }
// accumulating forms, one fused multiply-add per product: acc + a.b and acc + a x b
ODG_DEV float dot_acc(float acc, V3 a, V3 b) { return odg_fma_rn(a.z, b.z, odg_fma_rn(a.y, b.y, odg_fma_rn(a.x, b.x, acc))); }
ODG_DEV float cross1_acc(float acc, float a, float b, float c, float d) { return odg_fma_rn(a, b, odg_fma_rn(-c, d, acc)); }
ODG_DEV V3 cross_acc(V3 acc, V3 a, V3 b) {
  return mk3(cross1_acc(acc.x, a.y, b.z, a.z, b.y), cross1_acc(acc.y, a.z, b.x, a.x, b.z), cross1_acc(acc.z, a.x, b.y, a.y, b.x));
}
ODG_DEV float comp(V3 a, int i) { return i == 0 ? a.x : (i == 1 ? a.y : a.z); }

// 16-byte records for per-contact data in local memory: one 128-bit load / store instead of three or four 32-bit ones
ODG_DEV float4 mk4(V3 v, float w) { float4 r; r.x = v.x; r.y = v.y; r.z = v.z; r.w = w; return r; }
ODG_DEV V3 xyz(float4 q) { return mk3(q.x, q.y, q.z); }
#ifdef ODG_HOST_EMU
static inline float odg_int_bits(int i) { float f; memcpy(&f, &i, 4); return f; }
static inline int odg_float_bits(float f) { int i; memcpy(&i, &f, 4); return i; }
#else
#define odg_int_bits __int_as_float
#define odg_float_bits __float_as_int
#endif

struct M3 { float m[9]; };   // row-major
ODG_DEV V3 mul(const M3& R, V3 v) {
  return mk3(dot3(R.m[0], R.m[1], R.m[2], v.x, v.y, v.z), dot3(R.m[3], R.m[4], R.m[5], v.x, v.y, v.z),
             dot3(R.m[6], R.m[7], R.m[8], v.x, v.y, v.z));
}
ODG_DEV V3 tmul(const M3& R, V3 v) {
  return mk3(dot3(R.m[0], R.m[3], R.m[6], v.x, v.y, v.z), dot3(R.m[1], R.m[4], R.m[7], v.x, v.y, v.z),
             dot3(R.m[2], R.m[5], R.m[8], v.x, v.y, v.z));
}
ODG_DEV M3 mul(const M3& A, const M3& B) {
  M3 C;
  ODG_UNROLL for (int i = 0; i < 3; i++)
    ODG_UNROLL for (int j = 0; j < 3; j++)
      C.m[i * 3 + j] = A.m[i * 3] * B.m[j] + A.m[i * 3 + 1] * B.m[3 + j] + A.m[i * 3 + 2] * B.m[6 + j];
  return C;
}
ODG_DEV V3 col(const M3& R, int k) { return mk3(R.m[k], R.m[3 + k], R.m[6 + k]); }

// symmetric 3x3: xx xy xz yy yz zz
struct S3 { float xx, xy, xz, yy, yz, zz; };
ODG_DEV V3 mul(const S3& A, V3 v) {
  return mk3(dot3(A.xx, A.xy, A.xz, v.x, v.y, v.z), dot3(A.xy, A.yy, A.yz, v.x, v.y, v.z),
             dot3(A.xz, A.yz, A.zz, v.x, v.y, v.z));
}
ODG_DEV S3 zero_s3() { S3 s; s.xx = s.xy = s.xz = s.yy = s.yz = s.zz = 0.f; return s; }
ODG_DEV void add_outer(S3& A, V3 a, V3 b) {   // A += sym part of a b^T + b a^T scaled 0.5 ... used only with a==b scaled
  A.xx += a.x * b.x; A.xy += a.x * b.y; A.xz += a.x * b.z; A.yy += a.y * b.y; A.yz += a.y * b.z; A.zz += a.z * b.z;
}
// R * A * R^T for symmetric A
ODG_DEV S3 rotate_sym(const M3& R, const S3& A) {
  V3 c0 = mul(A, mk3(R.m[0], R.m[1], R.m[2]));   // A * row0(R)^T
  V3 c1 = mul(A, mk3(R.m[3], R.m[4], R.m[5]));
  V3 c2 = mul(A, mk3(R.m[6], R.m[7], R.m[8]));
  V3 r0 = mk3(R.m[0], R.m[1], R.m[2]), r1 = mk3(R.m[3], R.m[4], R.m[5]), r2 = mk3(R.m[6], R.m[7], R.m[8]);
  S3 o;
  o.xx = dot(r0, c0); o.xy = dot(r0, c1); o.xz = dot(r0, c2);
  o.yy = dot(r1, c1); o.yz = dot(r1, c2); o.zz = dot(r2, c2);
  return o;
}

// spatial inertia about O, world aligned
struct SpI { float m; V3 h; S3 I; };
ODG_DEV SpI spi_make(float mass, V3 c, const S3& Iw) {
  SpI s; s.m = mass; s.h = mass * c;
  float cc = dot(c, c);
  s.I.xx = Iw.xx + mass * (cc - c.x * c.x); s.I.yy = Iw.yy + mass * (cc - c.y * c.y); s.I.zz = Iw.zz + mass * (cc - c.z * c.z);
  s.I.xy = Iw.xy - mass * c.x * c.y; s.I.xz = Iw.xz - mass * c.x * c.z; s.I.yz = Iw.yz - mass * c.y * c.z;
  return s;
}
ODG_DEV SpI spi_add(const SpI& a, const SpI& b) {
  SpI s; s.m = a.m + b.m; s.h = a.h + b.h;
  s.I.xx = a.I.xx + b.I.xx; s.I.xy = a.I.xy + b.I.xy; s.I.xz = a.I.xz + b.I.xz;
  s.I.yy = a.I.yy + b.I.yy; s.I.yz = a.I.yz + b.I.yz; s.I.zz = a.I.zz + b.I.zz;
  return s;
}

// ---- 4-lane group collectives
#ifdef ODG_HOST_EMU
ODG_DEV float grp_xor(float v, int m, unsigned) { return odg_emu_shfl_xor(v, m); }
#else
ODG_DEV float grp_xor(float v, int m, unsigned gmask) { return __shfl_xor_sync(gmask, v, m); }
#endif
#ifdef ODG_HOST_EMU
ODG_DEV double grp_xor_d(double v, int m, unsigned) { return odg_emu_shfl_xor_d(v, m); }
#else
ODG_DEV double grp_xor_d(double v, int m, unsigned gmask) { return __shfl_xor_sync(gmask, v, m); }
#endif
#ifdef ODG_HOST_EMU
ODG_DEV void grp_sync(unsigned) { (void)odg_emu_shfl_xor(0.f, 1); }
#else
ODG_DEV void grp_sync(unsigned gmask) { __syncwarp(gmask); }
#endif
ODG_DEV float grp_sum(float v, unsigned gm) { v += grp_xor(v, 1, gm); v += grp_xor(v, 2, gm); return v; }
ODG_DEV float grp_sum21(float v, unsigned gm) { v += grp_xor(v, 2, gm); v += grp_xor(v, 1, gm); return v; }
// Sum of 28 values over the 4 lanes of a group through shared memory, in two stages: every lane stores its 28 values as
// one row (stride kRedStride floats), then lane l sums columns [8l, 8l + 8) of the four rows — in lane order 0,1,2,3, so
// the result does not depend on who computes it — back into row 0 (nobody else reads those columns), which all four lanes
// then read. The rows must not grow: at 65536 envs four blocks per SM sit just under a shared-memory carve-out step, and
// the next step takes 32 KB of L1 away from the local-memory traffic (-25 %). 7 + 2 STS.128,
// 8 + 7 LDS.128 and 24 FADD per lane instead of 28 LDS.128 + 84 FADD when every lane sums everything (or 56 shuffles, each
// of which costs a WARPSYNC / collective region under a partial mask): the Newton body is instruction-fetch bound.
constexpr int kRedVals = 28, kRedStride = 36, kRedGroup = 4 * kRedStride;     // 4 rows per group
constexpr int kSupportCells = 24;     // direction cells of the support-vertex candidate lists: dominant axis (3) x signs (8)
ODG_DEV void grp_sum28(float (&v)[kRedVals], float* ODG_RESTRICT s_red, int leg, unsigned gm) {
  grp_sync(gm);                                    // earlier readers of the rows are done
  float4* mine = reinterpret_cast<float4*>(s_red + leg * kRedStride);
  ODG_UNROLL for (int k = 0; k < kRedVals / 4; k++) { float4 t; t.x = v[4 * k]; t.y = v[4 * k + 1]; t.z = v[4 * k + 2]; t.w = v[4 * k + 3]; mine[k] = t; }
  grp_sync(gm);
  float4* res = reinterpret_cast<float4*>(s_red);
  ODG_UNROLL for (int h = 0; h < 2; h++) {         // (columns 28..31 are padding: whatever they hold is summed and never read)
    const int k = 2 * leg + h;
    const float4 a = reinterpret_cast<const float4*>(s_red)[k];
    const float4 b = reinterpret_cast<const float4*>(s_red + kRedStride)[k];
    const float4 c = reinterpret_cast<const float4*>(s_red + 2 * kRedStride)[k];
    const float4 d = reinterpret_cast<const float4*>(s_red + 3 * kRedStride)[k];
    float4 t;
    t.x = ((a.x + b.x) + c.x) + d.x; t.y = ((a.y + b.y) + c.y) + d.y; t.z = ((a.z + b.z) + c.z) + d.z; t.w = ((a.w + b.w) + c.w) + d.w;
    res[k] = t;
  }
  grp_sync(gm);
  ODG_UNROLL for (int k = 0; k < kRedVals / 4; k++) {
    const float4 t = res[k];
    v[4 * k] = t.x; v[4 * k + 1] = t.y; v[4 * k + 2] = t.z; v[4 * k + 3] = t.w;
  }
}
// One sum and two maxima over the 4 lanes of a group in a single shared-memory round (the rows of grp_sum28): one
// STS.128 + four LDS.128 instead of six partial-mask shuffles.
ODG_DEV void grp_sum_max2(float& sum, float& m0, float& m1, float* ODG_RESTRICT s_red, int leg, unsigned gm) {
  grp_sync(gm);                                    // earlier readers of the rows are done
  float4 t; t.x = sum; t.y = m0; t.z = m1; t.w = 0.f;
  *reinterpret_cast<float4*>(s_red + leg * kRedStride) = t;
  grp_sync(gm);
  const float4 a = *reinterpret_cast<const float4*>(s_red), b = *reinterpret_cast<const float4*>(s_red + kRedStride);
  const float4 c = *reinterpret_cast<const float4*>(s_red + 2 * kRedStride), d = *reinterpret_cast<const float4*>(s_red + 3 * kRedStride);
  sum = ((a.x + b.x) + c.x) + d.x;
  m0 = fmaxf(fmaxf(a.y, b.y), fmaxf(c.y, d.y));
  m1 = fmaxf(fmaxf(a.z, b.z), fmaxf(c.z, d.z));
}
ODG_DEV float grp_max(float v, unsigned gm) { v = fmaxf(v, grp_xor(v, 1, gm)); v = fmaxf(v, grp_xor(v, 2, gm)); return v; }
ODG_DEV V3 grp_sum(V3 v, unsigned gm) { return mk3(grp_sum(v.x, gm), grp_sum(v.y, gm), grp_sum(v.z, gm)); }
ODG_DEV float grp_bcast(float v, int src_leg, int leg, unsigned gm) {   // value of lane `src_leg` to all 4
  float a = grp_xor(v, 1, gm); float m1 = ((leg ^ src_leg) & 1) ? a : v;      // now correct within pair parity
  float b = grp_xor(m1, 2, gm); return ((leg ^ src_leg) & 2) ? b : m1;
}

// ---- Philox4x32-10 (same stream definition as oracle/odg_oracle.c)
ODG_DEV void philox4x32(uint32_t k0, uint32_t k1, uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t out[4]) {
  ODG_UNROLL for (int r = 0; r < 10; r++) {
    uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
    uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n1 = (uint32_t)p1;
    uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1, n3 = (uint32_t)p0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3; k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}
ODG_DEV float u01(uint32_t x) { return (float)(x >> 8) * 5.9604644775390625e-08f; }
constexpr uint32_t kStreamReset = 0x52534554u, kStreamDesvel = 0x44564c00u;

// MPPI action row of one sample: action[a] = clamp(mean[a] + sigma * eps, -1, 1), eps from Philox4x32-10 keyed by
// (seed, sample, iteration, t, block) turned into Box-Muller pairs. One definition for the stand-alone sampler kernel
// and for the rollout mode of the step kernel.
constexpr uint32_t kStreamMppi = 0x4d505049u;
#ifndef ODG_HOST_EMU
ODG_DEV void mppi_sample_row(const float* ODG_RESTRICT mean, float sigma, int n, int A, uint32_t seed_lo, uint32_t seed_hi,
                             uint32_t iteration, uint32_t t, float* ODG_RESTRICT action) {
  for (int blk = 0; blk * 4 < A; blk++) {
    uint32_t r[4];
    philox4x32(seed_lo, seed_hi, (uint32_t)n, iteration, (t << 8) | (uint32_t)blk, kStreamMppi, r);
    for (int pr = 0; pr < 2; pr++) {
      const float u1 = ((float)(r[2 * pr] >> 8) + 1.0f) * 5.9604644775390625e-08f;
      const float u2 = u01(r[2 * pr + 1]);
      const float rad = sqrtf(-2.0f * logf(u1));
      float sn, cs; sincosf(6.283185307179586f * u2, &sn, &cs);
      const float e[2] = { rad * cs, rad * sn };
      for (int q = 0; q < 2; q++) {
        const int a = blk * 4 + pr * 2 + q;
        if (a < A) action[(size_t)n * A + a] = fminf(1.f, fmaxf(-1.f, mean[a] + sigma * e[q]));
      }
    }
  }
}
#endif

// ---- solimp impedance (mj_makeImpedance::getimpedance); imp5 = d0,dmax,width,mid,power (pre-clamped on host)
ODG_NOINLINE float impedance_pow(float x, float mid, float power) {      // generic power (reference models use 2)
  return x <= mid ? powf(x, power) / powf(mid, power - 1.f) : 1.f - powf(1.f - x, power) / powf(1.f - mid, power - 1.f);
}
ODG_DEV float impedance(const float* imp5, float pos_minus_margin) {
  const float d0 = imp5[0], d1 = imp5[1], width = imp5[2], mid = imp5[3], power = imp5[4];
  const bool flat = d0 == d1 || width <= 1e-15f;
  // x clamped to [0, 1]: the sigmoid is 0 at 0 and 1 at 1, so the d0 / d1 plateaus need no branches
  const float x = fminf(fabsf(odg_fdiv_fast(pos_minus_margin, flat ? 1.f : width)), 1.f);
  float y;
  if (power == 2.f) {                              // (uniform: the reference models use the default power 2)
    const bool low = x <= mid;
    const float t = low ? x : 1.f - x;
    const float q = odg_fdiv_fast(t * t, low ? mid : 1.f - mid);
    y = low ? q : 1.f - q;
  } else if (power == 1.f) {
    y = x;
  } else {
    y = (x <= 0.f) ? 0.f : ((x >= 1.f) ? 1.f : impedance_pow(x, mid, power));
  }
  return flat ? 0.5f * (d0 + d1) : d0 + y * (d1 - d0);
}

// friction-loss (Huber) row: z -> ds/dz, d2s/dz2   (D * R == 1, so clamping D*z at +-f is the linear zone)
ODG_DEV void fl_eval(float z, float f, float R, float D, float& g, float& hh) {
  g = fminf(fmaxf(D * z, -f), f);
  hh = fabsf(z) < R * f ? D : 0.f;
}

// elliptic-cone contact block. z = (zx, zy, zn) in world axes (normal = +z). Returns the zone.
ODG_DEV int cone_eval(V3 z, float Dn, float Dt, float mu, float fri, float dmk, int condim, V3& g, S3& H) {
  // Branch-free: both the sticking-zone and the cone-surface blocks are formed and one is selected (top zone and
  // D = 0 rows select zeros). Branches here cost more than the arithmetic they skip: every lane of the warp walks the
  // contact loop anyway, and a branch ends the basic block the scheduler can interleave over.
  // A frictionless (condim 1) row is the same cone with fri = Dt = 0: T = 0, zone = (N >= 0 ? top : bottom).
  if (condim == 1) { fri = 0.f; Dt = 0.f; }
  const float U1 = z.x * fri, U2 = z.y * fri, N = z.z * mu;
  // (sums of two products are written with explicit fused operations: "a*b + c*d" can be contracted either way round,
  //  and the two instantiations of the step kernel inline this function into differently shaped code)
  const float T2 = odg_fma_rn(U1, U1, odg_fmul_rn(U2, U2));
  const float iT = odg_rsqrt(fmaxf(T2, 1e-20f));
  const float T = T2 * iT;
  const bool top = N >= mu * T;                      // separating (T == 0: N >= 0)
  const bool bot = !top && (mu * N + T <= 0.f);      // sticking
  const bool mid = !top && !bot;                     // on the cone surface, sliding
  // cost = Dm/2 * e^2 with e = N - mu*T < 0 on the cone surface. With u = U/T, w = de/dz = (-mu*u*fri, mu) and
  // v = (u_perp*fri, 0):   g = Dm*e*w,   H = Dm * w w^T + kappa * v v^T,   kappa = Dm*mu*|e|/T >= 0.
  // Written as this sum of two rank-1 PSD terms the block cannot turn indefinite in fp32; the algebraically equal
  // closed form mu*N/T^3*U U^T + (mu^2 - mu*N/T) I cancels catastrophically when T is small.
  const float Dm = Dn * dmk;
  const float e = N - mu * T;
  const float ux = U1 * iT, uy = U2 * iT;
  const V3 w = mk3(-mu * ux * fri, -mu * uy * fri, mu);
  const float De = Dm * e;
  const float kap = -Dm * mu * e * iT;
  const float vx = -uy * fri, vy = ux * fri;
  g.x = mid ? De * w.x : (bot ? Dt * z.x : 0.f);
  g.y = mid ? De * w.y : (bot ? Dt * z.y : 0.f);
  g.z = mid ? De * w.z : (bot ? Dn * z.z : 0.f);
  const float Dwx = Dm * w.x, Dwy = Dm * w.y, kvx = kap * vx;
  H.xx = mid ? odg_fma_rn(Dwx, w.x, odg_fmul_rn(kvx, vx)) : (bot ? Dt : 0.f);
  H.yy = mid ? odg_fma_rn(Dwy, w.y, odg_fmul_rn(odg_fmul_rn(kap, vy), vy)) : (bot ? Dt : 0.f);
  H.zz = mid ? Dm * w.z * w.z : (bot ? Dn : 0.f);
  H.xy = mid ? odg_fma_rn(Dwx, w.y, odg_fmul_rn(kvx, vy)) : 0.f;
  H.xz = mid ? Dm * w.x * w.z : 0.f;
  H.yz = mid ? Dm * w.y * w.z : 0.f;
  return top ? 0 : (bot ? 1 : 2);
}

// Line search over one contact block, in two parts. `cone_line_prep` (once per Newton iteration, when the search
// direction is known) reduces the block to nine numbers: |U(alpha)|^2 = cA + 2 alpha cB + alpha^2 cC and U.V = cB + alpha cC
// as polynomials in the step length (U, V = scaled tangential parts of z0, dz), the normal part N0 + alpha Nd, the
// sticking-zone quadratic q1 + alpha q2, the cone-surface stiffness Dm and mu. `cone_line_eval` (every pass of the search)
// adds d/dalpha cost(z0 + al[k] dz) at W step lengths from those nine numbers alone — no per-slot constants, no vector
// arithmetic in the search's inner loop. Branch-free zone selection so the W evaluations interleave. The line search only
// positions the step and sets how many iterations the solve takes (tests/test_solver_optimality.py); with one or two
// passes it can stall at the iteration cap (odg_prep.h rejects ls_iterations < 3).
struct LineCoef { float N0, Nd, cA, cB, cC, q1, q2, Dm, mu; };
ODG_DEV LineCoef cone_line_prep(V3 z0, V3 dz, float Dn, float Dt, float mu, float fri, float dmk, int condim) {
  // a frictionless (condim 1) row is the same cone with no tangential part: fri = Dt = 0 gives T = 0, zone = (N >= 0 ?
  // top : bottom) and phi' = Dn * dz.z * min(z.z, 0) without a branch
  if (condim == 1) { fri = 0.f; Dt = 0.f; }
  // (explicitly rounded / fused operations: the lean instantiation of the step kernel inlines this into every pass of
  //  the search, the other one into the preparation loop, and both must produce the same bits)
  const float U0x = odg_fmul_rn(z0.x, fri), U0y = odg_fmul_rn(z0.y, fri), Vx = odg_fmul_rn(dz.x, fri), Vy = odg_fmul_rn(dz.y, fri);
  LineCoef k;
  k.N0 = odg_fmul_rn(z0.z, mu); k.Nd = odg_fmul_rn(dz.z, mu);
  k.Dm = odg_fmul_rn(Dn, dmk); k.mu = mu;
  const float zt = odg_fma_rn(z0.x, dz.x, odg_fmul_rn(z0.y, dz.y)), dt = odg_fma_rn(dz.x, dz.x, odg_fmul_rn(dz.y, dz.y));
  k.q1 = odg_fma_rn(Dt, zt, odg_fmul_rn(odg_fmul_rn(Dn, z0.z), dz.z));      // sticking zone: phi' = q1 + alpha*q2
  k.q2 = odg_fma_rn(Dt, dt, odg_fmul_rn(odg_fmul_rn(Dn, dz.z), dz.z));
  k.cA = odg_fma_rn(U0x, U0x, odg_fmul_rn(U0y, U0y)); k.cB = odg_fma_rn(U0x, Vx, odg_fmul_rn(U0y, Vy));
  k.cC = odg_fma_rn(Vx, Vx, odg_fmul_rn(Vy, Vy));
  return k;
}
template <int W>
ODG_DEV void cone_line_eval(const LineCoef& c, const float (&al)[W], float (&f)[W]) {
  ODG_UNROLL for (int k = 0; k < W; k++) {
    const float a = al[k];
    const float N = c.N0 + a * c.Nd;
    const float UV = c.cB + a * c.cC;
    const float T2 = fmaxf(c.cA + a * (c.cB + UV), 0.f);
    const float iT = odg_rsqrt(fmaxf(T2, 1e-20f));
    const float T = T2 * iT;
    const float Td = UV * iT;
    const float e = N - c.mu * T;                   // >= 0: separating (T == 0: N >= 0)
    const float fmid = c.Dm * e * (c.Nd - c.mu * Td);
    const float fbot = c.q1 + a * c.q2;
    const bool bot = c.mu * N + T <= 0.f;           // sticking
    f[k] += e >= 0.f ? 0.f : (bot ? fbot : fmid);
  }
}

// ---- condim-6 elliptic cone (sliding + torsional + rolling friction). z = (linear acceleration of the contact point,
// angular acceleration of the geom's body), both in world axes minus their references; the plane's frame is
// (n, t1, t2) = (+z, +y, -x), so the normal row is zl.z, the sliding rows zl.x / zl.y, the torsional row za.z and the
// rolling rows za.x / za.y (the two sliding and the two rolling rows have equal coefficients: the signs and the order
// within a pair do not matter). Index order here: 0,1 sliding, 2 normal, 3,4 rolling, 5 torsional.
struct Cone6 { float sc[6], D[6]; float mu, Dm; };
ODG_DEV Cone6 cone6_make(float Dn, float impratio, float mu, float fri, float dmk, float frt, float frr, float rt, float rr,
                         int condim = 3) {
  Cone6 k;
  if (condim == 1) { fri = 0.f; impratio = 0.f; }            // frictionless: normal row only (see cone_eval)
  k.sc[0] = fri; k.sc[1] = fri; k.sc[2] = mu; k.sc[3] = frr; k.sc[4] = frr; k.sc[5] = frt;
  const float Dt = Dn * impratio;
  k.D[0] = Dt; k.D[1] = Dt; k.D[2] = Dn; k.D[3] = Dn * rr; k.D[4] = Dn * rr; k.D[5] = Dn * rt;
  k.mu = mu; k.Dm = Dn * dmk;
  return k;
}
// gradient g (6) and Hessian H (6x6, symmetric, full storage) of the block's cost at z. Branch-free like cone_eval; a
// row whose friction coefficient is 0 (condim 3 contact in the same kernel) has sc = D = 0 and drops out exactly.
ODG_DEV void cone6_eval(const float (&z)[6], const Cone6& k, float (&g)[6], float (&H)[6][6]) {
  float U[6];
  ODG_UNROLL for (int i = 0; i < 6; i++) U[i] = z[i] * k.sc[i];
  const float N = U[2], mu = k.mu;
  const float T2 = U[0] * U[0] + U[1] * U[1] + U[3] * U[3] + U[4] * U[4] + U[5] * U[5];
  const float iT = odg_rsqrt(fmaxf(T2, 1e-20f));
  const float T = T2 * iT;
  const bool top = N >= mu * T;
  const bool bot = !top && (mu * N + T <= 0.f);
  const bool mid = !top && !bot;
  const float e = N - mu * T;
  const float De = k.Dm * e, kap = -k.Dm * mu * e * iT;
  float u[6], w[6];
  ODG_UNROLL for (int i = 0; i < 6; i++) { u[i] = (i == 2) ? 0.f : U[i] * iT; w[i] = (i == 2) ? mu : -mu * u[i] * k.sc[i]; }
  ODG_UNROLL for (int i = 0; i < 6; i++) g[i] = mid ? De * w[i] : (bot ? k.D[i] * z[i] : 0.f);
  ODG_UNROLL for (int i = 0; i < 6; i++)
    ODG_UNROLL for (int j = 0; j <= i; j++) {
      // cone surface: Dm w w^T + kappa * S (I - u u^T) S on the tangential rows (PSD term by term, see cone_eval)
      float hm = k.Dm * w[i] * w[j];
      if (i != 2 && j != 2) hm += kap * k.sc[i] * k.sc[j] * ((i == j ? 1.f : 0.f) - u[i] * u[j]);
      const float hb = (i == j) ? k.D[i] : 0.f;
      const float h = mid ? hm : (bot ? hb : 0.f);
      H[i][j] = h; H[j][i] = h;
    }
}
ODG_DEV LineCoef cone6_line_prep(const float (&z0)[6], const float (&dz)[6], const Cone6& k) {
  LineCoef c;
  c.cA = 0.f; c.cB = 0.f; c.cC = 0.f; c.q1 = 0.f; c.q2 = 0.f;
  ODG_UNROLL for (int i = 0; i < 6; i++) {           // (explicit fused operations, as in cone_line_prep)
    c.q1 = odg_fma_rn(odg_fmul_rn(k.D[i], z0[i]), dz[i], c.q1); c.q2 = odg_fma_rn(odg_fmul_rn(k.D[i], dz[i]), dz[i], c.q2);
    if (i != 2) {
      const float a = odg_fmul_rn(z0[i], k.sc[i]), b = odg_fmul_rn(dz[i], k.sc[i]);
      c.cA = odg_fma_rn(a, a, c.cA); c.cB = odg_fma_rn(a, b, c.cB); c.cC = odg_fma_rn(b, b, c.cC);
    }
  }
  c.N0 = odg_fmul_rn(z0[2], k.mu); c.Nd = odg_fmul_rn(dz[2], k.mu); c.mu = k.mu; c.Dm = k.Dm;
  return c;
}

// unrolled dense Cholesky solve of a 6x6 SPD system held in registers. S is overwritten by its factor.
ODG_DEV void chol6_solve(float (&S)[6][6], float (&x)[6]) {
  ODG_UNROLL for (int j = 0; j < 6; j++) {
    const float djj = S[j][j];
    float s = djj;
    ODG_UNROLL for (int k = 0; k < j; k++) s -= S[j][k] * S[j][k];
    // relative pivot floor: with contact stiffness D up to ~5e5 (deep penetration, impratio 100) against inertias of
    // ~1e-2 the Schur complement can lose positive-definiteness in fp32; a floored pivot keeps the direction finite
    // (the line search then decides whether it is still a descent direction) instead of producing NaN
    s = fmaxf(s, 1e-6f * fabsf(djj) + 1e-20f);
    float inv = odg_rsqrt(s);
    S[j][j] = inv;                                // store 1/L_jj
    ODG_UNROLL for (int i = j + 1; i < 6; i++) {
      float t = S[i][j];
      ODG_UNROLL for (int k = 0; k < j; k++) t -= S[i][k] * S[j][k];
      S[i][j] = t * inv;
    }
  }
  ODG_UNROLL for (int i = 0; i < 6; i++) {
    float t = x[i];
    ODG_UNROLL for (int k = 0; k < i; k++) t -= S[i][k] * x[k];
    x[i] = t * S[i][i];
  }
  ODG_UNROLL for (int i = 5; i >= 0; i--) {
    float t = x[i];
    ODG_UNROLL for (int k = i + 1; k < 6; k++) t -= S[k][i] * x[k];
    x[i] = t * S[i][i];
  }
}

// in-place inverse of a small SPD matrix (NJL x NJL), NJL in {1,2,3}
template <int N>
ODG_DEV void spd_inverse(float (&A)[N][N]) {
  if (N == 1) { A[0][0] = 1.f / A[0][0]; return; }
  if (N == 2) {
    float det = A[0][0] * A[1][1] - A[0][1] * A[0][1];
    float id = 1.f / det;
    float a = A[1][1] * id, b = -A[0][1] * id, c = A[0][0] * id;
    A[0][0] = a; A[0][1] = b; A[1][0] = b; A[1][1] = c; return;
  }
  // N == 3: adjugate
  float a = A[0][0], b = A[0][1], c = A[0][2], d = A[1][1], e = A[1][2], f = A[2][2];
  float c00 = d * f - e * e, c01 = c * e - b * f, c02 = b * e - c * d;
  float det = a * c00 + b * c01 + c * c02;
  float id = 1.f / det;
  A[0][0] = c00 * id; A[0][1] = A[1][0] = c01 * id; A[0][2] = A[2][0] = c02 * id;
  A[1][1] = (a * f - c * c) * id; A[1][2] = A[2][1] = (b * c - a * e) * id; A[2][2] = (a * d - b * b) * id;
}

// Cholesky factor of a small SPD matrix in place: A[i][k] (k < i) = L_ik, iL[i] = 1 / L_ii (relative pivot floor)
template <int N>
ODG_DEV void chol_small(float (&A)[N][N], float (&iL)[N]) {
  ODG_UNROLL for (int j = 0; j < N; j++) {
    const float djj = A[j][j];
    float s = djj;
    ODG_UNROLL for (int k = 0; k < j; k++) s -= A[j][k] * A[j][k];
    s = fmaxf(s, 1e-6f * fabsf(djj) + 1e-20f);
    iL[j] = odg_rsqrt(s);
    ODG_UNROLL for (int i = j + 1; i < N; i++) {
      float t = A[i][j];
      ODG_UNROLL for (int k = 0; k < j; k++) t -= A[i][k] * A[j][k];
      A[i][j] = t * iL[j];
    }
  }
}

struct Vec6 { V3 t, w; };   // linear / angular(world) parts
ODG_DEV float dot6(const Vec6& a, const Vec6& b) { return dot(a.t, b.t) + dot(a.w, b.w); }

// data the post-step code needs from the last forward pass
template <int NJL>
struct LastPass {
  int foot_contact;            // this leg's foot geom has a contact (paws_in_ground)
  V3 foot_force;               // (f_normal, f_t1, f_t2) of the LAST foot contact in MuJoCo's contact frame
  M3 R_last;                   // rotation of the last link (xquat[paw_body-1])
  float act[NJL];              // actuator forces
  Vec6 a_b; float a_l[NJL];    // qacc (trunk: linear, angular WORLD)
  int ncon, iters, ls_evals; float fn;
  // mj_rnePostConstraint's cfrc_ext of this leg's bodies, [torque about the whole robot's centre of mass, force] in
  // world axes, and this lane's share of the trunk's (3-joint legs only: the Go1 task rewards read them)
  float cfrc[NJL == 3 ? NJL + 1 : 1][6];
};

#define LCF(f, j) s_lc[((j) * LC_COUNT + (f)) * 4 + leg]
#define GCF(f, s) s_gc[((s) * GC_COUNT + (f)) * 4 + leg]

// One mj_step (or one mj_forward when integrate == false) for the 4-lane group of one environment.
// Every contact is an elliptic-cone block against the plane z = 0; a frictionless (condim 1) row is the same block
// with no tangential part (cone_eval / cone_line4).
// FAT = keep more per-contact data in (L1-cached) local memory instead of recomputing it: the joints' Jacobian columns at
// the contact point (once per substep) and the nine line-search coefficients (once per Newton iteration). Same
// arithmetic either way (results are bit-identical: the GPU suite compares a FAT handle with a lean one). It pays when
// a warp has a scheduler to itself (+6.5 % at 4096 envs) and costs when 8 warps per SM share the L1 — 26 instead of 14
// words per contact no longer fit (-18 % at 65536 envs) — so the host picks per batch size like it picks lockstep.
template <int NJL, bool FAT>
ODG_DEV void substep(const DevConst& C, const float* ODG_RESTRICT s_lc, const float* ODG_RESTRICT s_gc,
                     const float4* ODG_RESTRICT s_vert, int leg, unsigned gm,
                     V3& bp, float (&bq)[4], V3& bv, V3& bwl, float (&q)[NJL], float (&qd)[NJL],
                     const float (&ctrl)[NJL], V3& warm_v, V3& warm_wl, float (&warm_l)[NJL],
                     bool integrate, bool last, LastPass<NJL>& out, int& work, float* ODG_RESTRICT s_red) {
  const bool lane0 = (leg == 0);
  // ------------------------------------------------------------------ kinematics (mj_kinematics)
  {
    float n2 = bq[0] * bq[0] + bq[1] * bq[1] + bq[2] * bq[2] + bq[3] * bq[3];
    const bool degenerate = n2 < 1e-30f;
    const float in = odg_rsqrt(fmaxf(n2, 1e-30f));
    bq[0] = degenerate ? 1.f : bq[0] * in; bq[1] = degenerate ? 0.f : bq[1] * in;
    bq[2] = degenerate ? 0.f : bq[2] * in; bq[3] = degenerate ? 0.f : bq[3] * in;
  }
  M3 R0;
  {
    float w = bq[0], x = bq[1], y = bq[2], z = bq[3];
    R0.m[0] = w * w + x * x - y * y - z * z; R0.m[1] = 2.f * (x * y - w * z); R0.m[2] = 2.f * (x * z + w * y);
    R0.m[3] = 2.f * (x * y + w * z); R0.m[4] = w * w - x * x + y * y - z * z; R0.m[5] = 2.f * (y * z - w * x);
    R0.m[6] = 2.f * (x * z - w * y); R0.m[7] = 2.f * (y * z + w * x); R0.m[8] = w * w - x * x - y * y + z * z;
  }
  const V3 w0 = mul(R0, bwl);
  M3 R[NJL]; V3 pos[NJL], anc[NJL], ax[NJL], com[NJL];
  {
    M3 Rp = R0; V3 pp = mk3(0.f, 0.f, 0.f);
    ODG_UNROLL for (int j = 0; j < NJL; j++) {
      V3 pre = pp + mul(Rp, mk3(LCF(LC_BP0, j), LCF(LC_BP1, j), LCF(LC_BP2, j)));
      M3 Rpre = Rp;
      if (!C.body_rot_identity) {
        M3 Bq; ODG_UNROLL for (int k = 0; k < 9; k++) Bq.m[k] = LCF(LC_BR0 + k, j);
        Rpre = mul(Rp, Bq);
      }
      V3 jp = mk3(LCF(LC_JP0, j), LCF(LC_JP1, j), LCF(LC_JP2, j));
      V3 u = mk3(LCF(LC_JA0, j), LCF(LC_JA1, j), LCF(LC_JA2, j));
      anc[j] = pre + mul(Rpre, jp);
      ax[j] = mul(Rpre, u);
      float s, c; sincosf(q[j], &s, &c);
      float t = 1.f - c;
      M3 Rl;
      Rl.m[0] = c + t * u.x * u.x; Rl.m[1] = t * u.x * u.y - s * u.z; Rl.m[2] = t * u.x * u.z + s * u.y;
      Rl.m[3] = t * u.x * u.y + s * u.z; Rl.m[4] = c + t * u.y * u.y; Rl.m[5] = t * u.y * u.z - s * u.x;
      Rl.m[6] = t * u.x * u.z - s * u.y; Rl.m[7] = t * u.y * u.z + s * u.x; Rl.m[8] = c + t * u.z * u.z;
      R[j] = mul(Rpre, Rl);
      pos[j] = anc[j] - mul(R[j], jp);
      com[j] = pos[j] + mul(R[j], mk3(LCF(LC_IP0, j), LCF(LC_IP1, j), LCF(LC_IP2, j)));
      Rp = R[j]; pp = pos[j];
    }
  }
  // ------------------------------------------------------------------ inertias, CRBA (mj_crb)
  S3 Iw[NJL]; SpI cmp[NJL];
  ODG_UNROLL for (int j = 0; j < NJL; j++) {
    S3 Il; Il.xx = LCF(LC_IXX, j); Il.xy = LCF(LC_IXY, j); Il.xz = LCF(LC_IXZ, j);
    Il.yy = LCF(LC_IYY, j); Il.yz = LCF(LC_IYZ, j); Il.zz = LCF(LC_IZZ, j);
    Iw[j] = rotate_sym(R[j], Il);
    cmp[j] = spi_make(LCF(LC_MASS, j), com[j], Iw[j]);
  }
  ODG_UNROLL for (int j = NJL - 2; j >= 0; j--) cmp[j] = spi_add(cmp[j], cmp[j + 1]);
  // trunk body
  const V3 com0 = mul(R0, mk3(C.base_ip[0], C.base_ip[1], C.base_ip[2]));
  S3 Ib; Ib.xx = C.base_I[0]; Ib.xy = C.base_I[1]; Ib.xz = C.base_I[2]; Ib.yy = C.base_I[3]; Ib.yz = C.base_I[4]; Ib.zz = C.base_I[5];
  const S3 Iw0 = rotate_sym(R0, Ib);
  SpI T;                                           // trunk composite = trunk body + all legs
  {
    SpI b = spi_make(C.base_mass, com0, Iw0);
    T.m = b.m + grp_sum(cmp[0].m, gm);
    T.h = b.h + grp_sum(cmp[0].h, gm);
    T.I.xx = b.I.xx + grp_sum(cmp[0].I.xx, gm); T.I.xy = b.I.xy + grp_sum(cmp[0].I.xy, gm);
    T.I.xz = b.I.xz + grp_sum(cmp[0].I.xz, gm); T.I.yy = b.I.yy + grp_sum(cmp[0].I.yy, gm);
    T.I.yz = b.I.yz + grp_sum(cmp[0].I.yz, gm); T.I.zz = b.I.zz + grp_sum(cmp[0].I.zz, gm);
  }
  // leg blocks of M:  Mlb[j] = momentum (p, L about O) of composite j under unit joint velocity
  Vec6 Mlb[NJL]; float Mll[NJL][NJL]; V3 vax[NJL];
  ODG_UNROLL for (int j = 0; j < NJL; j++) {
    vax[j] = cross(anc[j], ax[j]);                 // velocity at O of unit rotation about the hinge
    Mlb[j].t = cmp[j].m * vax[j] + cross(ax[j], cmp[j].h);
    Mlb[j].w = mul(cmp[j].I, ax[j]) + cross(cmp[j].h, vax[j]);
  }
  ODG_UNROLL for (int j = 0; j < NJL; j++)
    ODG_UNROLL for (int i = 0; i <= j; i++) {
      float v = dot(ax[i], Mlb[j].w) + dot(vax[i], Mlb[j].t);
      if (i == j) v += LCF(LC_ARM, j);
      Mll[j][i] = v; Mll[i][j] = v;
    }
  // M_bb acts as: p = m*av + aw x h + arm_t.*av ; L = I*aw + h x av + arm_r*aw
  auto Mbb_mul = [&](const Vec6& a) {
    Vec6 r;
    r.t = T.m * a.t + cross(a.w, T.h) + mk3(C.base_arm_t[0] * a.t.x, C.base_arm_t[1] * a.t.y, C.base_arm_t[2] * a.t.z);
    r.w = mul(T.I, a.w) + cross(T.h, a.t) + C.base_arm_r * a.w;
    return r;
  };
  // ------------------------------------------------------------------ bias forces (mj_rne, flg_acc = 0)
  float cbias[NJL]; Vec6 cb;                       // cb = total inertial+gravity wrench about O (world)
  {
    const V3 g = mk3(C.gx, C.gy, C.gz);
    V3 F[NJL], tauO[NJL];
    V3 w = w0, al = mk3(0.f, 0.f, 0.f), r = mk3(0.f, 0.f, 0.f), aref = mk3(0.f, 0.f, 0.f);
    ODG_UNROLL for (int j = 0; j < NJL; j++) {
      V3 rho = anc[j] - r;
      aref = aref + cross(al, rho) + cross(w, cross(w, rho));
      r = anc[j];
      al = al + qd[j] * cross(w, ax[j]);
      w = w + qd[j] * ax[j];
      V3 rc = com[j] - r;
      V3 acom = aref + cross(al, rc) + cross(w, cross(w, rc));
      F[j] = LCF(LC_MASS, j) * (acom - g);
      V3 N = mul(Iw[j], al) + cross(w, mul(Iw[j], w));
      tauO[j] = cross(com[j], F[j]) + N;
    }
    V3 Fs = mk3(0.f, 0.f, 0.f), Ts = mk3(0.f, 0.f, 0.f);
    ODG_UNROLL for (int j = NJL - 1; j >= 0; j--) {
      Fs = Fs + F[j]; Ts = Ts + tauO[j];
      cbias[j] = dot(ax[j], Ts - cross(anc[j], Fs));
    }
    V3 a0 = cross(w0, cross(w0, com0));
    V3 F0 = C.base_mass * (a0 - g);
    V3 N0 = cross(w0, mul(Iw0, w0));
    cb.t = F0 + grp_sum(Fs, gm);
    cb.w = cross(com0, F0) + N0 + grp_sum(Ts, gm);
  }
  // ------------------------------------------------------------------ actuation + qfrc_smooth
  float tau_l[NJL];
  ODG_UNROLL for (int j = 0; j < NJL; j++) {
    float f = 0.f;
    if (LCF(LC_HASACT, j) != 0.f) {
      float c = ctrl[j];
      if (LCF(LC_CLIM, j) != 0.f) c = fmaxf(LCF(LC_CLO, j), fminf(LCF(LC_CHI, j), c));
      f = LCF(LC_KP, j) * c - LCF(LC_KP, j) * q[j] - LCF(LC_KV, j) * qd[j];
      if (LCF(LC_FLIM, j) != 0.f) f = fmaxf(LCF(LC_FLO, j), fminf(LCF(LC_FHI, j), f));
    }
    out.act[j] = f;
    tau_l[j] = f - cbias[j] - LCF(LC_DAMP, j) * qd[j];
  }
  // ------------------------------------------------------------------ collision: floor plane vs hulls
  // cone rows of this leg's contacts, as 16-byte records: (r, Dn) — Dn holds the distance until the rows are built —,
  // (aref, slot index bits), (z0, -)
  float4 c_ra[kMaxConLeg], c_af[kMaxConLeg], c_z0[kMaxConLeg];
  float4 c_lc[FAT ? kMaxConLeg : 1][3];                           // FAT: their line-search coefficients (LineCoef) for the current direction
  float4 c_dz[FAT ? 1 : kMaxConLeg];                              // lean: the direction's row values (coefficients are re-derived per pass)
  float4 c_cj[FAT ? kMaxConLeg : 1][NJL];                                       // Jacobian columns of this leg's joints at the contact point
                                                                  // (zero for joints below the contact's link)
  // 3-joint legs (Go1): every contact carries the three angular rows of condim 6 as well (torsional + rolling friction,
  // go1.xml:61-64); contacts of condim-3 geoms have zero coefficients there and reduce to the 3-row cone exactly
  constexpr bool kG = (NJL == 3);
  // FAT with 3-row cones: the spare words of a contact's records carry its cone constants — mu and the friction coefficient
  // (0 for a frictionless row) next to the two Jacobian columns, 1 / (mu^2 (1 + mu^2)) in place of the slot index once
  // the rows are built — so the iteration's loops need no per-slot constant lookups (dependent constant-bank loads)
  constexpr bool kStash = FAT && !kG && NJL >= 2;
  constexpr int kConA = kG ? kMaxConLeg : 1;
  float4 c_arefa[kConA], c_z0a[kConA], c_dza[(kG && !FAT) ? kMaxConLeg : 1];
  int nc = 0;
  int foot_last = -1;
  auto add_contact = [&](float px, float py, float pz_mid, float dist, int s) {
    if (nc >= kMaxConLeg) return;
    c_ra[nc] = mk4(mk3(px, py, pz_mid), dist);
    c_af[nc] = mk4(mk3(0.f, 0.f, 0.f), odg_int_bits(s));
    if (C.slot_isfoot[s]) foot_last = nc;
    nc++;
  };
  for (int s = 0; s < C.nslot; s++) {
    const int link = C.slot_link[s];
    M3 Rl = R[0]; V3 pl = pos[0];
    ODG_UNROLL for (int j = 1; j < NJL; j++) if (link == j) { Rl = R[j]; pl = pos[j]; }
    const float margin = C.slot_margin[s];
    if constexpr (kG) {
      if (C.per_lane_geoms) {
        // Primitive colliders against the plane (go1.xml:26-64): the lane's own geom of this slot. Trunk colliders
        // (link -1) are dealt out over the four lanes. Restates mjc_PlaneSphere / PlaneCapsule / PlaneCylinder / PlaneBox
        // (oracle/odg_oracle.c: odgo_collision holds the same rules in double).
        if (link < 0) { Rl = R0; pl = mk3(0.f, 0.f, 0.f); }
        const int type = (int)GCF(GC_TYPE, s);
        if (type == PRIM_NONE) continue;
        const V3 cc = pl + mul(Rl, mk3(GCF(GC_CX, s), GCF(GC_CY, s), GCF(GC_CZ, s)));
        const float s0 = GCF(GC_S0, s), s1 = GCF(GC_S1, s), s2 = GCF(GC_S2, s);
        const float cz = bp.z + cc.z;
        if (cz - (s0 + s1 + s2) > margin) continue;              // (cull: no primitive reaches further than the sum of its sizes)
        if (type == PRIM_SPHERE) {
          const float dist = cz - s0;
          if (dist <= margin) add_contact(cc.x, cc.y, cc.z - s0 - 0.5f * dist, dist, s);
          continue;
        }
        M3 Gm; ODG_UNROLL for (int k = 0; k < 9; k++) Gm.m[k] = GCF(GC_R0 + k, s);
        const M3 Mw = mul(Rl, Gm);
        if (type == PRIM_CAPSULE) {
          const V3 axc = col(Mw, 2);
          for (int e = 0; e < 2; e++) {                          // +axis end first
            const V3 pe = cc + ((e ? -s1 : s1) * axc);
            const float dist = bp.z + pe.z - s0;
            if (dist <= margin) add_contact(pe.x, pe.y, pe.z - s0 - 0.5f * dist, dist, s);
          }
        } else if (type == PRIM_BOX) {
          int cnt = 0;
          for (int i = 0; i < 8 && cnt < 4; i++) {                // corners in index order, the first four that qualify
            const V3 cr = mul(Mw, mk3((i & 1) ? s0 : -s0, (i & 2) ? s1 : -s1, (i & 4) ? s2 : -s2));
            if (cz + cr.z > margin || cr.z > 0.f) continue;
            const float dist = cz + cr.z;
            add_contact(cc.x + cr.x, cc.y + cr.y, cc.z + cr.z - 0.5f * dist, dist, s);
            cnt++;
          }
        } else {                                                  // cylinder
          V3 axc = col(Mw, 2);
          float prjaxis = axc.z;
          if (prjaxis > 0.f) { axc = -axc; prjaxis = -prjaxis; }
          V3 vec = mk3(axc.x * prjaxis, axc.y * prjaxis, axc.z * prjaxis - 1.f);
          const float len2 = dot(vec, vec);
          if (len2 >= 1e-30f) vec = (s0 * odg_rsqrt(len2)) * vec; else vec = s0 * col(Mw, 0);
          const float prjvec = vec.z, prjaxs = prjaxis * s1;
          const V3 axs = s1 * axc;
          const float d1 = cz + prjaxs + prjvec;
          if (d1 <= margin) {
            add_contact(cc.x + vec.x + axs.x, cc.y + vec.y + axs.y, cc.z + vec.z + axs.z - 0.5f * d1, d1, s);
            const float d2 = cz - prjaxs + prjvec;
            if (d2 <= margin) add_contact(cc.x + vec.x - axs.x, cc.y + vec.y - axs.y, cc.z + vec.z - axs.z - 0.5f * d2, d2, s);
            const float d3 = cz + prjaxs - 0.5f * prjvec;
            if (d3 <= margin) {
              V3 v1 = cross(vec, axc);
              const float l2 = dot(v1, v1);
              v1 = (l2 > 0.f ? s0 * 0.8660254037844386f * odg_rsqrt(l2) : 0.f) * v1;
              const V3 pm = cc + axs - 0.5f * vec;
              add_contact(pm.x + v1.x, pm.y + v1.y, pm.z + v1.z - 0.5f * d3, d3, s);
              add_contact(pm.x - v1.x, pm.y - v1.y, pm.z - v1.z - 0.5f * d3, d3, s);
            }
          }
        }
        continue;
      }
    }
    const float zoff = bp.z + pl.z;
    if (C.slot_type[s] == 1) {                     // sphere
      V3 cc = pl + mul(Rl, mk3(GCF(GC_CX, s), GCF(GC_CY, s), GCF(GC_CZ, s)));
      float dist = bp.z + cc.z - C.slot_radius[s];
      if (dist <= margin) add_contact(cc.x, cc.y, cc.z - C.slot_radius[s] - 0.5f * dist, dist, s);
      continue;
    }
    {                                               // conservative cull: lowest point of the hull's bounding box (link
                                                    // frame) clear of the margin. Measured on the bench workload: the calf
                                                    // hull passed a bounding-SPHERE cull 65 % of the time without ever touching.
      const V3 bc = pl + mul(Rl, mk3(GCF(GC_BX, s), GCF(GC_BY, s), GCF(GC_BZ, s)));
      const float ext = fabsf(Rl.m[6]) * GCF(GC_HX, s) + fabsf(Rl.m[7]) * GCF(GC_HY, s) + fabsf(Rl.m[8]) * GCF(GC_HZ, s);
      if (bp.z + bc.z - ext > margin) continue;
    }
    const int vs = C.slot_vstart[s];
    const V3 rz = mk3(Rl.m[6], Rl.m[7], Rl.m[8]);
    // Foot hulls: one pass over the vertices finds the support vertex towards the floor (lowest world z) and towards
    // the three tilted directions of the multi-contact search at once — each vertex is loaded once and the four running
    // arg-extrema are independent chains (somewhere in the warp a paw touches the floor in nearly every substep, so
    // the warp walks the tilted scans anyway). Other hulls (thigh, calf) often pass the box cull without touching: they
    // get the cheap z-only pass first and the three tilted directions only when they do touch. The choice depends on
    // the slot index alone, so it is uniform across the warp.
    V3 dl[3];
    ODG_UNROLL for (int i = 0; i < 3; i++) dl[i] = tmul(Rl, mk3(C.tilt_dir[i][0], C.tilt_dir[i][1], C.tilt_dir[i][2]));
    // Only the hull vertices whose normal cone meets the (widened) cell of the floor direction -rz in the link frame
    // can win any of the four searches: the host lists them per cell (dominant axis x component signs; odg_prep.h:
    // hull_vertex_is_candidate), in index order, so the first-index tie rule of a full scan is preserved.
    const float arx = fabsf(rz.x), ary = fabsf(rz.y), arz = fabsf(rz.z);
    const int axis = (arx >= ary && arx >= arz) ? 0 : (ary >= arz ? 1 : 2);
    const int oct = (rz.x > 0.f ? 1 : 0) | (rz.y > 0.f ? 2 : 0) | (rz.z > 0.f ? 4 : 0);     // signs of -rz
    const int oct_ent = reinterpret_cast<const int*>(s_gc + C.oct_off)[(s * kSupportCells + axis * 8 + oct) * 4 + leg];
    const unsigned char* ODG_RESTRICT cand = reinterpret_cast<const unsigned char*>(s_gc + C.idx_off) + (oct_ent & 0xFFFF);
    const int ncand = oct_ent >> 16;
    float zmin = 1e30f; int best = 0;
    float smax[3] = { -1e30f, -1e30f, -1e30f }; int bi3[3] = { 0, 0, 0 };
    if (C.slot_isfoot[s]) {
      for (int kk = 0; kk < ncand; kk++) {
        const int k = cand[kk];
        const float4 v = s_vert[(vs + k) * 4 + leg];
        const float z = zoff + rz.x * v.x + rz.y * v.y + rz.z * v.z;
        const bool lower = z < zmin;
        zmin = lower ? z : zmin; best = lower ? k : best;
        ODG_UNROLL for (int i = 0; i < 3; i++) {
          const float sc = dl[i].x * v.x + dl[i].y * v.y + dl[i].z * v.z;
          const bool more = sc > smax[i];
          smax[i] = more ? sc : smax[i]; bi3[i] = more ? k : bi3[i];
        }
      }
    } else {
      for (int kk = 0; kk < ncand; kk++) {
        const int k = cand[kk];
        const float4 v = s_vert[(vs + k) * 4 + leg];
        const float z = zoff + rz.x * v.x + rz.y * v.y + rz.z * v.z;
        const bool lower = z < zmin;
        zmin = lower ? z : zmin; best = lower ? k : best;
      }
      if (zmin > margin) continue;
      for (int kk = 0; kk < ncand; kk++) {
        const int k = cand[kk];
        const float4 v = s_vert[(vs + k) * 4 + leg];
        ODG_UNROLL for (int i = 0; i < 3; i++) {
          const float sc = dl[i].x * v.x + dl[i].y * v.y + dl[i].z * v.z;
          const bool more = sc > smax[i];
          smax[i] = more ? sc : smax[i]; bi3[i] = more ? k : bi3[i];
        }
      }
    }
    if (zmin > margin) continue;
    int found[4] = { best, -1, -1, -1 }; int nf = 1;
    {
      float4 v = s_vert[(vs + best) * 4 + leg];
      V3 pw = pl + mul(Rl, mk3(v.x, v.y, v.z));
      add_contact(pw.x, pw.y, 0.5f * zmin - bp.z, zmin, s);
    }
    ODG_UNROLL for (int i = 0; i < 3; i++) {
      if (i >= C.n_tilt) continue;
      const int bi = bi3[i];
      bool dup = false;
      ODG_UNROLL for (int k = 0; k < 4; k++) dup |= (found[k] == bi);
      if (dup) continue;
      float4 v = s_vert[(vs + bi) * 4 + leg];
      V3 pw = pl + mul(Rl, mk3(v.x, v.y, v.z));
      float z = bp.z + pw.z;
      if (z > margin) continue;
      ODG_UNROLL for (int k = 1; k < 4; k++) if (k == nf) found[k] = bi;
      nf++;
      add_contact(pw.x, pw.y, 0.5f * z - bp.z, z, s);
    }
  }
  // ------------------------------------------------------------------ constraint rows (mj_makeConstraint/Impedance)
  // contacts: c_ra.w currently holds dist; turn into D_n and build aref
  for (int c = 0; c < nc; c++) {
    const float4 ra = c_ra[c];
    const int s = odg_float_bits(c_af[c].w);
    const int link = C.slot_link[s];
    const float dist = ra.w;
    const float margin = C.slot_margin[s];
    float active = dist < margin ? 1.f : 0.f;       // excluded if in the gap (gap = 0: never for dist==margin only)
    float imp = impedance(C.slot_imp[s], dist - margin);
    float Rn = fmaxf(1e-15f, odg_fdiv_fast(1.f - imp, imp) * GCF(GC_INVW, s));
    const float Bc = C.slot_B[s], Kc = C.slot_K[s];
    const V3 r = xyz(ra);
    c_ra[c] = mk4(r, odg_fdiv_fast(active, Rn));
    V3 vc = bv + cross(w0, r);
    ODG_UNROLL for (int j = 0; j < NJL; j++) {
      const V3 cjv = (j <= link) ? cross(ax[j], r - anc[j]) : mk3(0.f, 0.f, 0.f);
      if (FAT) c_cj[c][j] = mk4(cjv, j == 0 ? C.slot_mu[s] : (C.slot_condim[s] == 1 ? 0.f : C.slot_fri[s]));
      vc = vc + qd[j] * cjv;
    }
    c_af[c] = mk4(mk3(-Bc * vc.x, -Bc * vc.y, -Bc * vc.z - Kc * imp * (dist - margin)), kStash ? C.slot_dmk[s] : odg_int_bits(s));
    if constexpr (kG) {                             // torsional / rolling rows: aref = -B * (angular velocity of the body)
      V3 wb = w0;
      ODG_UNROLL for (int j = 0; j < NJL; j++) {
        const float on = fminf(fmaxf((float)(link - j + 1), 0.f), 1.f);
        wb = wb + (on * qd[j]) * ax[j];
      }
      c_arefa[c] = mk4(mk3(-Bc * wb.x, -Bc * wb.y, -Bc * wb.z), 0.f);
    }
  }
  // own-joint friction-loss and limit rows
  float aref_fl[NJL], lim_sgn[NJL], lim_aref[NJL], lim_D[NJL];
  ODG_UNROLL for (int j = 0; j < NJL; j++) {
    aref_fl[j] = -C.B_fl * qd[j];
    {
      // (branch-free: an inactive or absent limit ends up with sgn = D = aref = 0)
      const float dlo = q[j] - LCF(LC_LO, j), dhi = LCF(LC_HI, j) - q[j];
      const bool lim = LCF(LC_LIMITED, j) != 0.f, lo_on = lim && dlo < 0.f, hi_on = lim && !lo_on && dhi < 0.f;
      const float dist = lo_on ? dlo : (hi_on ? dhi : 0.f), sg = lo_on ? 1.f : (hi_on ? -1.f : 0.f);
      const float imp = impedance(C.lim_imp, dist);
      const float Rr = fmaxf(1e-15f, odg_fdiv_fast(1.f - imp, imp) * LCF(LC_INVW, j));
      lim_sgn[j] = sg; lim_D[j] = sg != 0.f ? odg_fdiv_fast(1.f, Rr) : 0.f;
      lim_aref[j] = sg != 0.f ? -C.B_lim * (sg * qd[j]) - C.K_lim * imp * dist : 0.f;
    }
  }
  // trunk friction-loss rows (DoFs in MuJoCo's frames: world linear, trunk-frame angular)
  const int bfi = leg < 3 ? leg : 0;
  const V3 bf_e = mk3(leg == 0 ? 1.f : 0.f, leg == 1 ? 1.f : 0.f, leg == 2 ? 1.f : 0.f);   // world axis of the row
  const V3 bf_c = leg == 0 ? col(R0, 0) : (leg == 1 ? col(R0, 1) : col(R0, 2));             // trunk axis, world
  const float bf_ft = leg < 3 ? C.base_fl[bfi] : 0.f, bf_Rt = C.base_Rfl[bfi], bf_Dt = C.base_Dfl[bfi];
  const float bf_fr = leg < 3 ? C.base_fl[3 + bfi] : 0.f, bf_Rr = C.base_Rfl[3 + bfi], bf_Dr = C.base_Dfl[3 + bfi];
  const float bf_aref_t = -C.B_fl * dot(bf_e, bv);
  const float bf_aref_r = -C.B_fl * comp(bwl, bfi);
  const Vec6 tau_b = { -cb.t, -cb.w };
  // ------------------------------------------------------------------ Newton solve of the primal problem
  Vec6 a_b; float a_l[NJL];
  a_b.t = warm_v; a_b.w = mul(R0, warm_wl);
  ODG_UNROLL for (int j = 0; j < NJL; j++) a_l[j] = warm_l[j];
  const float l0f = lane0 ? 1.f : 0.f;
  int iters = 0, ls_evals = 0;
  bool conv = false;
  for (int it = 0; it < C.solver_iters; it++) {
#if !defined(ODG_NO_LOCKSTEP) && !defined(ODG_HOST_EMU)
    // All warps of the block walk the Newton-iteration body (~26 KB of SASS) together, so its instruction-cache lines
    // are fetched once per block instead of once per warp: with more than ~4 independent instruction streams per SM
    // the step kernel is instruction-fetch bound on B200 (32 KB L1.5 I-cache; stall reason no_instruction, profiles/).
    // Every thread of the block reaches this barrier the same number of times: substeps are uniform and padding
    // environments are stepped like real ones. It pays when the batch is several waves deep (+27 % at 65536 envs,
    // although 13 % of the samples then sit here) and costs a little when every warp has a scheduler to itself
    // (-2 % at 4096), so the host enables it per batch size (DevConst::lockstep).
    if (C.lockstep) {
      // lockstep == 2: PAIRS of warps inside a larger block (named barrier 1 + pair index, 64 threads): the pairing that
      // is fastest, with the block's constants staged once for two pairs — half the shared memory per SM, which keeps
      // four pairs under a smaller carve-out and leaves the L1 to the local-memory traffic
      int any;
      if (C.lockstep == 2) {
        asm volatile("{\n .reg .pred p, q;\n setp.ne.u32 q, %1, 0;\n bar.red.or.pred p, %2, 64, q;\n selp.u32 %0, 1, 0, p;\n}\n"
                     : "=r"(any) : "r"(conv ? 0u : 1u), "r"(1u + (threadIdx.x >> 6)) : "memory");
      } else {
        any = __syncthreads_or(conv ? 0 : 1);
      }
      if (!any) break;
      if (conv) continue;
    } else if (conv) break;
#else
    if (conv) break;
#endif
    iters = it + 1;
    // ---- gradient and Hessian at a
    float g_l[NJL], Hll[NJL][NJL]; Vec6 Hlb[NJL]; Vec6 gb;
    S3 Htt = zero_s3(), Hww = zero_s3(); float Htw[3][3];
    ODG_UNROLL for (int i = 0; i < 3; i++) ODG_UNROLL for (int k = 0; k < 3; k++) Htw[i][k] = 0.f;
    Vec6 Mab = Mbb_mul(a_b);
    gb.t = l0f * (Mab.t - tau_b.t); gb.w = l0f * (Mab.w - tau_b.w);
    float gauss_l[NJL];
    ODG_UNROLL for (int j = 0; j < NJL; j++) {
      float s = dot6(Mlb[j], a_b);
      ODG_UNROLL for (int i = 0; i < NJL; i++) { s += Mll[j][i] * a_l[i]; Hll[j][i] = Mll[j][i]; }
      gauss_l[j] = s - tau_l[j];
      g_l[j] = gauss_l[j];
      Hlb[j] = Mlb[j];
      gb.t = gb.t + a_l[j] * Mlb[j].t; gb.w = gb.w + a_l[j] * Mlb[j].w;
    }
    const Vec6 gauss_b = gb;                        // lane-partial of (M a - tau)_trunk
    // joint friction-loss + limits
    // (branch-free: a row that does not exist has fl = 0 / D = 0 and adds exactly 0)
    ODG_UNROLL for (int j = 0; j < NJL; j++) {
      {
        float g, hh; fl_eval(a_l[j] - aref_fl[j], LCF(LC_FL, j), LCF(LC_RFL, j), LCF(LC_DFL, j), g, hh);
        g_l[j] += g; Hll[j][j] += hh;
      }
      {
        const float z = lim_sgn[j] * a_l[j] - lim_aref[j];
        const float Dl = z < 0.f ? lim_D[j] : 0.f;
        g_l[j] += lim_sgn[j] * Dl * z; Hll[j][j] += Dl;
      }
    }
    // trunk friction-loss rows: lane l < 3 owns translational row l and rotational row l
    {
      float g, hh; fl_eval(dot(bf_e, a_b.t) - bf_aref_t, bf_ft, bf_Rt, bf_Dt, g, hh);
      gb.t = gb.t + g * bf_e;
      Htt.xx += hh * bf_e.x; Htt.yy += hh * bf_e.y; Htt.zz += hh * bf_e.z;
    }
    {
      float g, hh; fl_eval(dot(bf_c, a_b.w) - bf_aref_r, bf_fr, bf_Rr, bf_Dr, g, hh);
      gb.w = gb.w + g * bf_c;
      Hww.xx += hh * bf_c.x * bf_c.x; Hww.xy += hh * bf_c.x * bf_c.y; Hww.xz += hh * bf_c.x * bf_c.z;
      Hww.yy += hh * bf_c.y * bf_c.y; Hww.yz += hh * bf_c.y * bf_c.z; Hww.zz += hh * bf_c.z * bf_c.z;
    }
    // contacts
    ODG_NO_UNROLL for (int c = 0; c < nc; c++) {
      const float4 ra = c_ra[c], af = c_af[c];
      const int s = kStash ? 0 : odg_float_bits(af.w);
      const int link = C.slot_link[s];
      const V3 r = xyz(ra);
      V3 cj[NJL];
      float cjw[NJL];                               // (kStash: mu, friction)
      V3 ap = cross_acc(a_b.t, a_b.w, r);
      ODG_UNROLL for (int j = 0; j < NJL; j++) {
        const float4 q = FAT ? c_cj[c][j] : mk4(((j <= link) ? cross(ax[j], r - anc[j]) : mk3(0.f, 0.f, 0.f)), 0.f);
        cj[j] = xyz(q); cjw[j] = q.w;
        ap = ap + a_l[j] * cj[j];
      }
      V3 z = ap - xyz(af);
      c_z0[c] = mk4(z, 0.f);
      const float Dn = ra.w;
      if constexpr (kG) {
        // 6-row block: linear rows through the contact point's Jacobian (column of DoF d: cl_d), angular rows through
        // the body's rotational Jacobian (column ca_d): trunk translation (e_i, 0), trunk rotation (e_k x r, e_k),
        // joint j (cj[j], ax[j]) when the joint is above the contact's link
        V3 aj[NJL];
        V3 alb = a_b.w;
        ODG_UNROLL for (int j = 0; j < NJL; j++) {
          aj[j] = (j <= link) ? ax[j] : mk3(0.f, 0.f, 0.f);
          alb = alb + a_l[j] * aj[j];
        }
        const V3 za = alb - xyz(c_arefa[c]);
        c_z0a[c] = mk4(za, 0.f);
        const Cone6 K6 = cone6_make(Dn, C.impratio, C.slot_mu[s], C.slot_fri[s], C.slot_dmk[s], C.slot_frt[s], C.slot_frr[s],
                                    C.slot_dt_tor[s], C.slot_dt_roll[s], C.slot_condim[s]);
        const float z6[6] = { z.x, z.y, z.z, za.x, za.y, za.z };
        float g6[6], H6[6][6];
        cone6_eval(z6, K6, g6, H6);
        const V3 gL = mk3(g6[0], g6[1], g6[2]), gA = mk3(g6[3], g6[4], g6[5]);
        gb.t = gb.t + gL; gb.w = gb.w + cross(r, gL) + gA;
        auto HLL = [&](V3 v) { return mk3(H6[0][0] * v.x + H6[0][1] * v.y + H6[0][2] * v.z, H6[1][0] * v.x + H6[1][1] * v.y + H6[1][2] * v.z,
                                          H6[2][0] * v.x + H6[2][1] * v.y + H6[2][2] * v.z); };
        auto HLA = [&](V3 v) { return mk3(H6[0][3] * v.x + H6[0][4] * v.y + H6[0][5] * v.z, H6[1][3] * v.x + H6[1][4] * v.y + H6[1][5] * v.z,
                                          H6[2][3] * v.x + H6[2][4] * v.y + H6[2][5] * v.z); };
        auto HAL = [&](V3 v) { return mk3(H6[3][0] * v.x + H6[3][1] * v.y + H6[3][2] * v.z, H6[4][0] * v.x + H6[4][1] * v.y + H6[4][2] * v.z,
                                          H6[5][0] * v.x + H6[5][1] * v.y + H6[5][2] * v.z); };
        auto HAA = [&](V3 v) { return mk3(H6[3][3] * v.x + H6[3][4] * v.y + H6[3][5] * v.z, H6[4][3] * v.x + H6[4][4] * v.y + H6[4][5] * v.z,
                                          H6[5][3] * v.x + H6[5][4] * v.y + H6[5][5] * v.z); };
        Htt.xx += H6[0][0]; Htt.xy += H6[0][1]; Htt.xz += H6[0][2]; Htt.yy += H6[1][1]; Htt.yz += H6[1][2]; Htt.zz += H6[2][2];
        // trunk rotation k: linear column X_k = e_k x r, angular column e_k
        const V3 Xk[3] = { mk3(0.f, -r.z, r.y), mk3(r.z, 0.f, -r.x), mk3(-r.y, r.x, 0.f) };
        const V3 Ek[3] = { mk3(1.f, 0.f, 0.f), mk3(0.f, 1.f, 0.f), mk3(0.f, 0.f, 1.f) };
        V3 hL[3], hA[3];                             // H * column k: linear / angular parts
        ODG_UNROLL for (int k = 0; k < 3; k++) { hL[k] = HLL(Xk[k]) + HLA(Ek[k]); hA[k] = HAL(Xk[k]) + HAA(Ek[k]); }
        ODG_UNROLL for (int k = 0; k < 3; k++) { Htw[0][k] += hL[k].x; Htw[1][k] += hL[k].y; Htw[2][k] += hL[k].z; }
        Hww.xx += dot(Xk[0], hL[0]) + hA[0].x; Hww.xy += dot(Xk[0], hL[1]) + hA[1].x; Hww.xz += dot(Xk[0], hL[2]) + hA[2].x;
        Hww.yy += dot(Xk[1], hL[1]) + hA[1].y; Hww.yz += dot(Xk[1], hL[2]) + hA[2].y; Hww.zz += dot(Xk[2], hL[2]) + hA[2].z;
        ODG_UNROLL for (int j = 0; j < NJL; j++) {
          const V3 hcL = HLL(cj[j]) + HLA(aj[j]), hcA = HAL(cj[j]) + HAA(aj[j]);
          g_l[j] += dot(cj[j], gL) + dot(aj[j], gA);
          Hlb[j].t = Hlb[j].t + hcL; Hlb[j].w = Hlb[j].w + cross(r, hcL) + hcA;
          ODG_UNROLL for (int i = 0; i <= j; i++) {
            float v = dot(cj[i], hcL) + dot(aj[i], hcA);
            Hll[j][i] += v; if (i != j) Hll[i][j] += v;
          }
        }
        continue;
      }
      V3 g; S3 H;
      if constexpr (kStash) cone_eval(z, Dn, cjw[1] != 0.f ? Dn * C.impratio : 0.f, cjw[0], cjw[1], af.w, 3, g, H);
      else cone_eval(z, Dn, Dn * C.impratio, C.slot_mu[s], C.slot_fri[s], C.slot_dmk[s], C.slot_condim[s], g, H);
      // (separated rows and rows with D = 0 come back as g = 0, H = 0 and add exactly 0 below)
      gb.t = gb.t + g; gb.w = cross_acc(gb.w, r, g);
      // H * X, X = -[r]x : column i of X is e_i x r = (0, -r.z, r.y), (r.z, 0, -r.x), (-r.y, r.x, 0). Written out with the
      // zeros dropped: every entry of H X and of X^T (H X) is one "a*b - c*d".
      const V3 HX0 = mk3(cross1(H.xz, r.y, H.xy, r.z), cross1(H.yz, r.y, H.yy, r.z), cross1(H.zz, r.y, H.yz, r.z));
      const V3 HX1 = mk3(cross1(H.xx, r.z, H.xz, r.x), cross1(H.xy, r.z, H.yz, r.x), cross1(H.xz, r.z, H.zz, r.x));
      const V3 HX2 = mk3(cross1(H.xy, r.x, H.xx, r.y), cross1(H.yy, r.x, H.xy, r.y), cross1(H.yz, r.x, H.xz, r.y));
      Htt.xx += H.xx; Htt.xy += H.xy; Htt.xz += H.xz; Htt.yy += H.yy; Htt.yz += H.yz; Htt.zz += H.zz;
      Htw[0][0] += HX0.x; Htw[1][0] += HX0.y; Htw[2][0] += HX0.z;
      Htw[0][1] += HX1.x; Htw[1][1] += HX1.y; Htw[2][1] += HX1.z;
      Htw[0][2] += HX2.x; Htw[1][2] += HX2.y; Htw[2][2] += HX2.z;
      // X0 . v = r.y v.z - r.z v.y,  X1 . v = r.z v.x - r.x v.z,  X2 . v = r.x v.y - r.y v.x
      Hww.xx = cross1_acc(Hww.xx, r.y, HX0.z, r.z, HX0.y); Hww.xy = cross1_acc(Hww.xy, r.y, HX1.z, r.z, HX1.y);
      Hww.xz = cross1_acc(Hww.xz, r.y, HX2.z, r.z, HX2.y); Hww.yy = cross1_acc(Hww.yy, r.z, HX1.x, r.x, HX1.z);
      Hww.yz = cross1_acc(Hww.yz, r.z, HX2.x, r.x, HX2.z); Hww.zz = cross1_acc(Hww.zz, r.x, HX2.y, r.y, HX2.x);
      ODG_UNROLL for (int j = 0; j < NJL; j++) {    // (cj[j] = 0 for joints below the contact's link: adds exactly 0)
        V3 hc = mul(H, cj[j]);
        g_l[j] = dot_acc(g_l[j], cj[j], g);
        Hlb[j].t = Hlb[j].t + hc; Hlb[j].w = cross_acc(Hlb[j].w, r, hc);
        ODG_UNROLL for (int i = 0; i <= j; i++) Hll[j][i] = dot_acc(Hll[j][i], cj[i], hc);   // (lower triangle: all chol_small reads)
      }
    }
    // ---- eliminate the leg block: Schur complement on the trunk
    // block Cholesky: Hll = L L^T, W = L^-1 Hlb, y = L^-1 g_l (forward substitutions). The Schur complement is then
    // P - W^T W — a symmetric subtraction that stays positive semi-definite in fp32, unlike P - Hlb^T (Hll^-1 Hlb) with
    // an explicit adjugate inverse, which turned indefinite for stiff contacts (Go1 feet: D ~ 5e5 against 1e-2 inertias).
    float iL[NJL];
    chol_small<NJL>(Hll, iL);
    Vec6 W[NJL]; float y[NJL];
    ODG_UNROLL for (int j = 0; j < NJL; j++) {
      W[j] = Hlb[j]; y[j] = g_l[j];
      ODG_UNROLL for (int i = 0; i < j; i++) {
        W[j].t = W[j].t - Hll[j][i] * W[i].t; W[j].w = W[j].w - Hll[j][i] * W[i].w;
        y[j] -= Hll[j][i] * y[i];
      }
      W[j].t = iL[j] * W[j].t; W[j].w = iL[j] * W[j].w; y[j] *= iL[j];
    }
    float S[6][6]; float rhs[6];
    {
      // lane-partial trunk block: (lane0 ? M_bb : 0) + friction/contact terms - sum_j Hlb[j]^T W[j]
      float P[6][6];
      ODG_UNROLL for (int i = 0; i < 6; i++) ODG_UNROLL for (int k = 0; k < 6; k++) P[i][k] = 0.f;
      P[0][0] = Htt.xx; P[1][0] = Htt.xy; P[2][0] = Htt.xz; P[1][1] = Htt.yy; P[2][1] = Htt.yz; P[2][2] = Htt.zz;
      P[3][3] = Hww.xx; P[4][3] = Hww.xy; P[5][3] = Hww.xz; P[4][4] = Hww.yy; P[5][4] = Hww.yz; P[5][5] = Hww.zz;
      ODG_UNROLL for (int i = 0; i < 3; i++) ODG_UNROLL for (int k = 0; k < 3; k++) P[3 + k][i] = Htw[i][k];
      // M_bb (lane 0): [[m I + arm_t, -[h]x], [[h]x, I + arm_r]]  (lower triangle rows w, cols t = [h]x)
      P[0][0] += l0f * (T.m + C.base_arm_t[0]); P[1][1] += l0f * (T.m + C.base_arm_t[1]); P[2][2] += l0f * (T.m + C.base_arm_t[2]);
      P[3][3] += l0f * (T.I.xx + C.base_arm_r); P[4][3] += l0f * T.I.xy; P[5][3] += l0f * T.I.xz;
      P[4][4] += l0f * (T.I.yy + C.base_arm_r); P[5][4] += l0f * T.I.yz; P[5][5] += l0f * (T.I.zz + C.base_arm_r);
      // [h]x = [[0,-hz,hy],[hz,0,-hx],[-hy,hx,0]] -> P[3+row][col]
      P[3][1] += l0f * (-T.h.z); P[3][2] += l0f * (T.h.y);
      P[4][0] += l0f * (T.h.z);  P[4][2] += l0f * (-T.h.x);
      P[5][0] += l0f * (-T.h.y); P[5][1] += l0f * (T.h.x);
      float gbv[6] = { gb.t.x, gb.t.y, gb.t.z, gb.w.x, gb.w.y, gb.w.z };   // gb itself stays the lane-partial gradient
      ODG_UNROLL for (int j = 0; j < NJL; j++) {
        float wl[6] = { W[j].t.x, W[j].t.y, W[j].t.z, W[j].w.x, W[j].w.y, W[j].w.z };
        ODG_UNROLL for (int i = 0; i < 6; i++) {
          ODG_UNROLL for (int k = 0; k <= i; k++) P[i][k] -= wl[i] * wl[k];
          gbv[i] -= wl[i] * y[j];
        }
      }
      float red[kRedVals];
      {
        int n = 0;
        ODG_UNROLL for (int i = 0; i < 6; i++) ODG_UNROLL for (int k = 0; k <= i; k++) red[n++] = P[i][k];
        ODG_UNROLL for (int i = 0; i < 6; i++) red[21 + i] = gbv[i];
        red[27] = 0.f;
      }
      grp_sum28(red, s_red, leg, gm);
      {
        int n = 0;
        ODG_UNROLL for (int i = 0; i < 6; i++) ODG_UNROLL for (int k = 0; k <= i; k++) S[i][k] = red[n++];
        ODG_UNROLL for (int i = 0; i < 6; i++) rhs[i] = -red[21 + i];
      }
    }
    chol6_solve(S, rhs);
    Vec6 p_b; p_b.t = mk3(rhs[0], rhs[1], rhs[2]); p_b.w = mk3(rhs[3], rhs[4], rhs[5]);
    float p_l[NJL];
    // back substitution: p_l = -L^-T (y + W p_b)
    ODG_UNROLL for (int j = NJL - 1; j >= 0; j--) {
      float u = -y[j] - dot6(W[j], p_b);
      ODG_UNROLL for (int i = j + 1; i < NJL; i++) u -= Hll[i][j] * p_l[i];
      p_l[j] = u * iL[j];
    }
    // ---- exact line search on phi(alpha) = cost(a + alpha p)  (convex, C1, piecewise quadratic)
    // lane-partials of the Gauss part: phi'_gauss(alpha) = G + alpha*Hq
    float G = dot6(gauss_b, p_b), Hq = 0.f;
    {
      Vec6 Mpb = Mbb_mul(p_b);
      Hq = l0f * dot6(Mpb, p_b);
      ODG_UNROLL for (int j = 0; j < NJL; j++) {
        float mlp = dot6(Mlb[j], p_b);
        G += p_l[j] * gauss_l[j];
        float s = 2.f * mlp;
        ODG_UNROLL for (int i = 0; i < NJL; i++) s += Mll[j][i] * p_l[i];
        Hq += p_l[j] * s;
      }
    }
    // the nine line-search coefficients of contact c for the direction whose row values are (dz, dza)
    auto line_coef = [&](int c, V3 dz, V3 dza) {
      const int s = kStash ? 0 : odg_float_bits(c_af[c].w);
      const float Dn = c_ra[c].w;
      if constexpr (kG) {
        const Cone6 K6 = cone6_make(Dn, C.impratio, C.slot_mu[s], C.slot_fri[s], C.slot_dmk[s], C.slot_frt[s], C.slot_frr[s],
                                    C.slot_dt_tor[s], C.slot_dt_roll[s], C.slot_condim[s]);
        const V3 zl = xyz(c_z0[c]), za = xyz(c_z0a[c]);
        const float z6[6] = { zl.x, zl.y, zl.z, za.x, za.y, za.z }, d6[6] = { dz.x, dz.y, dz.z, dza.x, dza.y, dza.z };
        return cone6_line_prep(z6, d6, K6);
      } else if constexpr (kStash) {
        const float mu = c_cj[c][0].w, fri = c_cj[c][1].w;
        return cone_line_prep(xyz(c_z0[c]), dz, Dn, fri != 0.f ? Dn * C.impratio : 0.f, mu, fri, c_af[c].w, 3);
      } else {
        return cone_line_prep(xyz(c_z0[c]), dz, Dn, Dn * C.impratio, C.slot_mu[s], C.slot_fri[s], C.slot_dmk[s], C.slot_condim[s]);
      }
    };
    ODG_NO_UNROLL for (int c = 0; c < nc; c++) {
      const int link = kStash ? 0 : C.slot_link[odg_float_bits(c_af[c].w)];
      const V3 r = xyz(c_ra[c]);
      V3 dz = cross_acc(p_b.t, p_b.w, r);
      ODG_UNROLL for (int j = 0; j < NJL; j++)       // (zero columns below the contact's link)
        dz = dz + p_l[j] * (FAT ? xyz(c_cj[c][j]) : ((j <= link) ? cross(ax[j], r - anc[j]) : mk3(0.f, 0.f, 0.f)));
      V3 dza = p_b.w;
      if constexpr (kG) {
        ODG_UNROLL for (int j = 0; j < NJL; j++) {
          const float on = fminf(fmaxf((float)(link - j + 1), 0.f), 1.f);
          dza = dza + (on * p_l[j]) * ax[j];
        }
      }
      if constexpr (FAT) {
        const LineCoef k = line_coef(c, dz, dza);
        float4 q;
        q.x = k.N0; q.y = k.Nd; q.z = k.cA; q.w = k.cB; c_lc[c][0] = q;
        q.x = k.cC; q.y = k.q1; q.z = k.q2; q.w = k.Dm; c_lc[c][1] = q;
        q.x = k.mu; q.y = 0.f; q.z = 0.f; q.w = 0.f; c_lc[c][2] = q;
      } else { c_dz[c] = mk4(dz, 0.f); if constexpr (kG) c_dza[c] = mk4(dza, 0.f); }
    }
    const float bf_zt = dot(bf_e, a_b.t) - bf_aref_t, bf_dzt = dot(bf_e, p_b.t);
    const float bf_zr = dot(bf_c, a_b.w) - bf_aref_r, bf_dzr = dot(bf_c, p_b.w);
    // phi'(0) = p . grad  (lane-partials of the trunk gradient were kept in gb)
    float d10 = dot6(gb, p_b);
    ODG_UNROLL for (int j = 0; j < NJL; j++) d10 += p_l[j] * g_l[j];
    // size of the full Newton step relative to the iterate: when it is already negligible this is the last iteration
    // and the step is taken without a line search
    float amax = 0.f, smax = 0.f;
    smax = fmaxf(fmaxf(fabsf(p_b.t.x), fabsf(p_b.t.y)), fmaxf(fabsf(p_b.t.z), fmaxf(fabsf(p_b.w.x), fmaxf(fabsf(p_b.w.y), fabsf(p_b.w.z)))));
    amax = fmaxf(fmaxf(fabsf(a_b.t.x), fabsf(a_b.t.y)), fmaxf(fabsf(a_b.t.z), fmaxf(fabsf(a_b.w.x), fmaxf(fabsf(a_b.w.y), fabsf(a_b.w.z)))));
    ODG_UNROLL for (int j = 0; j < NJL; j++) { smax = fmaxf(smax, fabsf(p_l[j])); amax = fmaxf(amax, fabsf(a_l[j])); }
    grp_sum_max2(d10, smax, amax, s_red, leg, gm);
    // phi'(alpha) at four step lengths at once (lane-partial sums, then one group reduction per value). The four
    // evaluations are independent, which gives the scheduler 4-way ILP in the kernel's hottest loop, and the
    // number of passes is fixed (<= C.ls_iters), so environments sharing a warp do not diverge here.
    constexpr int LW = ODG_LS_WIDTH;                // step lengths evaluated per trip through the row code
    auto evalw = [&](const float (&al)[LW], float (&f)[LW]) {
      ODG_UNROLL for (int k = 0; k < LW; k++) f[k] = G + al[k] * Hq;
      // friction-loss and limit rows, branch-free: a row that does not exist has fl = 0 / D = 0 and adds exactly 0
      ODG_UNROLL for (int j = 0; j < NJL; j++) {
        const float fl = LCF(LC_FL, j);
        {
          const float D = LCF(LC_DFL, j), z0 = a_l[j] - aref_fl[j], dz = p_l[j];
          ODG_UNROLL for (int k = 0; k < LW; k++) f[k] += fminf(fmaxf(D * (z0 + al[k] * dz), -fl), fl) * dz;
        }
        {
          const float dzl = lim_sgn[j] * p_l[j], z0 = lim_sgn[j] * a_l[j] - lim_aref[j], Dd = lim_D[j] * dzl;
          ODG_UNROLL for (int k = 0; k < LW; k++) f[k] += fminf(z0 + al[k] * dzl, 0.f) * Dd;
        }
      }
      ODG_UNROLL for (int k = 0; k < LW; k++) f[k] += fminf(fmaxf(bf_Dt * (bf_zt + al[k] * bf_dzt), -bf_ft), bf_ft) * bf_dzt;
      ODG_UNROLL for (int k = 0; k < LW; k++) f[k] += fminf(fmaxf(bf_Dr * (bf_zr + al[k] * bf_dzr), -bf_fr), bf_fr) * bf_dzr;
      ODG_NO_UNROLL for (int c = 0; c < nc; c++) {               // (a row with D = 0 adds exactly 0: no skip, no branch)
        if constexpr (FAT) {
          const float4 q0 = c_lc[c][0], q1 = c_lc[c][1], q2 = c_lc[c][2];
          LineCoef k;
          k.N0 = q0.x; k.Nd = q0.y; k.cA = q0.z; k.cB = q0.w; k.cC = q1.x; k.q1 = q1.y; k.q2 = q1.z; k.Dm = q1.w; k.mu = q2.x;
          cone_line_eval<LW>(k, al, f);
        } else {
          cone_line_eval<LW>(line_coef(c, xyz(c_dz[c]), kG ? xyz(c_dza[c]) : mk3(0.f, 0.f, 0.f)), al, f);
        }
      }
      ODG_UNROLL for (int k = 0; k < LW; k++) f[k] = grp_sum(f[k], gm);
    };
    auto eval4 = [&](const float (&al)[4], float (&f)[4]) {
      if (LW == 4) {
        float a4[LW], f4[LW];
        ODG_UNROLL for (int k = 0; k < LW; k++) a4[k] = al[k % 4];
        evalw(a4, f4);
        ODG_UNROLL for (int k = 0; k < LW; k++) f[k % 4] = f4[k];
      } else {
        // narrower row code run 4/LW times in a rolled loop: a smaller Newton-iteration body (instruction fetch is what
        // bounds this kernel) for less instruction-level parallelism
        ODG_NO_UNROLL for (int h = 0; h < 4 / LW; h++) {
          float aw[LW], fw[LW];
          ODG_UNROLL for (int k = 0; k < LW; k++) {
            aw[k] = al[k];
            ODG_UNROLL for (int g = 1; g < 4 / LW; g++) aw[k] = (h == g) ? al[(g * LW + k) % 4] : aw[k];
          }
          evalw(aw, fw);
          ODG_UNROLL for (int k = 0; k < LW; k++)
            ODG_UNROLL for (int g = 0; g < 4 / LW; g++) if (h == g) f[(g * LW + k) % 4] = fw[k];
        }
      }
    };
    const bool tiny = smax <= C.tol * (1.f + amax);
    float alpha = (tiny && d10 < 0.f) ? 1.f : 0.f;
#ifdef ODG_EMU_STATS
    const int ls_before = ls_evals;
#endif
    if (d10 < 0.f && !tiny) {                       // else: negligible step, or not a descent direction (converged to rounding)
      // phi' is increasing (phi convex): bracket its zero with the first pass, shrink the bracket 5x per further
      // pass, stop as soon as one evaluated point has |phi'| <= ls_tol*|phi'(0)|, else finish with the zero of the
      // chord on the last bracket
      const float ftol = C.ls_tol * fabsf(d10);
      float al[4] = { 0.25f, 0.5f, 1.f, 2.f }, f[4];
      float lo = 0.f, flo = d10, hi = -1.f, fhi = 0.f;
      bool done = false;
      ODG_NO_UNROLL for (int ls = 0; ls < C.ls_iters && !done; ls++) {
        {
          // further passes: 4 interior points of the bracket — or, while the zero lies below every step tried so far, a
          // geometric ladder, which resolves zeros that are orders of magnitude smaller than the Newton step (a stiff
          // row switching on right next to the iterate) in one pass. Selects, not branches.
          const bool first = ls == 0, ladder = lo == 0.f;
          const float w = (hi - lo) * 0.2f, lo0 = lo;
          const float lad[4] = { 0.008f, 0.04f, 0.2f, 0.6f };
          ODG_UNROLL for (int k = 0; k < 4; k++) {
            const float nxt = ladder ? lad[k] * hi : lo0 + w * (float)(k + 1);
            al[k] = first ? al[k] : nxt;
          }
        }
        eval4(al, f);
        ls_evals++;
        bool found = false;                         // a pass always starts without a new upper end
        ODG_UNROLL for (int k = 0; k < 4; k++) {
          const bool hit = !done && fabsf(f[k]) <= ftol;
          alpha = hit ? al[k] : alpha; done = done || hit;
          const bool up = !found && f[k] >= 0.f, dn = !found && !(f[k] >= 0.f);
          hi = up ? al[k] : hi; fhi = up ? f[k] : fhi;
          lo = dn ? al[k] : lo; flo = dn ? f[k] : flo;
          found = found || up;
        }
        {
          const bool run = !done && hi < 0.f;       // still descending at the largest step tried
          alpha = run ? al[3] : alpha; done = done || run;
        }
      }
      if (!done) {
        // zero of the chord — unless phi' is an order of magnitude smaller at the upper end: then a stiff row switches
        // on between lo and hi (phi' flat, then very steep), the chord lands on or before that kink, the next Hessian is
        // assembled without the row, and the iteration repeats the same tiny step until the cap (seen with Go1's feet,
        // D ~ 5e5). The upper end is past the kink and within the bracket width of the zero.
        alpha = lo - flo * odg_fdiv_fast(hi - lo, fhi - flo);
        alpha = (alpha >= lo && alpha <= hi) ? alpha : 0.5f * (lo + hi);
        alpha = (fhi < -0.1f * flo) ? hi : alpha;
      }
    }
#ifdef ODG_EMU_STATS
    if (lane0) odg_emu_stat(it, odg_fdiv_fast(smax, 1.f + amax), alpha, ls_evals - ls_before, nc, d10);
#endif
    // ---- take the step, test convergence on the step size
    a_b.t = a_b.t + alpha * p_b.t; a_b.w = a_b.w + alpha * p_b.w;
    ODG_UNROLL for (int j = 0; j < NJL; j++) a_l[j] += alpha * p_l[j];
    // converged: the full Newton step is negligible, or p is no longer a descent direction in fp32 (nothing left to
    // gain at this precision; without this exit such an environment idles until the iteration cap)
    conv = tiny || !(d10 < 0.f);
  }
  work += iters + ls_evals;
  // ------------------------------------------------------------------ outputs of the forward pass
  if (last) {
    out.a_b = a_b; ODG_UNROLL for (int j = 0; j < NJL; j++) out.a_l[j] = a_l[j];
    out.ncon = nc; out.iters = iters; out.ls_evals = ls_evals; out.R_last = R[NJL - 1];
    out.foot_contact = foot_last >= 0 ? 1 : 0;
    out.foot_force = mk3(0.f, 0.f, 0.f);
    if constexpr (kG) { ODG_UNROLL for (int q = 0; q <= NJL; q++) ODG_UNROLL for (int k = 0; k < 6; k++) out.cfrc[q][k] = 0.f; }
    float fn = 0.f;
    for (int c = 0; c < nc; c++) {
      const int s = kStash ? 0 : odg_float_bits(c_af[c].w);
      const int link = C.slot_link[s];
      const float Dn = c_ra[c].w;
      if (Dn == 0.f) continue;
      const V3 r = xyz(c_ra[c]);
      V3 ap = a_b.t + cross(a_b.w, r);
      ODG_UNROLL for (int j = 0; j < NJL; j++)
        ap = ap + a_l[j] * (FAT ? xyz(c_cj[c][j]) : ((j <= link) ? cross(ax[j], r - anc[j]) : mk3(0.f, 0.f, 0.f)));
      V3 g; S3 H;
      if constexpr (kG) {
        V3 alb = a_b.w;
        ODG_UNROLL for (int j = 0; j < NJL; j++) if (j <= link) alb = alb + a_l[j] * ax[j];
        const V3 zl = ap - xyz(c_af[c]), za = alb - xyz(c_arefa[c]);
        const Cone6 K6 = cone6_make(Dn, C.impratio, C.slot_mu[s], C.slot_fri[s], C.slot_dmk[s], C.slot_frt[s], C.slot_frr[s],
                                    C.slot_dt_tor[s], C.slot_dt_roll[s], C.slot_condim[s]);
        const float z6[6] = { zl.x, zl.y, zl.z, za.x, za.y, za.z };
        float g6[6], H6[6][6];
        cone6_eval(z6, K6, g6, H6);
        g = mk3(g6[0], g6[1], g6[2]);
        // wrench on the body: force -gL at the contact point, torque -gA; moved to the robot's centre of mass
        const V3 fw = -g, tw = mk3(-g6[3], -g6[4], -g6[5]);
        const V3 arm = r - odg_fdiv_rn(1.f, T.m) * T.h;
        const V3 tq = tw + cross(arm, fw);
        const int b = link < 0 ? NJL : link;
        ODG_UNROLL for (int q = 0; q <= NJL; q++) if (q == b) {
          out.cfrc[q][0] += tq.x; out.cfrc[q][1] += tq.y; out.cfrc[q][2] += tq.z;
          out.cfrc[q][3] += fw.x; out.cfrc[q][4] += fw.y; out.cfrc[q][5] += fw.z;
        }
      } else {
        if constexpr (kStash) {
          const float mu = c_cj[c][0].w, fri = c_cj[c][1].w;
          cone_eval(ap - xyz(c_af[c]), Dn, fri != 0.f ? Dn * C.impratio : 0.f, mu, fri, c_af[c].w, 3, g, H);
        } else {
          cone_eval(ap - xyz(c_af[c]), Dn, Dn * C.impratio, C.slot_mu[s], C.slot_fri[s], C.slot_dmk[s], C.slot_condim[s], g, H);
        }
      }
      fn += -g.z;
      if (c == foot_last) out.foot_force = mk3(-g.z, -g.y, g.x);   // MuJoCo frame: n=+z, t1=+y, t2=-x
    }
    out.fn = fn;
  }
  // ------------------------------------------------------------------ semi-implicit Euler (mj_Euler)
  const V3 acc_wl = tmul(R0, a_b.w);
  if (integrate) {
    const float h = C.h;
    Vec6 v_b = a_b; float v_l[NJL];                 // acceleration used for the velocity update
    ODG_UNROLL for (int j = 0; j < NJL; j++) v_l[j] = a_l[j];
    if (C.any_damping) {
      // mj_Euler with joint damping: solve (M + h*B) x = M*qacc (= qfrc_smooth + qfrc_constraint) and advance the
      // velocity with x. Same block-arrow elimination as the Newton system: leg block per lane, 6x6 Schur complement
      // on the trunk reduced over the group.
      Vec6 rb = Mbb_mul(a_b);
      rb.t = l0f * rb.t; rb.w = l0f * rb.w;
      float rl[NJL], A[NJL][NJL];
      ODG_UNROLL for (int j = 0; j < NJL; j++) {
        float s = dot6(Mlb[j], a_b);
        ODG_UNROLL for (int i = 0; i < NJL; i++) { s += Mll[j][i] * a_l[i]; A[j][i] = Mll[j][i]; }
        A[j][j] += h * LCF(LC_DAMP, j);
        rl[j] = s;
        rb.t = rb.t + a_l[j] * Mlb[j].t; rb.w = rb.w + a_l[j] * Mlb[j].w;
      }
      spd_inverse<NJL>(A);
      Vec6 W[NJL]; float y[NJL];
      ODG_UNROLL for (int j = 0; j < NJL; j++) {
        W[j].t = mk3(0.f, 0.f, 0.f); W[j].w = mk3(0.f, 0.f, 0.f); y[j] = 0.f;
        ODG_UNROLL for (int i = 0; i < NJL; i++) {
          W[j].t = W[j].t + A[j][i] * Mlb[i].t; W[j].w = W[j].w + A[j][i] * Mlb[i].w;
          y[j] += A[j][i] * rl[i];
        }
      }
      float P[6][6], S[6][6], rhs[6];
      ODG_UNROLL for (int i = 0; i < 6; i++) ODG_UNROLL for (int k = 0; k < 6; k++) P[i][k] = 0.f;
      P[0][0] = l0f * (T.m + C.base_arm_t[0]); P[1][1] = l0f * (T.m + C.base_arm_t[1]); P[2][2] = l0f * (T.m + C.base_arm_t[2]);
      P[3][3] = l0f * (T.I.xx + C.base_arm_r); P[4][3] = l0f * T.I.xy; P[5][3] = l0f * T.I.xz;
      P[4][4] = l0f * (T.I.yy + C.base_arm_r); P[5][4] = l0f * T.I.yz; P[5][5] = l0f * (T.I.zz + C.base_arm_r);
      P[3][1] = l0f * (-T.h.z); P[3][2] = l0f * (T.h.y);
      P[4][0] = l0f * (T.h.z);  P[4][2] = l0f * (-T.h.x);
      P[5][0] = l0f * (-T.h.y); P[5][1] = l0f * (T.h.x);
      float rbv[6] = { rb.t.x, rb.t.y, rb.t.z, rb.w.x, rb.w.y, rb.w.z };
      ODG_UNROLL for (int j = 0; j < NJL; j++) {
        float hl[6] = { Mlb[j].t.x, Mlb[j].t.y, Mlb[j].t.z, Mlb[j].w.x, Mlb[j].w.y, Mlb[j].w.z };
        float wl[6] = { W[j].t.x, W[j].t.y, W[j].t.z, W[j].w.x, W[j].w.y, W[j].w.z };
        ODG_UNROLL for (int i = 0; i < 6; i++) {
          ODG_UNROLL for (int k = 0; k <= i; k++) P[i][k] -= hl[i] * wl[k];
          rbv[i] -= hl[i] * y[j];
        }
      }
      ODG_UNROLL for (int i = 0; i < 6; i++) {
        ODG_UNROLL for (int k = 0; k <= i; k++) S[i][k] = grp_sum(P[i][k], gm);
        rhs[i] = grp_sum(rbv[i], gm);
      }
      chol6_solve(S, rhs);
      v_b.t = mk3(rhs[0], rhs[1], rhs[2]); v_b.w = mk3(rhs[3], rhs[4], rhs[5]);
      ODG_UNROLL for (int j = 0; j < NJL; j++) v_l[j] = y[j] - dot6(W[j], v_b);
    }
    bv = bv + h * v_b.t;
    bwl = bwl + h * tmul(R0, v_b.w);
    ODG_UNROLL for (int j = 0; j < NJL; j++) { qd[j] += h * v_l[j]; q[j] += h * qd[j]; }
    bp = bp + h * bv;
    float wn = sqrtf(dot(bwl, bwl));
    if (wn > 1e-15f) {
      float s, c; sincosf(0.5f * h * wn, &s, &c);
      float k = s / wn;
      float dw = c, dx = k * bwl.x, dy = k * bwl.y, dz = k * bwl.z;
      float w = bq[0], x = bq[1], y = bq[2], z = bq[3];
      float nw = w * dw - x * dx - y * dy - z * dz;
      float nx = w * dx + x * dw + y * dz - z * dy;
      float ny = w * dy - x * dz + y * dw + z * dx;
      float nz = w * dz + x * dy - y * dx + z * dw;
      float in = odg_rsqrt(nw * nw + nx * nx + ny * ny + nz * nz);
      bq[0] = nw * in; bq[1] = nx * in; bq[2] = ny * in; bq[3] = nz * in;
    }
  }
  warm_v = a_b.t; warm_wl = acc_wl;
  ODG_UNROLL for (int j = 0; j < NJL; j++) warm_l[j] = a_l[j];
}

// reward_calc:372-390 in double
ODG_DEV void euler_from_quat(double w, double x, double y, double z, double& roll, double& pitch, double& yaw) {
  double t0 = 2.0 * (w * x + y * z), t1 = 1.0 - 2.0 * (x * x + y * y);
  roll = atan2(t0, t1);
  double t2 = 2.0 * (w * y - z * x);
  t2 = t2 > 1.0 ? 1.0 : t2; t2 = t2 < -1.0 ? -1.0 : t2;
  pitch = asin(t2);
  double t3 = 2.0 * (w * z + x * y), t4 = 1.0 - 2.0 * (y * y + z * z);
  yaw = atan2(t3, t4);
}

// get_projected_gravity (walk_environment_reward_calc.py / landing_environment_reward_calc.py:88-98): the reference's
// formula, not a rotation of g: with e = (roll, pitch, yaw), v = (g . e) e, returned normalised unless |v| == 0.
ODG_DEV void projected_gravity(const DevConst& C, const float (&quat)[4], float (&pg)[3]) {
  double e[3];
  euler_from_quat((double)quat[0], (double)quat[1], (double)quat[2], (double)quat[3], e[0], e[1], e[2]);
  const double d = (double)C.gx * e[0] + (double)C.gy * e[1] + (double)C.gz * e[2];
  const double v0 = d * e[0], v1 = d * e[1], v2 = d * e[2];
  const double n = sqrt(v0 * v0 + v1 * v1 + v2 * v2);
  pg[0] = (float)(n == 0.0 ? v0 : v0 / n); pg[1] = (float)(n == 0.0 ? v1 : v1 / n); pg[2] = (float)(n == 0.0 ? v2 : v2 / n);
}

// diagonal_gait_reward (reward_calc:203-234); pattern table :54-63, order FL FR BL BR = legs 0..3
ODG_DEV int gait_call(int& idx, int& cnt, int paws_mask, float vx) {
  const unsigned char pat[8] = { 0xF, 0xB, 0x9, 0xD, 0xF, 0x7, 0x6, 0xF };   // bit l = leg l on the ground
  bool match = (paws_mask == (int)pat[idx]) && (vx >= 0.5f);
  if (match) { cnt += 8; idx = (idx + 1) & 7; return cnt; }
  cnt = 0; idx = 0; return 0;
}

// What a caller that keeps stepping the same environment inside one kernel (MPPI rollouts) needs back from env_step.
struct StepResult { float reward_unclipped; bool terminated, truncated; };

// Full environment step for one 4-lane group: load state, frame_skip substeps, obs/reward/termination,
// optional auto-reset, store state.
template <int NJL, bool FAT>
ODG_DEV StepResult env_step(const DevConst& C, const float* ODG_RESTRICT s_lc, const float* ODG_RESTRICT s_gc,
                            const float4* ODG_RESTRICT s_vert, const SimPtrs& P, const StepArgs& A,
                            const float* action, int env, int leg, unsigned gm, float* ODG_RESTRICT s_red) {
  const int N = P.N;
  const bool real = env < P.n;                     // padding environments never touch caller-owned buffers
  const int obs_dim = C.obs_dim;
  constexpr bool kG = (NJL == 3);
  const bool jump = kG && C.task == 1;             // JumpEnvironmentV0 (environments/JumpEnvironment.py) on the Go1 model
  // ---- load
  V3 bp = mk3(P.qpos[0 * N + env], P.qpos[1 * N + env], P.qpos[2 * N + env]);
  float bq[4] = { P.qpos[3 * N + env], P.qpos[4 * N + env], P.qpos[5 * N + env], P.qpos[6 * N + env] };
  V3 bv = mk3(P.qvel[0 * N + env], P.qvel[1 * N + env], P.qvel[2 * N + env]);
  V3 bwl = mk3(P.qvel[3 * N + env], P.qvel[4 * N + env], P.qvel[5 * N + env]);
  V3 warm_v = mk3(P.warm[0 * N + env], P.warm[1 * N + env], P.warm[2 * N + env]);
  V3 warm_wl = mk3(P.warm[3 * N + env], P.warm[4 * N + env], P.warm[5 * N + env]);
  float q[NJL], qd[NJL], warm_l[NJL], ctrl[NJL], prev_act[NJL];
  ODG_UNROLL for (int j = 0; j < NJL; j++) {
    q[j] = P.qpos[(7 + leg * NJL + j) * N + env];
    qd[j] = P.qvel[(6 + leg * NJL + j) * N + env];
    warm_l[j] = P.warm[(6 + leg * NJL + j) * N + env];
    const int u = (int)LCF(LC_UIDX, j);
    float a = (LCF(LC_HASACT, j) != 0.f && real) ? action[env * C.nu + u] : 0.f;
    if (C.scale_actions && A.mode == 0) {
      // ScaleActionEnvironment.py:21-23 in float32, numpy evaluation order
      float lo = LCF(LC_SLO, j), hi = LCF(LC_SHI, j);
      a = odg_fadd_rn(lo, odg_fdiv_rn(odg_fmul_rn(odg_fadd_rn(a, 1.0f), odg_fsub_rn(hi, lo)), 2.0f));
    }
    ctrl[j] = a;
    prev_act[j] = LCF(LC_HASACT, j) != 0.f ? P.last_action[u * N + env] : 0.f;
  }
  int step = P.step[env], gidx = P.gait_idx[env], gcnt = P.gait_cnt[env];
  const bool fresh = P.fresh[env] != 0;
  const V3 desvel = mk3(P.desvel[0 * N + env], P.desvel[1 * N + env], P.desvel[2 * N + env]);

  // ---- physics
  LastPass<NJL> lp;
  int work = 0;
  {
    // mode 0: frame_skip x mj_step; mode 1 (odg_evaluate): one mj_forward, no integration. One call site, so the
    // (large) substep body exists once in the kernel.
    const bool stepping = A.mode == 0;
    const int nsub = stepping ? C.frame_skip : 1;
    if (stepping) step += 1;
    // Warm start of substep s >= 2: linear extrapolation of the previous two solutions (2*a[s-1] - a[s-2]) instead of
    // MuJoCo's plain a[s-1]. Only the starting point of the Newton iteration changes (-8 % iterations + line-search
    // passes on the bench workload); the solution it converges to does not.
    V3 pv = warm_v, pw = warm_wl; float pl[NJL];
    ODG_UNROLL for (int j = 0; j < NJL; j++) pl[j] = warm_l[j];
    for (int s = 0; s < nsub; s++) {
      {
      const V3 ov = warm_v, ow = warm_wl; float ol[NJL];
      ODG_UNROLL for (int j = 0; j < NJL; j++) ol[j] = warm_l[j];
      if (s >= 2) {                                 // (in every launch shape, lockstep or not, so that a result never depends
                                                    //  on the shape: measured +4 % free-running, -2 % under lockstep)
        warm_v = warm_v + (warm_v - pv); warm_wl = warm_wl + (warm_wl - pw);
        ODG_UNROLL for (int j = 0; j < NJL; j++) warm_l[j] += warm_l[j] - pl[j];
      }
      pv = ov; pw = ow;
      ODG_UNROLL for (int j = 0; j < NJL; j++) pl[j] = ol[j];
      }
      substep<NJL, FAT>(C, s_lc, s_gc, s_vert, leg, gm, bp, bq, bv, bwl, q, qd, ctrl, warm_v, warm_wl, warm_l,
                        stepping, s == nsub - 1, lp, work, s_red);
    }
  }

  // ---- observation (WalkEnvironment.py:115-136), float32
  float* obs = (A.obs && real) ? A.obs + (size_t)env * obs_dim : nullptr;
  float* tobs = (A.terminal_obs && A.mode == 0 && real) ? A.terminal_obs + (size_t)env * obs_dim : nullptr;
  auto clip = [](float v) { return fminf(100.f, fmaxf(-100.f, v)); };
  const int ob = C.obs_layout ? 12 : 9;           // first joint entry (OdgEnvConfig::obs_layout)
  auto write_obs = [&](float* o, V3 v, V3 wl, const float (&quat)[4], const float (&qq)[NJL], const float (&qqd)[NJL],
                       const float (&la)[NJL]) {
    if (!o) return;
    if (jump) {
      // JumpEnvironment.py:95-117: [0.3 - x, 0.3 - z, v (3), v_z, projected_gravity (3), utils.last_action (12)], all
      // scales 1. utils.last_action is never written by the environment (it stores self._last_action instead), so the
      // last 12 entries are the zeros of its constructor.
      if (leg == 0) {
        o[0] = clip(0.3f - bp.x); o[1] = clip(0.3f - bp.z);
        o[2] = clip(v.x); o[3] = clip(v.y); o[4] = clip(v.z); o[5] = clip(v.z);
        float pg[3]; projected_gravity(C, quat, pg); o[6] = pg[0]; o[7] = pg[1]; o[8] = pg[2];
      }
      ODG_UNROLL for (int j = 0; j < NJL; j++) o[9 + leg * NJL + j] = 0.f;
      return;
    }
    if (leg == 0) {
      o[0] = clip(v.x * 2.0f); o[1] = clip(v.y * 2.0f); o[2] = clip(v.z * 2.0f);
      o[3] = clip(wl.x * 0.25f); o[4] = clip(wl.y * 0.25f); o[5] = clip(wl.z * 0.25f);
      if (C.obs_layout) { float pg[3]; projected_gravity(C, quat, pg); o[6] = pg[0]; o[7] = pg[1]; o[8] = pg[2]; }
      o[ob - 3] = clip(desvel.x * 2.0f); o[ob - 2] = clip(desvel.y * 2.0f); o[ob - 1] = clip(desvel.z * 2.0f);
    }
    ODG_UNROLL for (int j = 0; j < NJL; j++) {
      o[ob + leg * NJL + j] = clip(qq[j] - (C.obs_layout ? LCF(LC_HOMEQ, j) : C.obs_joint_offset));
      o[ob + C.nu + leg * NJL + j] = clip(qqd[j] * 0.05f);
      if (LCF(LC_HASACT, j) != 0.f) o[ob + 2 * C.nu + (int)LCF(LC_UIDX, j)] = clip(la[j]);
    }
  };
  write_obs(obs, bv, bwl, bq, q, qd, prev_act);
  if (tobs) write_obs(tobs, bv, bwl, bq, q, qd, prev_act);

  // ---- reward / termination (WalkEnvironment.py:81-109, reward_calc.py), double where the reference is
  const double lim = 15.0 * 3.14159265358979323846 / 180.0;
  bool finite = isfinite(bp.x) && isfinite(bp.y) && isfinite(bp.z) && isfinite(bq[0]) && isfinite(bq[1]) &&
                isfinite(bq[2]) && isfinite(bq[3]) && isfinite(bv.x) && isfinite(bv.y) && isfinite(bv.z) &&
                isfinite(bwl.x) && isfinite(bwl.y) && isfinite(bwl.z);
  float fin_l = 1.f;
  ODG_UNROLL for (int j = 0; j < NJL; j++) fin_l = (isfinite(q[j]) && isfinite(qd[j])) ? fin_l : 0.f;
  finite = finite && (grp_sum(fin_l, gm) == 4.f);
  double lin = 0.0;
  if (bp.x > 0.f) {
    double ex = (double)desvel.x - (double)bv.x, ey = (double)desvel.y - (double)bv.y;
    lin = exp(-(ex * ex + ey * ey) / 0.25);
  }
  double roll = 0, pitch = 0, yaw = 0, safe = 0;
  if (finite) {
    euler_from_quat((double)bq[0], (double)bq[1], (double)bq[2], (double)bq[3], roll, pitch, yaw);
    double dr = !(fabs(roll) > lim) ? lim - fabs(roll) : 0.0;
    double dp = !(fabs(pitch) > lim) ? lim - fabs(pitch) : 0.0;
    double dy = !(fabs(yaw) > lim) ? lim - fabs(yaw) : 0.0;
    safe = (dr + dp + dy) / (0.110 + lim + lim + lim);
  }
  // paws_in_ground bitmask, bit l = leg l (FL FR BL BR)
  int paws;
  {
    float bit = lp.foot_contact ? (float)(1 << leg) : 0.f;
    paws = (int)grp_sum(bit, gm);
  }
  const int gait = gait_call(gidx, gcnt, paws, bv.x);
  const double rewards = lin * 1.5 + safe * .015 + (double)gait * 3;
  // costs: joint deviation (double, numpy pairwise order), action rate (float32 unless fresh), |y|
  double jc = 0.0; float rate_f = 0.f; double rate_d = 0.0;
  {
    double s = 0.0; float sf = 0.f; double sd = 0.0;
    ODG_UNROLL for (int j = 0; j < NJL; j++) {
      double t = (double)q[j] - (double)C.key_ctrl[leg * NJL + j];
      s += t * t;
      if (LCF(LC_HASACT, j) != 0.f) {
        float d = odg_fsub_rn(prev_act[j], ctrl[j]);
        sf = odg_fadd_rn(sf, odg_fmul_rn(d, d));
        double dd = 0.0 - (double)ctrl[j];
        sd += dd * dd;
      }
    }
    // numpy pairwise order over joints (body order): ((l0)+(l1)) + ((l2)+(l3)); IEEE + is commutative
    double s2 = s + grp_xor_d(s, 1, gm);
    jc = s2 + grp_xor_d(s2, 2, gm);
    // actuator order FR BR FL BL: ((l1)+(l3)) + ((l0)+(l2)): xor 2 first, then xor 1
    float t2 = odg_fadd_rn(sf, grp_xor(sf, 2, gm));
    rate_f = odg_fadd_rn(t2, grp_xor(t2, 1, gm));
    double sd2 = sd + grp_xor_d(sd, 2, gm);
    rate_d = sd2 + grp_xor_d(sd2, 1, gm);
  }
  const double rate = fresh ? rate_d : (double)rate_f;
  const double ycost = fabs((double)bp.y);
  const double costs = jc * 0.1 + rate * 0.01 + ycost;
  double rr = rewards - costs;
  const bool healthy = finite && (-lim < roll && roll < lim) && (-lim < pitch && pitch < lim) && (-lim < yaw && yaw < lim);
  bool terminated = !healthy;
  const bool truncated = step >= C.max_steps;
  if constexpr (kG) {
    if (jump) {
      // JumpEnvironmentRewardCalc.compute_rewards (rewards/jump_environment_reward_calc.py:55-150), in double like the
      // reference, term by term in its order of evaluation; static_stability (:140-150) for termination.
      float c2 = 0.f;                                // ||cfrc_ext[[2,3,5,6,8,9,11,12]]||_F^2: hips and thighs of all legs
      ODG_UNROLL for (int b = 0; b < 2; b++) ODG_UNROLL for (int k = 0; k < 6; k++) c2 += lp.cfrc[b][k] * lp.cfrc[b][k];
      c2 = grp_sum(c2, gm);
      const double x = (double)bp.x, y = (double)bp.y, z = (double)bp.z;
      const double dx = 1.0 - x, dy = 0.0 - y;
      const double dist = sqrt(dx * dx + dy * dy);
      const double cube_h = 0.5;
      const double t_lp = (z >= cube_h ? exp(-dist) : 0.0) * 3.0;
      double jr = 0, jp = 0, jy = 0;
      if (finite) euler_from_quat((double)bq[0], (double)bq[1], (double)bq[2], (double)bq[3], jr, jp, jy);
      const double t_lo = exp(-(fabs(jr) + fabs(jp) + fabs(jy))) * 2.0;
      const double vx = (double)bv.x, vy = (double)bv.y, vz = (double)bv.z;
      const double t_cv = exp(-sqrt(vx * vx + vy * vy)) * 1.0;
      const double t_hc = (z - cube_h > 0.0 ? z - cube_h : 0.0) * .2;
      const double t_ps = -0.0 * 0.8;                // feet_air_time is never advanced by this calculator
      const double e0 = (double)desvel.x - vx, e1 = (double)desvel.y - vy, e2 = (double)desvel.z - vz;
      const double t_jv = exp(-((e0 * e0 + e1 * e1) + e2 * e2) / 0.45) * 1.0;
      const double jrew = ((((t_lp + t_lo) + t_cv) + t_hc) + t_ps) + t_jv;
      const double t_dl = (z < cube_h ? exp(dist) : 0.0) * 2.0;
      const double t_vv = (z >= cube_h ? vz * vz : 0.0) * 1.5;
      const double t_ob = (dist > 1.0 ? 1.0 : 0.0) * 3.0;
      const double t_cc = (sqrtf(c2) > 0.1f ? 1.0 : 0.0) * 1.0;
      const double jcost = ((t_dl + t_vv) + t_ob) + t_cc;
      rr = jrew - jcost;
      const double l20 = 20.0 * 3.14159265358979323846 / 180.0;
      terminated = !(finite && (-l20 <= jy && jy <= l20) && (-l20 <= jr && jr <= l20));
      if (A.want_info && A.task_terms && real && leg == 0) {
        float* o = A.task_terms + (size_t)env * 10;
        o[0] = (float)t_lp; o[1] = (float)t_lo; o[2] = (float)t_cv; o[3] = (float)t_hc; o[4] = (float)t_ps;
        o[5] = (float)t_jv; o[6] = (float)t_dl; o[7] = (float)t_vv; o[8] = (float)t_ob; o[9] = (float)t_cc;
      }
    }
    if (A.want_info && A.cfrc_ext && real) {
      // body order of the MuJoCo model: trunk, then (hip, thigh, calf) per leg; the trunk row sums the four lanes' shares
      float* o = A.cfrc_ext + (size_t)env * (1 + 4 * NJL) * 6;
      ODG_UNROLL for (int b = 0; b < NJL; b++) ODG_UNROLL for (int k = 0; k < 6; k++) o[(1 + leg * NJL + b) * 6 + k] = lp.cfrc[b][k];
      ODG_UNROLL for (int k = 0; k < 6; k++) { const float t = grp_sum(lp.cfrc[NJL][k], gm); if (leg == 0) o[k] = t; }
    }
  }
  const float reward = (float)(rr > 0.0 ? rr : 0.0);
  // ---- info
  if (A.want_info && real) {
    if (A.paw_forces) {
      // reward_calc:339-349,361-365: (R_c @ f) then R_calf^T
      V3 f = lp.foot_force;                        // (fn, ft1, ft2)
      V3 fg = mk3(f.z, f.y, -f.x);
      V3 fb = lp.foot_contact ? tmul(lp.R_last, fg) : mk3(0.f, 0.f, 0.f);
      float* o = A.paw_forces + ((size_t)env * 4 + leg) * 6;
      o[0] = fb.x; o[1] = fb.y; o[2] = fb.z; o[3] = 0.f; o[4] = 0.f; o[5] = 0.f;
    }
    if (A.paws_in_ground) A.paws_in_ground[(size_t)env * 4 + leg] = (unsigned char)lp.foot_contact;
    float tq = 0.f;
    ODG_UNROLL for (int j = 0; j < NJL; j++) tq += lp.act[j] * lp.act[j];
    tq = grp_sum(tq, gm);
    float fn = grp_sum(lp.fn, gm);
    float ncs = grp_sum((float)lp.ncon, gm);
    if (A.qacc) {
      ODG_UNROLL for (int j = 0; j < NJL; j++) A.qacc[(size_t)env * C.nv + 6 + leg * NJL + j] = lp.a_l[j];
    }
    if (leg == 0) {
      if (A.x_position) A.x_position[env] = bp.x;
      if (A.y_position) A.y_position[env] = bp.y;
      if (A.distance) A.distance[env] = sqrtf(bp.x * bp.x + bp.y * bp.y);
      if (A.lin_vel_reward) A.lin_vel_reward[env] = (float)lin;
      if (A.reward_ctrl) A.reward_ctrl[env] = tq;
      if (A.gait_reward) A.gait_reward[env] = gait;
      if (A.ncon) A.ncon[env] = (int)ncs;
      if (A.fn_sum) A.fn_sum[env] = fn;
      if (A.solver_iters) A.solver_iters[env] = lp.iters;
      if (A.ls_evals) A.ls_evals[env] = lp.ls_evals;
      if (A.reward_raw) A.reward_raw[env] = (float)rr;
      if (A.qacc) {
        float* o = A.qacc + (size_t)env * C.nv;
        o[0] = lp.a_b.t.x; o[1] = lp.a_b.t.y; o[2] = lp.a_b.t.z;
        o[3] = warm_wl.x; o[4] = warm_wl.y; o[5] = warm_wl.z;     // trunk-frame angular acceleration
      }
    }
  }
  // second diagonal_gait_reward call (info["patterns_matches"], WalkEnvironment.py:70; quirk C2)
  const int gait2 = gait_call(gidx, gcnt, paws, bv.x);
  if (leg == 0 && real) {
    if (A.want_info && A.patterns_matches) A.patterns_matches[env] = (float)gait2;
    if (A.reward) A.reward[env] = reward;
    if (A.terminated) A.terminated[env] = terminated ? 1 : 0;
    if (A.truncated) A.truncated[env] = truncated ? 1 : 0;
  }
  // ---- auto-reset (SB3 worker) or plain state write-back
  bool is_fresh = false;
  float last_act[NJL];
  ODG_UNROLL for (int j = 0; j < NJL; j++) last_act[j] = ctrl[j];          // set_last_action(action)
  unsigned episode = 0;
  const bool do_reset = (A.mode == 0) && C.auto_reset && (terminated || truncated);
  if (do_reset) {
    episode = P.episode[env];
    grp_sync(gm);                                  // all lanes read the counter before lane 0 bumps it
    const uint32_t gid = (uint32_t)(C.first_env_id + env);
    float key_noise[kMaxNQ];
    for (int blk = 0; blk * 4 < C.nq; blk++) {
      uint32_t r[4];
      philox4x32(C.seed_lo, C.seed_hi, gid, episode, (uint32_t)blk, kStreamReset, r);
      for (int k = 0; k < 4; k++) if (blk * 4 + k < kMaxNQ) {
        float u = u01(r[k]);
        float nz = odg_fadd_rn(-C.noise, odg_fmul_rn(2.0f * C.noise, u));
        key_noise[blk * 4 + k] = (blk * 4 + k < C.nq) ? odg_fadd_rn(C.key_qpos[blk * 4 + k], nz) : 0.f;
      }
    }
    bp = mk3(key_noise[0], key_noise[1], key_noise[2]);
    bq[0] = key_noise[3]; bq[1] = key_noise[4]; bq[2] = key_noise[5]; bq[3] = key_noise[6];
    bv = mk3(0.f, 0.f, 0.f); bwl = mk3(0.f, 0.f, 0.f);
    warm_v = mk3(0.f, 0.f, 0.f); warm_wl = mk3(0.f, 0.f, 0.f);
    ODG_UNROLL for (int j = 0; j < NJL; j++) {
      float v = 0.f;
      for (int k = 0; k < kMaxNQ; k++) if (k == 7 + leg * NJL + j) v = key_noise[k];
      q[j] = v; qd[j] = 0.f; warm_l[j] = 0.f; last_act[j] = 0.f;
    }
    step = 0; is_fresh = true; episode += 1;
    write_obs(obs, bv, bwl, bq, q, qd, last_act);
  }
  // ---- store
  ODG_UNROLL for (int j = 0; j < NJL; j++) {
    P.qpos[(7 + leg * NJL + j) * N + env] = q[j];
    P.qvel[(6 + leg * NJL + j) * N + env] = qd[j];
    P.warm[(6 + leg * NJL + j) * N + env] = warm_l[j];
    if (LCF(LC_HASACT, j) != 0.f && A.mode == 0) P.last_action[(int)LCF(LC_UIDX, j) * N + env] = last_act[j];
  }
  if (leg == 0) {
    P.qpos[0 * N + env] = bp.x; P.qpos[1 * N + env] = bp.y; P.qpos[2 * N + env] = bp.z;
    P.qpos[3 * N + env] = bq[0]; P.qpos[4 * N + env] = bq[1]; P.qpos[5 * N + env] = bq[2]; P.qpos[6 * N + env] = bq[3];
    P.qvel[0 * N + env] = bv.x; P.qvel[1 * N + env] = bv.y; P.qvel[2 * N + env] = bv.z;
    P.qvel[3 * N + env] = bwl.x; P.qvel[4 * N + env] = bwl.y; P.qvel[5 * N + env] = bwl.z;
    P.warm[0 * N + env] = warm_v.x; P.warm[1 * N + env] = warm_v.y; P.warm[2 * N + env] = warm_v.z;
    P.warm[3 * N + env] = warm_wl.x; P.warm[4 * N + env] = warm_wl.y; P.warm[5 * N + env] = warm_wl.z;
    P.gait_idx[env] = gidx; P.gait_cnt[env] = gcnt;
    if (P.work) P.work[env] = work;
    if (A.mode == 0) { P.step[env] = step; P.fresh[env] = is_fresh ? 1 : 0; }
    if (do_reset) P.episode[env] = episode;
  }
  StepResult res; res.reward_unclipped = (float)rr; res.terminated = terminated; res.truncated = truncated;
  return res;
}

// reset_model (WalkEnvironment.py:138-151) for one 4-lane group
template <int NJL>
ODG_DEV void env_reset(const DevConst& C, const float* ODG_RESTRICT s_lc, const SimPtrs& P, float* obs_out,
                       int env, int leg, unsigned gm) {
  const int N = P.N;
  const int obs_dim = C.obs_dim;
  const bool jump = (NJL == 3) && C.task == 1;
  const unsigned episode = P.episode[env];
  grp_sync(gm);                                    // all lanes read the counter before lane 0 bumps it
  const uint32_t gid = (uint32_t)(C.first_env_id + env);
  float kq[kMaxNQ];
  for (int blk = 0; blk * 4 < C.nq; blk++) {
    uint32_t r[4];
    philox4x32(C.seed_lo, C.seed_hi, gid, episode, (uint32_t)blk, kStreamReset, r);
    for (int k = 0; k < 4; k++) if (blk * 4 + k < kMaxNQ) {
      float u = u01(r[k]);
      float nz = odg_fadd_rn(-C.noise, odg_fmul_rn(2.0f * C.noise, u));
      kq[blk * 4 + k] = (blk * 4 + k < C.nq) ? odg_fadd_rn(C.key_qpos[blk * 4 + k], nz) : 0.f;
    }
  }
  float* obs = (obs_out && env < P.n) ? obs_out + (size_t)env * obs_dim : nullptr;
  auto clip = [](float v) { return fminf(100.f, fmaxf(-100.f, v)); };
  const int ob = C.obs_layout ? 12 : 9;
  for (int j = 0; j < NJL; j++) {
    const int qi = 7 + leg * NJL + j;
    P.qpos[qi * N + env] = kq[qi];
    P.qvel[(6 + leg * NJL + j) * N + env] = 0.f;
    P.warm[(6 + leg * NJL + j) * N + env] = 0.f;
    if (LCF(LC_HASACT, j) != 0.f) P.last_action[(int)LCF(LC_UIDX, j) * N + env] = 0.f;
    if (obs && jump) obs[9 + leg * NJL + j] = 0.f;
    else if (obs) {
      obs[ob + leg * NJL + j] = clip(kq[qi] - (C.obs_layout ? LCF(LC_HOMEQ, j) : C.obs_joint_offset));
      obs[ob + C.nu + leg * NJL + j] = 0.f;
      if (LCF(LC_HASACT, j) != 0.f) obs[ob + 2 * C.nu + (int)LCF(LC_UIDX, j)] = 0.f;
    }
  }
  if (leg == 0) {
    for (int i = 0; i < 7; i++) P.qpos[i * N + env] = kq[i];
    for (int i = 0; i < 6; i++) { P.qvel[i * N + env] = 0.f; P.warm[i * N + env] = 0.f; }
    P.step[env] = 0; P.fresh[env] = 1; P.episode[env] = episode + 1;
    if (obs && jump) {                               // JumpEnvironment.py:95-117 at zero velocity
      obs[0] = clip(0.3f - kq[0]); obs[1] = clip(0.3f - kq[2]);
      for (int i = 2; i < 6; i++) obs[i] = 0.f;
      const float quat[4] = { kq[3], kq[4], kq[5], kq[6] };
      float pg[3]; projected_gravity(C, quat, pg);
      for (int i = 0; i < 3; i++) obs[6 + i] = pg[i];
    } else if (obs) {
      for (int i = 0; i < 6; i++) obs[i] = 0.f;
      if (C.obs_layout) {
        const float quat[4] = { kq[3], kq[4], kq[5], kq[6] };
        float pg[3]; projected_gravity(C, quat, pg);
        for (int i = 0; i < 3; i++) obs[6 + i] = pg[i];
      }
      for (int i = 0; i < 3; i++) obs[ob - 3 + i] = clip(P.desvel[i * N + env] * 2.0f);
    }
  }
}

// Construction-time state of one environment (single lane): noise-free home keyframe, zero
// velocities, and the desired velocity sampled once (reward_calc:75,301-305: x ~ U[0.5, 1.0], y = z = 0).
ODG_DEV void env_init(const DevConst& C, const SimPtrs& P, int env) {
  const int N = P.N;
  for (int i = 0; i < C.nq; i++) P.qpos[i * N + env] = C.key_qpos[i];
  for (int i = 0; i < C.nv; i++) { P.qvel[i * N + env] = 0.f; P.warm[i * N + env] = 0.f; }
  for (int u = 0; u < C.nu; u++) P.last_action[u * N + env] = 0.f;
  uint32_t r[4];
  philox4x32(C.seed_lo, C.seed_hi, (uint32_t)(C.first_env_id + env), 0u, 0u, kStreamDesvel, r);
  if (C.task == 1) {      // jump_environment_reward_calc.py:33-35: U([1.20, -0, 1.20], [1.25, 0, 1.25]), sampled once
    P.desvel[0 * N + env] = odg_fadd_rn(1.20f, odg_fmul_rn(0.05f, u01(r[0])));
    P.desvel[1 * N + env] = 0.f;
    P.desvel[2 * N + env] = odg_fadd_rn(1.20f, odg_fmul_rn(0.05f, u01(r[1])));
  } else {
    P.desvel[0 * N + env] = odg_fadd_rn(0.5f, odg_fmul_rn(0.5f, u01(r[0])));
    P.desvel[1 * N + env] = 0.f; P.desvel[2 * N + env] = 0.f;
  }
  P.step[env] = 0; P.gait_idx[env] = 0; P.gait_cnt[env] = 0; P.episode[env] = 0u; P.fresh[env] = 1;
}

#undef LCF
#undef GCF

}  // namespace odg
