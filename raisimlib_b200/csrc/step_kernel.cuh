// Fused World::integrate() for a batch of environments -- hand-written sm_100a CUDA.
//
// One warp == one environment (BASELINE.json north_star).  A CTA of WPC warps shares the model
// constant block, staged global -> shared ONCE per CTA by a TMA bulk copy (cp.async.bulk +
// mbarrier; SASS: UBLKCP).  Every per-environment intermediate (body poses, M / its Cholesky
// factor, contact Jacobians, Delassus matrix) lives in that warp's shared-memory workspace; HBM is
// touched only for the coalesced state rows in, state rows + contact records out.
//
// Stages (SURVEY.md section 8a rows a2..a10, same math as oracle/rbd_oracle.hpp):
//   A  lane = body   : FK + RNEA forward walk down each body's own ancestor chain (registers),
//                      per-body force / composite-inertia terms, subtree sums by warp shuffles
//                      -> h, M (CRBA in a world-aligned frame centred on the base)
//   B  lane = point  : candidate point vs Ground / HeightMap, ballot-compacted contact list
//   C  lane = entry / column : b, Mhat = M + dt Kd + dt^2 Kp, branch-sparse Mhat = L^T L (Featherstone RBDA
//                      6.5) in compact-by-depth storage, z = L^-T b, Y = L^-T J^T (only the contact's own
//                      ancestor chain is touched), G = Y^T Y (sum up to the LCA depth)
//   D  lane = row    : per-contact Gauss-Seidel; slip by a 32-way section search (all lanes probe)
//   E  lane = dof    : v+ = v + L^-1 (dt z + Y lam), q+ = q (+) dt v+
//
// Compact-by-depth storage: the ancestors of a dof have distinct depths 0..d, so row i of the lower
// triangle of M (non-zero only at ancestors) is stored as Lc[i][t], t = depth of the ancestor.  For
// k in subtree(i), "the ancestor of k at depth(i)" IS i, which turns every tree-sparse update into
// plain strided loops over the contiguous DFS range of descendants.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/rsb.h"
#include "contact_solver.cuh"

namespace rsb {

constexpr int KMAX = RSB_KMAX;
constexpr int CMAX = 3 * KMAX;      // contact rows
constexpr int LMAX = RSB_LMAX;      // joint-limit rows (first LMAX violated joints)
constexpr int RMAX = CMAX + LMAX;   // constraint rows: one lane each (<= 32)
constexpr int CP = RMAX + 1;        // Y row stride (odd)
constexpr int GP = RMAX + 1;        // G row stride (odd: conflict-free row access by lane)
static_assert(RMAX <= 32, "one constraint row per lane");
constexpr int NSEC = 32;
constexpr int NROUNDS = 2;         // 32-section rounds of the slip search: bracket 2*pi/32^(r+1); two regula-falsi steps finish it (contact_solver.cuh)
constexpr int SEC_STRIDE = 36;      // (NSEC+1) padded
constexpr int CT_WORDS = 16;        // per-contact shared record
constexpr int EXT_WORDS = 12;       // external wrench row: body (int bits), force(3), torque(3), point in the body frame(3), 2 pad
constexpr int MAX_PT_SLOTS = 2;     // candidate points per lane (npts <= 64)
constexpr int HIST_WORDS = 6 * 32;  // Anderson history of the Gauss-Seidel sweep map (stage D)
constexpr int MAX_PEERS = 8;        // GPUs of one NVSwitch domain that receive this GPU's observation rows (fused all-gather)
constexpr unsigned FULL = 0xffffffffu;

enum BodyField {
  BF_PARENT = 0, BF_JTYPE = 1, BF_QIDX = 2, BF_VIDX = 3, BF_DEPTH = 4, BF_SUBTREE = 5,
  BF_JPOS = 6, BF_JROT = 9, BF_AXIS = 18, BF_MASS = 21, BF_COM = 22, BF_INERTIA = 25, BF_LO = 31, BF_HI = 32, BF_COUNT = 33
};
enum PoseField { PF_R = 0, PF_P = 9, PF_A = 12, PF_COUNT = 15 };
enum CtField { CF_POS = 0, CF_N = 3, CF_T1 = 6, CF_T2 = 9, CF_DEPTH = 12, CF_PT = 13, CF_BODY = 14, CF_PAIR = 15 };

// Model dimensions that fix every table offset.  A kernel can be compiled for a given Dims
// (offsets become immediates) or read them from the blob header at run time (generic path).
struct Dims { int nb, nq, nv, floating, maxdepth, maxdd; };

__host__ __device__ constexpr int round_up_c(int x, int m) { return (x + m - 1) / m * m; }
__host__ __device__ constexpr int max_c(int a, int b) { return a > b ? a : b; }

// header of the model constant blob (first 32 words)
struct BlobHeader {
  int nb, nq, nv, npts, floating, maxdepth, nbp, nptp, nvp, nqp;
  int off_body, off_anc, off_pts, off_gain, off_dofq, off_sec;
  // dof tree (floating base = chain of 6 dofs) for the branch-sparse factorisation
  int nbase, maxdd, dlp, nent;
  int off_ddepth, off_dsub, off_danc, off_dbody, off_bdof, off_lvl, off_lvldofs, off_entstart, off_ent, off_lcad;
  int off_coll, ncoll; // collision-body table (box features): [ncoll][COLL_WORDS] = half extents, body-frame position, rotation
  int words, flags;    // flags bit0: every joint origin has identity rotation (rpy = 0 in the URDF); bits 8..15: largest
                       // non-root subtree size - 1 (loop bound of stage A's subtree accumulation)
};
static_assert(sizeof(BlobHeader) == 136, "header is 34 words");
constexpr int HEADER_WORDS = 36;      // padded to a 16-byte multiple
constexpr int PT_ROWS = 15;           // candidate table rows: body, pos(3), radius, friction override, type, pos2(3), collision body, cull point(3), cull radius
constexpr int COLL_WORDS = 16;

// Every offset except off_ent / words depends on Dims only: the two variable-size tables
// (candidate points, factorisation entry list) sit at the end.
__host__ __device__ constexpr BlobHeader make_blob_header(Dims d, int npts, int nent, int ncoll = 0) {
  BlobHeader H{};
  H.nb = d.nb; H.nq = d.nq; H.nv = d.nv; H.npts = npts; H.floating = d.floating; H.maxdepth = d.maxdepth;
  H.nbp = d.nb | 1;                       // odd stride: field-major reads by body index stay conflict-free
  H.nptp = max_c(1, npts);
  H.nvp = round_up_c(max_c(d.nv, 1), 4);
  H.nqp = round_up_c(max_c(d.nq, 1), 4);
  H.nbase = d.floating ? 6 : 0; H.maxdd = d.maxdd; H.dlp = (d.maxdd + 1) | 1; H.nent = nent;
  const int DL = d.maxdd + 1;
  int off = HEADER_WORDS;
  H.off_body = off; off += 33 * H.nbp;
  H.off_anc = off; off += max_c(1, d.maxdepth) * H.nbp;
  H.off_gain = off; off += 3 * H.nvp;                 // kp, kd, actuator effort limit per dof
  H.off_dofq = off; off += H.nvp;
  H.off_sec = off; off += 2 * NROUNDS * SEC_STRIDE;
  H.off_ddepth = off; off += H.nvp;
  H.off_dsub = off; off += H.nvp;
  H.off_danc = off; off += DL * H.nvp;
  H.off_dbody = off; off += H.nvp;
  H.off_bdof = off; off += H.nbp;
  H.off_lvl = off; off += DL + 1;
  H.off_lvldofs = off; off += H.nvp;
  H.off_entstart = off; off += DL + 1;
  H.off_lcad = off; off += (d.nb * H.nbp + 3) / 4;
  H.off_pts = off; off += PT_ROWS * H.nptp;           // body, pos(3), radius, friction override (< 0: default material), type, pos2(3), collision body, cull point(3) + radius
  H.ncoll = ncoll; H.off_coll = off; off += COLL_WORDS * ncoll;
  H.off_ent = off; off += max_c(1, nent);
  H.words = round_up_c(off, 4);
  return H;
}

// per-warp workspace layout (word offsets)
struct WsLayout {
  int o_gc, o_gv, o_tau, o_pt, o_vt, o_L, o_invd, o_rhs, o_z, o_ct, o_Y, o_lam, o_u, o_lim, o_hist, o_sat;   // persistent
  int o_h, o_b, o_pose;                                                                  // union A
  int o_G;                                                                               // union B
  int words;
};

__host__ __device__ constexpr WsLayout make_ws_layout(Dims d) {
  WsLayout L{};
  const int nvp = round_up_c(max_c(d.nv, 1), 4), nqp = round_up_c(max_c(d.nq, 1), 4), nbp = d.nb | 1, dlp = (d.maxdd + 1) | 1;
  int o = 0;
  L.o_gc = o; o += nqp;
  L.o_gv = o; o += nvp;
  L.o_tau = o; o += nvp;
  L.o_pt = o; o += nqp;
  L.o_vt = o; o += nvp;
  L.o_L = o; o += round_up_c(max_c(1, d.nv) * dlp, 4);            // compact rows: [dof][ancestor depth]
  L.o_invd = o; o += nvp;
  L.o_rhs = o; o += nvp;
  L.o_z = o; o += nvp;
  L.o_ct = o; o += KMAX * CT_WORDS;
  L.o_Y = o; o += round_up_c((d.maxdd + 1) * CP, 4);              // [ancestor depth][contact row]
  L.o_lam = o; o += 32;
  L.o_u = o; o += CB_WORDS * KMAX;                                // per contact: G_ii (6), friction, its inverse (6): contact_solver.cuh
  L.o_lim = o; o += 4 * LMAX;                                     // joint-limit rows: dof, sign, violation
  L.o_sat = o; o += nvp;                                          // dof driven at its actuator effort limit in this sub-step (stage C -> E)
  L.o_hist = o; o += HIST_WORDS;                                  // Anderson acceleration: u0, x, g, f, dG, dF (one value per constraint row each)
  if (o - L.o_Y < 9 * 64) o = L.o_Y + 9 * 64;                     // stage B keeps its hit list (HL_CAP rows of HL_WORDS) in [o_Y, here): dead until stage C
  // union: {h, b, poses} (stages A-C) overlaid by G (stages C-D)
  int ua = 0;
  L.o_h = o + ua; ua += nvp;
  L.o_b = o + ua; ua += nvp;
  L.o_pose = o + ua; ua += round_up_c(15 * nbp, 4);
  L.o_G = o;
  const int ub = round_up_c(RMAX * GP, 4);
  o += max_c(ua, ub);
  L.words = round_up_c(o, 32);
  return L;
}

struct TerrainDesc {
  int type;            // 0 none, 1 Ground, 2 HeightMap
  float ground_z;
  int xs, ys;
  float x0, y0, dx, dy, xmax, ymax;   // grid origin, pitch, index bounds (xs-1, ys-1 as float)
  const float* h;
  const int* env_map;  // terrain atlas: height-map index of every environment (null: one shared map)
  int map_words;       // xs * ys
  float hmax;          // largest height of the map(s): a candidate whose lowest point is above it cannot touch (stage B cull)
  float inv_dx, inv_dy; // reciprocal pitch (sphere groups: cell of a point without an IEEE division)
};

// RaisimGym ANYmal locomotion task (SURVEY.md 8f N1; [RECALL] raisimGymTorch envs/rsg_anymal/Environment.hpp): constants of
// ENVIRONMENT::step() / isTerminalState() / reset(), all device pointers
struct GymConfig {
  const float* gc_init;      // [nq]
  const float* gv_init;      // [nv]
  const float* action_mean;  // [nq - 7]
  const float* action_std;   // [nq - 7]
  uint32_t foot_mask;        // bit b set: contacts on body b do not terminate the episode
  float torque_coeff, forward_vel_coeff, terminal_reward;
};

struct StepArgs {
  int num_envs, substeps;
  int gc_stride, gv_stride, pt_stride, vt_stride;   // vt_stride likewise for vtarget; pt_stride: row stride of ptarget (own padded buffer or a bound caller buffer)
  float *gc, *gv;
  const float *tau, *ptarget, *vtarget;
  int use_pd;
  float* pt_store;     // when the targets are read in place from a caller buffer (zero-copy, possibly pinned host memory):
  float* vt_store;     // keep a copy in the batch's own rows, so that setPdTarget semantics (targets persist) hold
  rsb_params prm;
  TerrainDesc ter;
  WsLayout ws;
  int blob_words;
  const uint32_t* blob;
  // outputs
  int* ncontacts;
  rsb_contact* contacts;
  int* contact_pt;     // [N][KMAX]
  int* iters;          // [N]
  int* diverged;       // [N] 1 when the stored state holds a non-finite value (caller resets those environments)
  float* resid;        // [N] largest impulse update of the last Gauss-Seidel sweep (< threshold: the solve converged)
  int* solver_status;  // [N] RSB_SOLVER_* of the last sub-step's solve
  float* tau_applied;  // [N][gv_stride] generalized force actually applied in the last sub-step (getGeneralizedForce)
  float *dbg_M, *dbg_h, *dbg_R, *dbg_p;   // optional (integrate1 / getters)
  float* obs;          // optional [N][ob_dim]: RaisimGym observation row of the final state, written by this kernel
  int ob_dim;
  const float* ext;    // optional [num_envs][EXT_WORDS] external wrench rows (body, F world, T world, point in body frame); null = none
  unsigned* prof;      // optional [num_envs][4 sub-steps][8] SM-clock stamps at the stage boundaries (tools/balance_probe.py)
  // fused observation all-gather (SURVEY 8e): every rank's kernel stores its observation rows straight into every peer's
  // [world * num_envs][ob_dim] buffer over NVLink (peer memory mapped into this process), then signals one counter per peer
  float* peer_obs[MAX_PEERS];      // peer p's gathered-rows buffer of this step (null = not in use)
  unsigned* peer_flag[MAX_PEERS];  // peer p's arrival counters [world]: += 1 per finished CTA of this rank
  int peer_world, peer_rank;
  unsigned peer_expected;          // arrival count every rank's counter reaches when its rows of THIS step have landed (steps so far x CTAs)
  unsigned* peer_done;             // CTAs of this launch that finished: the last one waits for the peers (set whenever peer_world > 0)
  // RaisimGym task fused into the step (rsb_batch_gym_step): the launch turns the action rows into PD targets before the first
  // sub-step and, after the last one, computes reward and termination, resets the terminated environments and writes the
  // observation rows of the (possibly reset) state -- VectorizedEnvironment::step() + observe() in ONE launch
  const float* gym_action;         // [num_envs][nq - 7] action rows (device memory or mapped pinned host memory); null = no task
  GymConfig gym;
  float* gym_reward;               // [num_envs]
  unsigned char* gym_done;         // [num_envs]
  int phase_mask;      // bit0: stop after stage B (integrate1: no state update); bit2: kinematics only (stage A + getters' buffers,
                       // the contact records of the last integrate() stay as they are)
  int substep_barrier; // 1: re-align the CTA's warps at every sub-step (instruction-cache locality experiment)
};

// ------------------------------------------------------------------ small device math ----------
struct f3 { float x, y, z; };
__device__ __forceinline__ f3 mk(float x, float y, float z) { f3 r; r.x = x; r.y = y; r.z = z; return r; }
__device__ __forceinline__ f3 operator+(f3 a, f3 b) { return mk(a.x + b.x, a.y + b.y, a.z + b.z); }
__device__ __forceinline__ f3 operator-(f3 a, f3 b) { return mk(a.x - b.x, a.y - b.y, a.z - b.z); }
__device__ __forceinline__ f3 operator*(float s, f3 a) { return mk(s * a.x, s * a.y, s * a.z); }
__device__ __forceinline__ float dot(f3 a, f3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
__device__ __forceinline__ f3 cross(f3 a, f3 b) { return mk(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x); }
__device__ __forceinline__ f3 mulR(const float* R, f3 v) {
  return mk(R[0] * v.x + R[1] * v.y + R[2] * v.z, R[3] * v.x + R[4] * v.y + R[5] * v.z, R[6] * v.x + R[7] * v.y + R[8] * v.z);
}
__device__ __forceinline__ f3 mulRt(const float* R, f3 v) {
  return mk(R[0] * v.x + R[3] * v.y + R[6] * v.z, R[1] * v.x + R[4] * v.y + R[7] * v.z, R[2] * v.x + R[5] * v.y + R[8] * v.z);
}
__device__ __forceinline__ void matmul3(const float* A, const float* B, float* C) {
#pragma unroll
  for (int i = 0; i < 3; i++)
#pragma unroll
    for (int j = 0; j < 3; j++) C[3 * i + j] = A[3 * i] * B[j] + A[3 * i + 1] * B[3 + j] + A[3 * i + 2] * B[6 + j];
}
__device__ __forceinline__ f3 shfl3(f3 v, int src) {
  return mk(__shfl_sync(FULL, v.x, src), __shfl_sync(FULL, v.y, src), __shfl_sync(FULL, v.z, src));
}

// ------------------------------------------------------------------ TMA bulk copy + mbarrier ---
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n" : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  // bounded spin: a TMA that never lands must trap, not hang the GPU
  for (uint32_t spin = 0; !mbar_try_wait(bar, parity); spin++)
    if (spin > (1u << 26)) __trap();
}
__device__ __forceinline__ void cp_async4(float* dst_smem, const float* src_gmem) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(dst_smem)), "l"(src_gmem) : "memory");
}
__device__ __forceinline__ void tma_bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// Observation arithmetic shared by rsb_observe_kernel and the fused write in rsb_step_kernel: explicit
// round-to-nearest intrinsics, so that both produce bit-identical rows whatever the compiler contracts elsewhere.
// c = column `col` (0..2) of the base rotation matrix of the unit quaternion (qw, qx, qy, qz).
__device__ __forceinline__ void obs_rot_column(float qw, float qx, float qy, float qz, int col, float& c0, float& c1, float& c2) {
  const float xx = __fmul_rn(qx, qx), yy = __fmul_rn(qy, qy), zz = __fmul_rn(qz, qz);
  const float xy = __fmul_rn(qx, qy), xz = __fmul_rn(qx, qz), yz = __fmul_rn(qy, qz);
  const float wx = __fmul_rn(qw, qx), wy = __fmul_rn(qw, qy), wz = __fmul_rn(qw, qz);
  const float r00 = __fsub_rn(1.f, __fmul_rn(2.f, __fadd_rn(yy, zz))), r01 = __fmul_rn(2.f, __fsub_rn(xy, wz)), r02 = __fmul_rn(2.f, __fadd_rn(xz, wy));
  const float r10 = __fmul_rn(2.f, __fadd_rn(xy, wz)), r11 = __fsub_rn(1.f, __fmul_rn(2.f, __fadd_rn(xx, zz))), r12 = __fmul_rn(2.f, __fsub_rn(yz, wx));
  const float r20 = __fmul_rn(2.f, __fsub_rn(xz, wy)), r21 = __fmul_rn(2.f, __fadd_rn(yz, wx)), r22 = __fsub_rn(1.f, __fmul_rn(2.f, __fadd_rn(xx, yy)));
  c0 = col == 0 ? r00 : col == 1 ? r01 : r02;
  c1 = col == 0 ? r10 : col == 1 ? r11 : r12;
  c2 = col == 0 ? r20 : col == 1 ? r21 : r22;
}
__device__ __forceinline__ float obs_dot3(float c0, float c1, float c2, float x, float y, float z) {
  return __fmaf_rn(c2, z, __fmaf_rn(c1, y, __fmul_rn(c0, x)));
}

// ------------------------------------------------------------------ terrain --------------------
__device__ __forceinline__ bool terrain_query(const TerrainDesc& t, int hm_offset, f3 P, float& dist, f3& n, int& pair) {
  if (t.type == 1) { dist = P.z - t.ground_z; n = mk(0.f, 0.f, 1.f); pair = 0; return true; }
  if (t.type != 2) return false;
  float gx = (P.x - t.x0) / t.dx, gy = (P.y - t.y0) / t.dy;
  if (!(gx >= 0.f) || !(gy >= 0.f) || !(gx < t.xmax) || !(gy < t.ymax)) return false;
  int ix = (int)gx, iy = (int)gy;
  float fx = gx - (float)ix, fy = gy - (float)iy;
  const float* H = t.h + hm_offset + iy * t.xs + ix;
  float h00 = __ldg(H), h10 = __ldg(H + 1), h01 = __ldg(H + t.xs), h11 = __ldg(H + t.xs + 1);
  float sx, sy; int tri;
  if (fx >= fy) { sx = h10 - h00; sy = h11 - h10; tri = 0; }
  else { sx = h11 - h01; sy = h01 - h00; tri = 1; }
  float zt = h00 + sx * fx + sy * fy;
  float nx = -sx / t.dx, ny = -sy / t.dy;
  float inv = 1.0f / sqrtf(nx * nx + ny * ny + 1.0f);
  n = mk(nx * inv, ny * inv, inv);
  dist = (P.z - zt) * inv;
  pair = 2 * (iy * (t.xs - 1) + ix) + tri;
  return true;
}

#include "narrow_phase.cuh"

// getters of integrate1(): full symmetric M rebuilt from the compact rows, h, body poses (cold path)
__device__ __noinline__ void write_debug(const StepArgs& args, int env, int lane, int nv, int nb, int nvp, int DLP, const float* s_L,
                                         const float* s_h, const int* ddepth, const int* danc, bool bvalid, const float* s_pose, int nbp) {
  float* gM = args.dbg_M + (size_t)env * nv * nv;
  for (int i = lane; i < nv * nv; i += 32) {
    int r = i / nv, c = i % nv;
    if (r < c) { int t = r; r = c; c = t; }
    int dc = ddepth[c];
    gM[i] = (dc <= ddepth[r] && danc[dc * nvp + r] == c) ? s_L[r * DLP + dc] : 0.f;
  }
  float* gh = args.dbg_h + (size_t)env * nv;
  for (int i = lane; i < nv; i += 32) gh[i] = s_h[i];
  if (bvalid) {
    float* gR = args.dbg_R + ((size_t)env * nb + lane) * 9;
    float* gp = args.dbg_p + ((size_t)env * nb + lane) * 3;
    for (int k = 0; k < 9; k++) gR[k] = s_pose[(PF_R + k) * nbp + lane];   // poses were published to shared memory by stage A
    for (int k = 0; k < 3; k++) gp[k] = s_pose[(PF_P + k) * nbp + lane];
  }
}


// 1/sqrt(x) and sqrt(x) for x > 0: MUFU.RSQ + one Newton step (relative error < 2e-7, the level of a float32 rounding);
// the IEEE sqrtf / division pair of the generic path costs ~27 instructions per pivot.
__device__ __forceinline__ float rsqrt_nr(float x) {
  float r;
  asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r * (1.5f - 0.5f * x * r * r);
}

// ---- compile-time topology: floating base + four serial chains of three joints (every 12-joint quadruped) -------------
// dof 0..5 = base, dof 6 + 3 leg + j = joint j of that leg (j = 0 hip abduction, 1 hip flexion, 2 knee); body b >= 1 carries
// dof 5 + b.  The compact row of dof (leg, j) holds its 6 base couplings at t = 0..5 and its chain entries at t = 6..6+j.
// Lane (leg = lane >> 3, t = lane & 7) keeps column t of its leg's three rows in registers: the leg blocks factorise with
// four shuffles per level and no table look-ups (the generic path walks entry lists, subtree ranges and level tables).
constexpr int QDLP = 9;   // compact row stride of the quadruped (maxdd + 1 = 9)
struct QuadLeg { float k, h, a, i8, i7, i6, k7, k6, h6; };   // column t of the knee / hip-flexion / hip-abduction rows; inverse pivots; couplings

__device__ __forceinline__ QuadLeg quad_factor_legs(float* s_L, float* s_invd, int lane) {
  const int leg = lane >> 3, t = lane & 7, l0 = lane & 24;
  const int rA = 6 + 3 * leg, rH = rA + 1, rK = rA + 2;
  QuadLeg q;
  q.k = s_L[rK * QDLP + t];
  q.h = s_L[rH * QDLP + t];
  q.a = t < 7 ? s_L[rA * QDLP + t] : 0.f;
  const float k8 = s_L[rK * QDLP + 8];
  q.i8 = rsqrt_nr(k8);
  q.k *= q.i8;                                          // level 8: the knee row has no descendants
  q.k7 = __shfl_sync(FULL, q.k, l0 + 7);
  q.h -= q.k7 * q.k;                                    // level 7: hip flexion, descendant = knee
  const float h7 = __shfl_sync(FULL, q.h, l0 + 7);
  q.i7 = rsqrt_nr(h7);
  q.h = (t == 7) ? h7 * q.i7 : q.h * q.i7;
  q.k6 = __shfl_sync(FULL, q.k, l0 + 6); q.h6 = __shfl_sync(FULL, q.h, l0 + 6);
  q.a -= q.k6 * q.k + q.h6 * q.h;                       // level 6: hip abduction, descendants = flexion, knee
  const float a6 = __shfl_sync(FULL, q.a, l0 + 6);
  q.i6 = rsqrt_nr(a6);
  q.a = (t == 6) ? a6 * q.i6 : q.a * q.i6;
  __syncwarp();   // every lane of the leg has read the knee pivot k8 above; lane t == 0 overwrites it below (racecheck: read / write without a barrier)
  s_L[rK * QDLP + t] = q.k; s_L[rH * QDLP + t] = q.h;
  if (t < 7) s_L[rA * QDLP + t] = q.a;
  if (t == 0) { s_L[rK * QDLP + 8] = k8 * q.i8; s_invd[rK] = q.i8; s_invd[rH] = q.i7; s_invd[rA] = q.i6; }
  return q;
}


// ------------------------------------------------------------------ stage B: narrow phase ------
// lane = contact candidate (SLOTS x 32 of them): Ground / HeightMap queries, ballot-compacted contact list in candidate order, the
// RSB_KMAX deepest kept.  Out of line (one call per sub-step) so that the candidate registers of both slots get an allocation of
// their own instead of being spilled around the rest of the 72-register kernel body.  Returns the number of contacts written to s_ct.
// Stage B writes every penetrating candidate into a per-warp hit list in shared memory (rows of HL_WORDS words, candidate order), keeps
// the KMAX deepest and emits the contact records.  Nothing per candidate survives in registers across the candidate slots, so the
// stage needs no register arrays (which ptxas had placed in local memory) and can be compiled out of line.
constexpr int HL_WORDS = 9;            // depth (<= 0: dropped), normal, position, pair, candidate index; odd stride: conflict-free by lane
constexpr int HL_CAP = 64;             // two candidate slots per lane at most

#ifndef RSB_STAGE_B_INLINE
#define RSB_STAGE_B_INLINE __forceinline__
#endif
// ter: the kernel parameter itself (constant bank); ter_s: its shared-memory copy, for the out-of-line shape routines
template <int SLOTS>
__device__ RSB_STAGE_B_INLINE int stage_b_narrow_phase(const TerrainDesc& ter, const TerrainDesc& ter_s, const uint32_t* blob_s, const float* s_pose, float* s_ct, float* s_list,
                                                 int env, int lane, int nbp, unsigned* prof) {
  const BlobHeader& H = *reinterpret_cast<const BlobHeader*>(blob_s);
  const float* ptsf = reinterpret_cast<const float*>(blob_s + H.off_pts);
  const int* ptsi = reinterpret_cast<const int*>(blob_s + H.off_pts);
  const int hm_offset = ter.env_map ? __ldg(ter.env_map + env) * ter.map_words : 0;   // terrain atlas
  const bool on_hm = ter.type == 2;
  // nothing whose lowest point is above the highest point of the terrain (the plane itself for a Ground) can touch it
  const float zcull = on_hm ? ter.hmax : ter.ground_z;
  const unsigned lt = (1u << lane) - 1u;
  int cnt = 0;
#pragma unroll 1
  for (int s = 0; s < SLOTS; s++) {
    const int k = lane + 32 * s;
    // ---- cull on the height alone: every candidate carries a bounding sphere (rows 11-14: centre in the body frame, radius; a body
    // welded to the world has radius -3e38 and never passes); third row of the body rotation, one dot product.  An upright robot
    // keeps its feet.
    bool alive = false;
    int pb = 0;
    if (k < H.npts && ter.type != 0) {
      pb = ptsi[0 * H.nptp + k];
      const float zc = s_pose[(PF_P + 2) * nbp + pb] + s_pose[(PF_R + 6) * nbp + pb] * ptsf[11 * H.nptp + k] + s_pose[(PF_R + 7) * nbp + pb] * ptsf[12 * H.nptp + k] +
                       s_pose[(PF_R + 8) * nbp + pb] * ptsf[13 * H.nptp + k];
      alive = zc - ptsf[14 * H.nptp + k] <= zcull;
    }
    if (!__any_sync(FULL, alive)) continue;
    bool hit = false, sph = false; float depth = 0.f; f3 n = mk(0, 0, 1), pos = mk(0, 0, 0); int pair = 0;
    if (alive) {
      const int ptype = ptsi[6 * H.nptp + k]; const float rad = ptsf[4 * H.nptp + k];
      const f3 pl = mk(ptsf[1 * H.nptp + k], ptsf[2 * H.nptp + k], ptsf[3 * H.nptp + k]);
      float Rb[9];
#pragma unroll
      for (int q = 0; q < 9; q++) Rb[q] = s_pose[(PF_R + q) * nbp + pb];
      const f3 pb_pos = mk(s_pose[(PF_P + 0) * nbp + pb], s_pose[(PF_P + 1) * nbp + pb], s_pose[(PF_P + 2) * nbp + pb]);
      f3 P = pb_pos + mulR(Rb, pl);
      float prad = rad;
      bool as_point = ptype == 0 && !(on_hm && rad > 0.f), live = true;
      if (ptype == 3) {
        // cylinder cap: the lowest point of its rim circle (centre P, radius rad, axis a), the point of the circle furthest along -z
        f3 a = P - (pb_pos + mulR(Rb, mk(ptsf[7 * H.nptp + k], ptsf[8 * H.nptp + k], ptsf[9 * H.nptp + k])));
        a = (1.0f / sqrtf(dot(a, a))) * a;
        const f3 dd = mk(a.z * a.x, a.z * a.y, a.z * a.z - 1.f);
        const float dn = sqrtf(dot(dd, dd));
        if (dn > 1e-6f) { P = P + (rad / dn) * dd; prad = 0.f; as_point = true; }
        else live = false;                                  // cap parallel to the ground: the fixed rim samples carry it
      }
      if (on_hm && as_point && P.z - prad > ter.hmax) live = false;
      if (!live) {
      } else if (as_point) {
        // Ground plane, or a zero-radius point on a HeightMap (box corner, cylinder rim point): the triangle directly beneath
        float dist; f3 nn; int pr;
        if (terrain_query(ter, hm_offset, P, dist, nn, pr)) {
          const float d = prad - dist;
          if (d > 0.f) { hit = true; depth = d; pair = pr; n = nn; pos = P - prad * nn; }
        }
      } else if (on_hm) {
        // HeightMap: the shape against every triangle under its bounding box (narrow_phase.cuh)
        if (ptype == 0) {
          sph = true; pos = P; depth = rad;     // parked: eight lanes take it below
        } else {
          HmBest hb; hb.hit = false;
          if (ptype == 1) {
            const f3 P2 = pb_pos + mulR(Rb, mk(ptsf[7 * H.nptp + k], ptsf[8 * H.nptp + k], ptsf[9 * H.nptp + k]));
            if (fminf(P.z, P2.z) - rad <= ter.hmax) hb = segment_vs_heightmap(ter_s, hm_offset, P, P2, rad);
          } else {
            const float* cb = reinterpret_cast<const float*>(blob_s + H.off_coll) + COLL_WORDS * ptsi[10 * H.nptp + k];
            const f3 hsz = mk(cb[0], cb[1], cb[2]);
            float Rw[9];
            matmul3(Rb, cb + 6, Rw);
            const f3 cw = pb_pos + mulR(Rb, mk(cb[3], cb[4], cb[5]));
            const float ez = fabsf(Rw[6]) * hsz.x + fabsf(Rw[7]) * hsz.y + fabsf(Rw[8]) * hsz.z;
            if (cw.z - ez <= ter.hmax) hb = box_vs_heightmap(ter_s, hm_offset, cw, Rw, hsz);
          }
          if (hb.hit) { hit = true; depth = hb.depth; pair = hb.pair; n = hb.n; pos = hb.pos; }
        }
      }
    }
    // ---- this slot's direct hits go to the list at once (nothing of them stays in registers across the sphere groups)
    {
      const unsigned hmask = __ballot_sync(FULL, hit);
      if (hit) {
        float* e = s_list + HL_WORDS * (cnt + __popc(hmask & lt));
        e[0] = depth; e[1] = n.x; e[2] = n.y; e[3] = n.z; e[4] = pos.x; e[5] = pos.y; e[6] = pos.z; e[7] = __int_as_float(pair); e[8] = __int_as_float(k);
      }
      cnt += __popc(hmask);
    }
    // ---- sphere candidates on a HeightMap: four at a time, eight lanes (= the eight triangles of the 2 x 2 cell block under it) each;
    // the lane whose triangle wins appends the contact itself (position = centre - r n)
    const unsigned sm = __ballot_sync(FULL, sph);
    if (sm != 0u) {
      const int nsph = __popc(sm);
#pragma unroll 1
      for (int base = 0; base < nsph; base += 4) {
        const int rk = base + (lane >> 3);
        const bool gvalid = rk < nsph;
        const int olane = gvalid ? __fns(sm, 0, rk + 1) : 0;
        const f3 C = shfl3(pos, olane); const float r = __shfl_sync(FULL, depth, olane);
        const SphereTri st = sphere_vs_heightmap_group(ter, hm_offset, C, r, gvalid, lane);
        const bool win = gvalid && st.winner == lane;
        const unsigned wmask = __ballot_sync(FULL, win);
        if (win) {
          float* e = s_list + HL_WORDS * (cnt + __popc(wmask & lt));
          e[0] = st.depth; e[1] = st.n.x; e[2] = st.n.y; e[3] = st.n.z; e[4] = C.x - r * st.n.x; e[5] = C.y - r * st.n.y; e[6] = C.z - r * st.n.z;
          e[7] = __int_as_float(st.pair); e[8] = __int_as_float(olane + 32 * s);
        }
        cnt += __popc(wmask);
      }
    }
  }
  __syncwarp();
  if (prof && lane == 0) { prof[6] = (unsigned)clock64(); prof[7] = (unsigned)cnt; }
  int total = cnt;
#pragma unroll 1
  while (total > KMAX) {   // drop the shallowest (ties: highest candidate index) until KMAX remain
    float dmin = 3.0e38f; int cmin = -1, imin = 0;     // depth, candidate index, list row of the entry to drop
#pragma unroll 1
    for (int e = lane; e < cnt; e += 32) {
      const float d = s_list[HL_WORDS * e]; const int c = __float_as_int(s_list[HL_WORDS * e + 8]);
      if (d > 0.f && (d < dmin || (d == dmin && c > cmin))) { dmin = d; cmin = c; imin = e; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float d2 = __shfl_xor_sync(FULL, dmin, o); const int c2 = __shfl_xor_sync(FULL, cmin, o), i2 = __shfl_xor_sync(FULL, imin, o);
      if (d2 < dmin || (d2 == dmin && c2 > cmin)) { dmin = d2; cmin = c2; imin = i2; }
    }
    __syncwarp();                                       // the scan above read the row that lane 0 now clears
    if (lane == 0) s_list[HL_WORDS * imin] = 0.f;
    __syncwarp();
    total--;
  }
  // contact records in candidate order (the list holds each slot's direct hits before its sphere hits): rank = live entries with a smaller index
#pragma unroll 1
  for (int e0 = 0; e0 < cnt; e0 += 32) {
    const int e = e0 + lane;
    const float* le = s_list + HL_WORDS * min(e, cnt - 1);
    const float depth = le[0];
    const bool live = e < cnt && depth > 0.f;
    const int cand = __float_as_int(le[8]);
    int rank = 0;
#pragma unroll 1
    for (int j = 0; j < cnt; j++) rank += (s_list[HL_WORDS * j] > 0.f && __float_as_int(s_list[HL_WORDS * j + 8]) < cand) ? 1 : 0;
    if (live) {
      float* ct = s_ct + rank * CT_WORDS;
      const f3 n = mk(le[1], le[2], le[3]);
      const f3 ex = (fabsf(n.x) < 0.9f) ? mk(1.f, 0.f, 0.f) : mk(0.f, 1.f, 0.f);
      const f3 t = ex - dot(ex, n) * n;
      const float inv = rsqrt_nr(dot(t, t));
      const f3 t1 = inv * t, t2 = cross(n, t1);
      ct[CF_POS] = le[4]; ct[CF_POS + 1] = le[5]; ct[CF_POS + 2] = le[6];
      ct[CF_N] = n.x; ct[CF_N + 1] = n.y; ct[CF_N + 2] = n.z;
      ct[CF_T1] = t1.x; ct[CF_T1 + 1] = t1.y; ct[CF_T1 + 2] = t1.z;
      ct[CF_T2] = t2.x; ct[CF_T2 + 1] = t2.y; ct[CF_T2 + 2] = t2.z;
      ct[CF_DEPTH] = depth;
      ct[CF_PT] = __int_as_float(cand); ct[CF_BODY] = __int_as_float(ptsi[cand]); ct[CF_PAIR] = le[7];
    }
  }
  return total;
}

// ------------------------------------------------------------------ the kernel -----------------
// SNB > 0: compiled for the model dimensions (SNB, SNQ, SNV, SFL, SMAXDEPTH, SMAXDD) -- every table and
// workspace offset is an immediate.  SNB == 0: generic, dimensions read from the blob header.
template <int WPC, int SLOTS, int SNB, int SNQ, int SNV, int SFL, int SMAXDEPTH, int SMAXDD>
__global__ void __launch_bounds__(WPC * 32, (WPC == 14 ? 2 : 1)) rsb_step_kernel(const __grid_constant__ StepArgs args) {
  extern __shared__ __align__(128) uint32_t smem[];
  __shared__ __align__(8) uint64_t tma_bar;
  const int lane = threadIdx.x & 31;     // (re-read wherever needed at 72 registers; S2R SR_LANEID instead, with or without a range assumption, measured 12 % slower)
  // the shuffle marks the warp index as warp-uniform for the compiler: the workspace base then lives in a uniform register
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
  constexpr bool ST = SNB > 0;
  // every 12-joint quadruped: the host selects this instance only when the parent table is base + 4 chains of 3 (pick_config)
  constexpr bool QUAD = SNB == 13 && SNQ == 19 && SNV == 18 && SFL == 1 && SMAXDEPTH == 3 && SMAXDD == 8;
  // deep trees on few resident warps (the humanoid instance: 14 warps per SM, latency-bound) get their dependent shared-memory loops of
  // stage C unrolled for memory-level parallelism; everything else keeps them rolled (instruction cache)
#ifndef RSB_DEEP_UNROLL
#define RSB_DEEP_UNROLL 4
#endif
  constexpr int UNR = (ST && !QUAD && SMAXDD >= 12) ? RSB_DEEP_UNROLL : 1;
  constexpr Dims SD{SNB, SNQ, SNV, SFL, SMAXDEPTH, SMAXDD};
  constexpr WsLayout LS = make_ws_layout(SD);
  constexpr BlobHeader HS = make_blob_header(SD, 0, 0);
#define WSO(f) (ST ? LS.f : args.ws.f)
  // shared memory: [WPC workspaces][model constant blob]
  uint32_t* const blob_s = smem + WPC * WSO(words);

  // ---- stage the model constant block once per CTA with one TMA bulk copy ----------------------
  // the out-of-line stages read the terrain descriptor and the solver parameters from shared memory: a reference to the kernel
  // parameters is a generic pointer there, and every field read through it a global-latency load (ncu: long scoreboard)
  __shared__ TerrainDesc s_ter;
  __shared__ rsb_params s_prm;
  if (threadIdx.x == 0) {
    mbar_init(&tma_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    s_ter = args.ter; s_prm = args.prm;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    mbar_expect_tx(&tma_bar, (uint32_t)args.blob_words * 4u);
    tma_bulk_g2s(blob_s, args.blob, (uint32_t)args.blob_words * 4u, &tma_bar);
  }
  mbar_wait(&tma_bar, 0);

  const BlobHeader& H = *reinterpret_cast<const BlobHeader*>(blob_s);
#define HO(f) (ST ? HS.f : H.f)
  const int nb = HO(nb), nq = HO(nq), nv = HO(nv), floating = HO(floating), maxdepth = HO(maxdepth);
  const int nbp = HO(nbp), nvp = HO(nvp);

  const float* bodyf = reinterpret_cast<const float*>(blob_s + HO(off_body));
  const int* bodyi = reinterpret_cast<const int*>(blob_s + HO(off_body));
  const int* anc = reinterpret_cast<const int*>(blob_s + HO(off_anc));
  const float* ptsf = reinterpret_cast<const float*>(blob_s + HO(off_pts));
  const float* kp = reinterpret_cast<const float*>(blob_s + HO(off_gain));
  const float* kd = kp + nvp;
  const float* emax = kp + 2 * nvp;     // actuator effort limit per dof (URDF <limit effort>, 3e38 = none)
  const int* dofq = reinterpret_cast<const int*>(blob_s + HO(off_dofq));
  const float* sec_c = reinterpret_cast<const float*>(blob_s + HO(off_sec));
  const int nbase = HO(nbase), maxdd = HO(maxdd), DLP = HO(dlp);
  const int* ddepth = reinterpret_cast<const int*>(blob_s + HO(off_ddepth));
  const int* dsub = reinterpret_cast<const int*>(blob_s + HO(off_dsub));
  const int* danc = reinterpret_cast<const int*>(blob_s + HO(off_danc));
  const int* dbody = reinterpret_cast<const int*>(blob_s + HO(off_dbody));
  const int* bdof = reinterpret_cast<const int*>(blob_s + HO(off_bdof));
  const int* lvl = reinterpret_cast<const int*>(blob_s + HO(off_lvl));
  const int* lvldofs = reinterpret_cast<const int*>(blob_s + HO(off_lvldofs));
  const int* entstart = reinterpret_cast<const int*>(blob_s + HO(off_entstart));
  const int* ent = reinterpret_cast<const int*>(blob_s + H.off_ent);
  const int8_t* lcad = reinterpret_cast<const int8_t*>(blob_s + HO(off_lcad));

  float* const ws = reinterpret_cast<float*>(smem) + warp * WSO(words);
  float* s_gc = ws + WSO(o_gc); float* s_gv = ws + WSO(o_gv); float* s_tau = ws + WSO(o_tau); float* s_pt = ws + WSO(o_pt); float* s_vt = ws + WSO(o_vt);
  float* s_L = ws + WSO(o_L); float* s_invd = ws + WSO(o_invd); float* s_rhs = ws + WSO(o_rhs); float* s_z = ws + WSO(o_z); float* s_ct = ws + WSO(o_ct);
  float* s_Y = ws + WSO(o_Y); float* s_lam = ws + WSO(o_lam); float* s_u = ws + WSO(o_u); float* s_lim = ws + WSO(o_lim); float* s_hist = ws + WSO(o_hist); float* s_sat = ws + WSO(o_sat);
  float* s_h = ws + WSO(o_h); float* s_b = ws + WSO(o_b); float* s_pose = ws + WSO(o_pose); float* s_G = ws + WSO(o_G);
#undef WSO
#undef HO
  // Long-lived per-thread values are kept to a minimum: at 72 registers (28 warps x 32 lanes per SM) everything cached
  // here is spilled, and 28 warps' spill slots do not fit the L1 next to the terrain gathers -- every reload was an L2
  // round trip on the critical path.  Kernel parameters are read in place (constant bank), model constants from the
  // shared-memory blob at the point of use.

  // body constants of this lane (lane == body)
  const int b = lane;
  const bool bvalid = b < nb;
  const int bb = bvalid ? b : 0;
#define MYB(f) (bodyi[(f) * nbp + bb])
  // (row, col) of the base 6x6 lower triangle owned by lanes 0..20, packed row | col << 3: one table per CTA
  __shared__ uint8_t s_tri[32];
  if (threadIdx.x < 32) {
    int pr = 0;
    for (int r = 0, e = 0; r < 6; r++) for (int c = 0; c <= r; c++, e++) if (e == (int)threadIdx.x) pr = r | (c << 3);
    s_tri[threadIdx.x] = (uint8_t)pr;
  }
  __syncthreads();

  const int warps_total = gridDim.x * WPC;
#pragma unroll 1
  for (int env = blockIdx.x * WPC + warp; env < args.num_envs; env += warps_total) {
    // ---- load this environment's rows (coalesced: one row per warp) -----------------------------
    {
      const float* g_gc = args.gc + (size_t)env * args.gc_stride;
      const float* g_gv = args.gv + (size_t)env * args.gv_stride;
#pragma unroll 1
      for (int i = lane; i < nq; i += 32) s_gc[i] = g_gc[i];
#pragma unroll 1
      for (int i = lane; i < nv; i += 32) s_gv[i] = g_gv[i];
#pragma unroll 1
      for (int i = lane; i < nv; i += 32) s_tau[i] = args.tau ? args.tau[(size_t)env * args.gv_stride + i] : 0.f;
      if (args.use_pd) {
        // PD targets are first needed in stage C: fetch them asynchronously (cp.async, global -> shared) so that a
        // caller buffer in pinned host memory (zero-copy control step) is read over PCIe behind stages A and B
        // gym task: the joint part of the position target is action * actionStd + actionMean (ENVIRONMENT::step(), first half); the base
        // part comes from the batch's own rows like every other target
        const int nfetch = args.gym_action ? 7 : nq;
#pragma unroll 1
        for (int i = lane; i < nfetch; i += 32) cp_async4(&s_pt[i], &args.ptarget[(size_t)env * args.pt_stride + i]);
#pragma unroll 1
        for (int i = lane; i < nv; i += 32) cp_async4(&s_vt[i], &args.vtarget[(size_t)env * args.vt_stride + i]);
        asm volatile("cp.async.commit_group;" ::: "memory");
        if (args.gym_action) {
          const int nj = nq - 7;
#pragma unroll 1
          for (int i = lane; i < nj; i += 32) s_pt[7 + i] = args.gym_action[(size_t)env * nj + i] * args.gym.action_std[i] + args.gym.action_mean[i];
        }
      }
    }
    __syncwarp();
    int K = 0, iters = 0;
    float resid = 0.f; int gs_status = RSB_SOLVER_CONVERGED;

#pragma unroll 1
    for (int sub = 0; sub < args.substeps; sub++) {
      // Re-align the CTA's warps (instruction-cache locality: 28 warps drifting through a 75 KB kernel miss the
      // instruction cache far more often than 28 warps in the same stage).  Only set by the host when every warp
      // owns exactly one environment, so all of them reach the barrier the same number of times.
      const int bar_threads = min(WPC, args.num_envs - (int)blockIdx.x * WPC) * 32;
      if (args.substep_barrier >= 1) asm volatile("bar.sync 1, %0;" ::"r"(bar_threads));
      if (args.prof && lane == 0) args.prof[((size_t)env * 4 + (sub & 3)) * 8 + 0] = (unsigned)clock64();
      // =========================== stage A: FK + RNEA + CRBA =====================================
      float R[9]; f3 p, w, v, wd, vd, ax;
      if (floating) {
        float qw = s_gc[3], qx = s_gc[4], qy = s_gc[5], qz = s_gc[6];
        float inv = 1.0f / sqrtf(qw * qw + qx * qx + qy * qy + qz * qz);
        qw *= inv; qx *= inv; qy *= inv; qz *= inv;
        R[0] = 1.f - 2.f * (qy * qy + qz * qz); R[1] = 2.f * (qx * qy - qw * qz); R[2] = 2.f * (qx * qz + qw * qy);
        R[3] = 2.f * (qx * qy + qw * qz); R[4] = 1.f - 2.f * (qx * qx + qz * qz); R[5] = 2.f * (qy * qz - qw * qx);
        R[6] = 2.f * (qx * qz - qw * qy); R[7] = 2.f * (qy * qz + qw * qx); R[8] = 1.f - 2.f * (qx * qx + qy * qy);
        p = mk(s_gc[0], s_gc[1], s_gc[2]);
        v = mk(s_gv[0], s_gv[1], s_gv[2]); w = mk(s_gv[3], s_gv[4], s_gv[5]);
      } else {
#pragma unroll
        for (int k = 0; k < 9; k++) R[k] = bodyf[(BF_JROT + k) * nbp];
        p = mk(bodyf[(BF_JPOS + 0) * nbp], bodyf[(BF_JPOS + 1) * nbp], bodyf[(BF_JPOS + 2) * nbp]);
        v = mk(0.f, 0.f, 0.f); w = mk(0.f, 0.f, 0.f);
      }
      const f3 O = p;                      // base origin: centre of the world-aligned CRBA frame
      const bool jrot_identity = (H.flags & 1) != 0;
      wd = mk(0.f, 0.f, 0.f); vd = mk(-args.prm.gravity[0], -args.prm.gravity[1], -args.prm.gravity[2]); ax = mk(0.f, 0.f, 0.f);
#pragma unroll 1
      for (int d = 1; d <= maxdepth; d++) {
        int j = (bvalid && d <= MYB(BF_DEPTH)) ? anc[(d - 1) * nbp + b] : -1;
        if (j >= 0) {
          f3 jp = mk(bodyf[(BF_JPOS + 0) * nbp + j], bodyf[(BF_JPOS + 1) * nbp + j], bodyf[(BF_JPOS + 2) * nbp + j]);
          float Rj[9];
          f3 al = mk(bodyf[(BF_AXIS + 0) * nbp + j], bodyf[(BF_AXIS + 1) * nbp + j], bodyf[(BF_AXIS + 2) * nbp + j]);
          f3 r = mulR(R, jp);
          if (jrot_identity) {
#pragma unroll
            for (int k = 0; k < 9; k++) Rj[k] = R[k];
          } else {
            float Jr[9];      // scoped here: declared outside the branch it was a maybe-uninitialised value carried (through the stack) round the loop
#pragma unroll
            for (int k = 0; k < 9; k++) Jr[k] = bodyf[(BF_JROT + k) * nbp + j];
            matmul3(R, Jr, Rj);
          }
          f3 aj = mulR(Rj, al);
          float q = s_gc[bodyi[BF_QIDX * nbp + j]], qd = s_gv[bodyi[BF_VIDX * nbp + j]];
          const bool rev = bodyi[BF_JTYPE * nbp + j] == 1;
          if (!rev) r = r + q * aj;
          f3 wxr = cross(w, r);
          f3 vn = v + wxr;
          f3 vdn = vd + cross(wd, r) + cross(w, wxr);
          f3 qa = qd * aj;
          if (rev) {
            float sq, cq;
            sincosf(q, &sq, &cq);
            float t = 1.f - cq;
            float Rq[9] = {t * al.x * al.x + cq, t * al.x * al.y - sq * al.z, t * al.x * al.z + sq * al.y,
                           t * al.x * al.y + sq * al.z, t * al.y * al.y + cq, t * al.y * al.z - sq * al.x,
                           t * al.x * al.z - sq * al.y, t * al.y * al.z + sq * al.x, t * al.z * al.z + cq};
            matmul3(Rj, Rq, R);
            wd = wd + cross(w, qa);
            w = w + qa;
          } else {
#pragma unroll
            for (int k = 0; k < 9; k++) R[k] = Rj[k];
            vn = vn + qa;
            vdn = vdn + 2.f * cross(w, qa);
          }
          p = p + r; v = vn; vd = vdn; ax = aj;
        }
      }
      // publish poses for stages B and C
      if (bvalid) {
#pragma unroll
        for (int k = 0; k < 9; k++) s_pose[(PF_R + k) * nbp + b] = R[k];
        s_pose[(PF_P + 0) * nbp + b] = p.x; s_pose[(PF_P + 1) * nbp + b] = p.y; s_pose[(PF_P + 2) * nbp + b] = p.z;
        s_pose[(PF_A + 0) * nbp + b] = ax.x; s_pose[(PF_A + 1) * nbp + b] = ax.y; s_pose[(PF_A + 2) * nbp + b] = ax.z;
      }
      // per-body force and inertia terms about O
      float X[16];   // F(3) N_O(3) m h(3) I_O(6)
      {
        float m = bvalid ? bodyf[BF_MASS * nbp + bb] : 0.f;
        f3 cl = mk(bodyf[(BF_COM + 0) * nbp + bb], bodyf[(BF_COM + 1) * nbp + bb], bodyf[(BF_COM + 2) * nbp + bb]);
        f3 c = mulR(R, cl);
        f3 cO = (p - O) + c;
        f3 ac = vd + cross(wd, c) + cross(w, cross(w, c));
        f3 f = m * ac;
        float I0 = bodyf[(BF_INERTIA + 0) * nbp + bb], I1 = bodyf[(BF_INERTIA + 1) * nbp + bb], I2 = bodyf[(BF_INERTIA + 2) * nbp + bb];
        float I3 = bodyf[(BF_INERTIA + 3) * nbp + bb], I4 = bodyf[(BF_INERTIA + 4) * nbp + bb], I5 = bodyf[(BF_INERTIA + 5) * nbp + bb];
        if (!bvalid) { I0 = I1 = I2 = I3 = I4 = I5 = 0.f; }
        // Iw = R I R^T
        float RI[9];
#pragma unroll
        for (int r = 0; r < 3; r++) {
          RI[3 * r + 0] = R[3 * r] * I0 + R[3 * r + 1] * I1 + R[3 * r + 2] * I2;
          RI[3 * r + 1] = R[3 * r] * I1 + R[3 * r + 1] * I3 + R[3 * r + 2] * I4;
          RI[3 * r + 2] = R[3 * r] * I2 + R[3 * r + 1] * I4 + R[3 * r + 2] * I5;
        }
        float W0 = RI[0] * R[0] + RI[1] * R[1] + RI[2] * R[2], W1 = RI[0] * R[3] + RI[1] * R[4] + RI[2] * R[5], W2 = RI[0] * R[6] + RI[1] * R[7] + RI[2] * R[8];
        float W3 = RI[3] * R[3] + RI[4] * R[4] + RI[5] * R[5], W4 = RI[3] * R[6] + RI[4] * R[7] + RI[5] * R[8], W5 = RI[6] * R[6] + RI[7] * R[7] + RI[8] * R[8];
        f3 Iw = mk(W0 * w.x + W1 * w.y + W2 * w.z, W1 * w.x + W3 * w.y + W4 * w.z, W2 * w.x + W4 * w.y + W5 * w.z);
        f3 Iwd = mk(W0 * wd.x + W1 * wd.y + W2 * wd.z, W1 * wd.x + W3 * wd.y + W4 * wd.z, W2 * wd.x + W4 * wd.y + W5 * wd.z);
        f3 n = Iwd + cross(w, Iw) + cross(cO, f);
        float cc = dot(cO, cO);
        X[0] = f.x; X[1] = f.y; X[2] = f.z; X[3] = n.x; X[4] = n.y; X[5] = n.z;
        X[6] = m; X[7] = m * cO.x; X[8] = m * cO.y; X[9] = m * cO.z;
        X[10] = W0 + m * (cc - cO.x * cO.x); X[11] = W1 - m * cO.x * cO.y; X[12] = W2 - m * cO.x * cO.z;
        X[13] = W3 + m * (cc - cO.y * cO.y); X[14] = W4 - m * cO.y * cO.z; X[15] = W5 + m * (cc - cO.z * cO.z);
      }
      if (args.ext) {   // ArticulatedSystem::setExternalForce / setExternalTorque: h -= J^T wrench, through the RNEA force terms
        const float* e = args.ext + (size_t)env * EXT_WORDS;
        if (bvalid && __float_as_int(e[0]) == b) {
          const f3 Fe = mk(e[1], e[2], e[3]), Te = mk(e[4], e[5], e[6]);
          const f3 re = (p - O) + mulR(R, mk(e[7], e[8], e[9]));
          const f3 Me = cross(re, Fe) + Te;
          X[0] -= Fe.x; X[1] -= Fe.y; X[2] -= Fe.z; X[3] -= Me.x; X[4] -= Me.y; X[5] -= Me.z;
        }
      }
      // subtree sums: bodies are in DFS pre-order, so subtree(b) = lanes [b, b + size)
      float A[16];
#pragma unroll
      for (int k = 0; k < 16; k++) A[k] = X[k];
      const int my_sub = MYB(BF_SUBTREE);
      const int max_inner = (H.flags >> 8) & 0xff;   // largest non-root subtree size - 1
#pragma unroll 1
      for (int s = 1; s <= max_inner; s++) {
        bool take = (b > 0) && (s < my_sub);
#pragma unroll
        for (int k = 0; k < 16; k++) {
          float x = __shfl_down_sync(FULL, X[k], s);
          if (take) A[k] += x;
        }
      }
      {   // root: everything
        float T[16];
#pragma unroll
        for (int k = 0; k < 16; k++) {
          float t = X[k];
          // lanes >= nb hold exact zeros (zero mass and inertia): with at most 16 bodies the xor-16 step adds 0 and is skipped
#pragma unroll
          for (int o = (ST && SNB <= 16) ? 8 : 16; o > 0; o >>= 1) t += __shfl_xor_sync(FULL, t, o);
          T[k] = t;
        }
        if (b == 0) {
#pragma unroll
          for (int k = 0; k < 16; k++) A[k] = T[k];
        }
      }
      // bias force h and CRBA columns (row i of M stored compactly: column index = ancestor depth)
      f3 rO = p - O;
      const bool rev = MYB(BF_JTYPE) == 1;
      f3 Sw = rev ? ax : mk(0.f, 0.f, 0.f);
      f3 Sv = rev ? cross(rO, ax) : ax;
      f3 Fc = mk(A[0], A[1], A[2]), Nc = mk(A[3], A[4], A[5]);
      f3 hh = mk(A[7], A[8], A[9]);
      f3 ff = A[6] * Sv + cross(Sw, hh);
      f3 nn = mk(A[10] * Sw.x + A[11] * Sw.y + A[12] * Sw.z, A[11] * Sw.x + A[13] * Sw.y + A[14] * Sw.z, A[12] * Sw.x + A[14] * Sw.y + A[15] * Sw.z) + cross(hh, Sv);
      const int my_vidx = MYB(BF_VIDX);
      const int my_dd = nbase + MYB(BF_DEPTH) - 1;          // depth of this body's dof in the dof tree
      if (bvalid && b > 0) {
        float* row = s_L + my_vidx * DLP;
        s_h[my_vidx] = dot(Sw, Nc) + dot(Sv, Fc);      // S^T [N_O; F]  (moment about O)
        row[my_dd] = dot(Sw, nn) + dot(Sv, ff);
        if (floating) { row[0] = ff.x; row[1] = ff.y; row[2] = ff.z; row[3] = nn.x; row[4] = nn.y; row[5] = nn.z; }
      }
      if (b == 0 && floating) {
        s_h[0] = Fc.x; s_h[1] = Fc.y; s_h[2] = Fc.z; s_h[3] = Nc.x; s_h[4] = Nc.y; s_h[5] = Nc.z;
        // lower triangle of [ m 1, -[h]x ; [h]x, I_O ]
        s_L[0 * DLP + 0] = A[6]; s_L[1 * DLP + 0] = 0.f; s_L[1 * DLP + 1] = A[6];
        s_L[2 * DLP + 0] = 0.f; s_L[2 * DLP + 1] = 0.f; s_L[2 * DLP + 2] = A[6];
        s_L[3 * DLP + 0] = 0.f; s_L[3 * DLP + 1] = -hh.z; s_L[3 * DLP + 2] = hh.y;
        s_L[4 * DLP + 0] = hh.z; s_L[4 * DLP + 1] = 0.f; s_L[4 * DLP + 2] = -hh.x;
        s_L[5 * DLP + 0] = -hh.y; s_L[5 * DLP + 1] = hh.x; s_L[5 * DLP + 2] = 0.f;
        s_L[3 * DLP + 3] = A[10]; s_L[4 * DLP + 3] = A[11]; s_L[5 * DLP + 3] = A[12];
        s_L[4 * DLP + 4] = A[13]; s_L[5 * DLP + 4] = A[14]; s_L[5 * DLP + 5] = A[15];
      }
      {   // M[vi][vj] for proper ancestors j (excluding the root): column = depth of j's dof
        int j = (bvalid && b > 0) ? MYB(BF_PARENT) : 0;
        int tj = my_dd - 1;
#pragma unroll 1
        for (int d = 2; d <= maxdepth; d++) {
          int src = j > 0 ? j : 0;
          f3 Swj = shfl3(Sw, src), Svj = shfl3(Sv, src);
          if (j > 0) {
            s_L[my_vidx * DLP + tj] = dot(Swj, nn) + dot(Svj, ff);
            j = bodyi[BF_PARENT * nbp + j];
            tj--;
          }
        }
      }
      __syncwarp();
      if (args.prof && lane == 0) args.prof[((size_t)env * 4 + (sub & 3)) * 8 + 1] = (unsigned)clock64();
      if (args.dbg_M)   // getters (integrate1): cold path, kept out of line to spare the instruction cache
        write_debug(args, env, lane, nv, nb, nvp, DLP, s_L, s_h, ddepth, danc, bvalid, s_pose, nbp);
      if (args.phase_mask & 4) { asm volatile("cp.async.wait_all;" ::: "memory"); __syncwarp(); break; }   // kinematics for the getters only

      // =========================== stage B: narrow phase ========================================
      K = stage_b_narrow_phase<SLOTS>(args.ter, s_ter, blob_s, s_pose, s_ct, s_Y, env, lane, nbp, args.prof ? args.prof + ((size_t)env * 4 + (sub & 3)) * 8 : nullptr);
      const int C = 3 * K;
      if (args.prof && lane == 0) args.prof[((size_t)env * 4 + (sub & 3)) * 8 + 2] = (unsigned)clock64();
      if (args.phase_mask & 1) { asm volatile("cp.async.wait_all;" ::: "memory"); __syncwarp(); break; }   // integrate1(): kinematics, collision, M, h only

      if (args.substep_barrier >= 2) asm volatile("bar.sync 1, %0;" ::"r"(bar_threads));
      // =========================== stage C: b, Mhat = L^T L, z, Y, G ==============================
      // a9 joint limits: the first LMAX joints found beyond their URDF limit become unilateral rows sign * qdot >= target
      int Lm = 0;
      if (args.prm.joint_limits) {
        float q = 0.f, lo = -3.0e38f, hi = 3.0e38f;
        if (bvalid && b > 0) { q = s_gc[bodyi[BF_QIDX * nbp + b]]; lo = bodyf[BF_LO * nbp + b]; hi = bodyf[BF_HI * nbp + b]; }
        const bool act = q < lo || q > hi;
        const unsigned lm_mask = __ballot_sync(FULL, act);
        const int slot = __popc(lm_mask & ((1u << lane) - 1u));
        if (act && slot < LMAX) {
          s_lim[4 * slot + 0] = __int_as_float(MYB(BF_VIDX));
          s_lim[4 * slot + 1] = q < lo ? 1.f : -1.f;
          s_lim[4 * slot + 2] = q < lo ? lo - q : q - hi;
        }
        Lm = min(__popc(lm_mask), LMAX);
        __syncwarp();
      }
      const int C3 = C, CR = C3 + Lm;   // contact rows, all constraint rows
      if (sub == 0 && args.use_pd) {     // the asynchronous target fetch of the prologue lands here
        asm volatile("cp.async.wait_all;" ::: "memory");
        __syncwarp();
        if (args.pt_store) {
#pragma unroll 1
          for (int i = lane; i < nq; i += 32) args.pt_store[(size_t)env * args.gc_stride + i] = s_pt[i];
        }
        if (args.vt_store) {
#pragma unroll 1
          for (int i = lane; i < nv; i += 32) args.vt_store[(size_t)env * args.gv_stride + i] = s_vt[i];
        }
      }
#pragma unroll 1
      for (int i = lane; i < nv; i += 32) {
        float bi = s_tau[i] - s_h[i];
        // actuator effort limit (oracle step()): when feed-forward + PD law at the current state exceed it, the joint is driven by the
        // constant limit torque over this step and gets no implicit PD terms
        float te = s_tau[i];
        const float kpi = args.use_pd ? kp[i] : 0.f, kdi = args.use_pd ? kd[i] : 0.f;
        const bool pd = kpi != 0.f || kdi != 0.f;
        const int qi = pd ? dofq[i] : 0;
        if (pd) te += kpi * (s_pt[qi] - s_gc[qi]) + kdi * (s_vt[i] - s_gv[i]);
        // ... judged on the torque the implicit law would really apply (the explicit value over 1 + (dt kd + dt^2 kp) / M_dd)
        const float soft = args.prm.dt * kdi + args.prm.dt * args.prm.dt * kpi;
        const bool sat = fabsf(te) > emax[i] * (1.f + soft / s_L[i * DLP + ddepth[i]]);
        s_sat[i] = sat ? 1.f : 0.f;          // remembered for stage E (generalized force applied)
        if (sat) bi += copysignf(emax[i], te) - s_tau[i];
        else if (pd) {
          bi += kpi * (s_pt[qi] - s_gc[qi] - args.prm.dt * s_gv[i]) + kdi * (s_vt[i] - s_gv[i]);
          s_L[i * DLP + ddepth[i]] += args.prm.dt * kdi + args.prm.dt * args.prm.dt * kpi;
        }
        s_b[i] = bi;
      }
      __syncwarp();
      if constexpr (QUAD) {
        // ---- Mhat = L^T L with the topology compiled in: leg blocks in registers (quad_factor_legs), base block by 21 lanes
        static_assert(!QUAD || make_blob_header(SD, 0, 0).dlp == QDLP, "compact row stride");
        const QuadLeg ql = quad_factor_legs(s_L, s_invd, lane);
        __syncwarp();
        const int er = s_tri[lane] & 7, ec = s_tri[lane] >> 3;
        float val = 0.f;
        if (lane < 21) {
          val = s_L[er * QDLP + ec];
#pragma unroll
          for (int k = 6; k < 18; k++) val -= s_L[k * QDLP + er] * s_L[k * QDLP + ec];
        }
#pragma unroll
        for (int i = 5; i >= 0; i--) {
          const int ti = i * (i + 1) / 2;
          const float dd = __shfl_sync(FULL, val, ti + i);
          const float inv = rsqrt_nr(dd);
          if (er == i) val = (ec == i) ? dd * inv : val * inv;
          const float lir = __shfl_sync(FULL, val, ti + min(er, i));
          const float lic = __shfl_sync(FULL, val, ti + min(ec, i));
          if (lane < 21 && er < i) val -= lir * lic;
          if (lane == 0) s_invd[i] = inv;
        }
        if (lane < 21) s_L[er * QDLP + ec] = val;
        // ---- z = L^-T b: the three chain dofs of a leg in registers, then the base against every leg
        const int leg = lane >> 3, t = lane & 7, rA = 6 + 3 * leg;
        const float zK = s_b[rA + 2] * ql.i8;
        const float zH = (s_b[rA + 1] - ql.k7 * zK) * ql.i7;
        const float zA = (s_b[rA] - ql.h6 * zH - ql.k6 * zK) * ql.i6;
        if (t == 0) { s_z[rA] = zA; s_z[rA + 1] = zH; s_z[rA + 2] = zK; }
        float part = t < 6 ? ql.k * zK + ql.h * zH + ql.a * zA : 0.f;     // this leg's share of sum_k L[k][t] z_k
        part += __shfl_xor_sync(FULL, part, 8);
        part += __shfl_xor_sync(FULL, part, 16);
        __syncwarp();          // the base block and invd[0..5] written above are read below
        float acc = lane < 6 ? s_b[lane] - part : 0.f;
#pragma unroll
        for (int i = 5; i >= 0; i--) {
          const float zi = __shfl_sync(FULL, acc, i) * s_invd[i];
          if (lane < i) acc -= s_L[i * QDLP + lane] * zi;
          if (lane == i) s_z[i] = zi;
        }
        __syncwarp();
      } else {
        // ---- branch-sparse factorisation Mhat = L^T L, "pull" form, one dof-tree level at a time (deepest first):
        //      L[i][t] = (M[i][t] - sum_{k in subtree(i), k != i} L[k][depth i] L[k][t]) / L[i][i]
  #pragma unroll 1
        for (int lev = maxdd; lev >= nbase; lev--) {
          const int e0 = entstart[lev], ne = entstart[lev + 1] - e0;
  #pragma unroll 1
          for (int e = lane; e < ne; e += 32) {
            const int pk = ent[e0 + e], i = pk & 255, t = pk >> 8;
            float acc = s_L[i * DLP + t];
            const int kend = i + dsub[i];
  #pragma unroll (UNR)
            for (int k = i + 1; k < kend; k++) acc -= s_L[k * DLP + lev] * s_L[k * DLP + t];
            s_L[i * DLP + t] = acc;
          }
          __syncwarp();
          const int d0 = lvl[lev], nd = lvl[lev + 1] - d0;
          if (lane < nd) {
            const int i = lvldofs[d0 + lane];
            float d = sqrtf(s_L[i * DLP + lev]);
            s_L[i * DLP + lev] = d;
            s_invd[i] = 1.0f / d;
          }
          __syncwarp();
  #pragma unroll 1
          for (int e = lane; e < ne; e += 32) {
            const int pk = ent[e0 + e], i = pk & 255, t = pk >> 8;
            if (t < lev) s_L[i * DLP + t] *= s_invd[i];
          }
          __syncwarp();
        }
        if (floating) {   // base 6x6 block: every other dof is a descendant of every base dof
          const int er = s_tri[lane] & 7, ec = s_tri[lane] >> 3;
          float val = 0.f;
          if (lane < 21) {
            val = s_L[er * DLP + ec];
  #pragma unroll 4
            for (int k = 6; k < nv; k++) val -= s_L[k * DLP + er] * s_L[k * DLP + ec];
          }
  #pragma unroll 1
          for (int i = 5; i >= 0; i--) {
            const int ti = i * (i + 1) / 2;
            float d = sqrtf(__shfl_sync(FULL, val, ti + i));
            float inv = 1.0f / d;
            if (er == i) val = (ec == i) ? d : val * inv;
            float lir = __shfl_sync(FULL, val, ti + min(er, i));
            float lic = __shfl_sync(FULL, val, ti + min(ec, i));
            if (lane < 21 && er < i) val -= lir * lic;
            if (lane == 0) s_invd[i] = inv;
          }
          if (lane < 21) s_L[er * DLP + ec] = val;
          __syncwarp();
        }
        // ---- z = L^-T b  (leaves to root)
  #pragma unroll 1
        for (int lev = maxdd; lev >= nbase; lev--) {
          const int d0 = lvl[lev], nd = lvl[lev + 1] - d0;
          if (lane < nd) {
            const int i = lvldofs[d0 + lane];
            float acc = s_b[i];
            const int kend = i + dsub[i];
  #pragma unroll (UNR)
            for (int k = i + 1; k < kend; k++) acc -= s_L[k * DLP + lev] * s_z[k];
            s_z[i] = acc * s_invd[i];
          }
          __syncwarp();
        }
        if (floating) {
          float acc = 0.f;
          if (lane < 6) {
            acc = s_b[lane];
  #pragma unroll 4
            for (int k = 6; k < nv; k++) acc -= s_L[k * DLP + lane] * s_z[k];
          }
  #pragma unroll 1
          for (int i = 5; i >= 0; i--) {
            float zi = __shfl_sync(FULL, acc, i) * s_invd[i];
            if (lane < i) acc -= s_L[i * DLP + lane] * zi;
            if (lane == i) s_z[i] = zi;
          }
          __syncwarp();
        }
      }
      // ---- Y = L^-T J^T, one constraint row per lane, only along the row's own ancestor chain
      float u_c = 0.f;
      int row_lm = 5;          // QUAD: (leg << 4) | depth of this lane's row (chain = base dofs 0..5, then 3 leg + t for t = 6..depth)
      if constexpr (QUAD) {
        if (lane < CR) {
          const int c = lane;
          const bool is_lim = c >= C3;
          const float* ct = s_ct + (is_lim ? 0 : c / 3) * CT_WORDS;
          const float* lm = s_lim + 4 * (is_lim ? c - C3 : 0);
          const int d = c % 3;
          const int fo = (d == 0) ? CF_T1 : (d == 1 ? CF_T2 : CF_N);
          const f3 axd = mk(ct[fo], ct[fo + 1], ct[fo + 2]);
          const f3 pos = mk(ct[CF_POS], ct[CF_POS + 1], ct[CF_POS + 2]);
          const int i0 = is_lim ? __float_as_int(lm[0]) : 5 + __float_as_int(ct[CF_BODY]);   // body b >= 1 carries dof 5 + b; the base "dof" is 5
          const int leg = i0 >= 6 ? (i0 - 6) / 3 : 0;
          const int m = i0 >= 6 ? i0 - 3 * leg : 5;                                           // depth of that dof in the dof tree
          row_lm = (leg << 4) | m;
          float y[9];
          float jv;
          if (is_lim) {   // J = sign * e_dof
#pragma unroll
            for (int t = 0; t < 9; t++) y[t] = (t == m) ? lm[1] : 0.f;
            jv = lm[1] * s_gv[i0];
          } else {
            const f3 rc = cross(pos - O, axd);
            y[0] = axd.x; y[1] = axd.y; y[2] = axd.z; y[3] = rc.x; y[4] = rc.y; y[5] = rc.z;
            jv = axd.x * s_gv[0] + axd.y * s_gv[1] + axd.z * s_gv[2] + rc.x * s_gv[3] + rc.y * s_gv[4] + rc.z * s_gv[5];
#pragma unroll
            for (int t = 6; t < 9; t++) {
              y[t] = 0.f;
              if (t <= m) {
                const int j = 3 * leg + t - 5;         // body of chain dof 3 leg + t
                const f3 aj = mk(s_pose[(PF_A + 0) * nbp + j], s_pose[(PF_A + 1) * nbp + j], s_pose[(PF_A + 2) * nbp + j]);
                f3 col = aj;
                if (bodyi[BF_JTYPE * nbp + j] == 1) {
                  const f3 pj = mk(s_pose[(PF_P + 0) * nbp + j], s_pose[(PF_P + 1) * nbp + j], s_pose[(PF_P + 2) * nbp + j]);
                  col = cross(aj, pos - pj);
                }
                y[t] = dot(col, axd);
                jv += y[t] * s_gv[3 * leg + t];
              }
            }
          }
          float yz = 0.f;
#pragma unroll
          for (int sI = 8; sI >= 0; sI--) {
            if (sI <= m) {
              const int a_s = sI < 6 ? sI : 3 * leg + sI;
              const float ys = y[sI] * s_invd[a_s];
              y[sI] = ys;
              yz += ys * s_z[a_s];
#pragma unroll
              for (int t = 0; t < sI; t++) y[t] -= s_L[a_s * QDLP + t] * ys;
            }
          }
#pragma unroll
          for (int t = 0; t < 9; t++) if (t <= m) s_Y[t * CP + c] = y[t];
          u_c = jv + args.prm.dt * yz;
          if (is_lim) u_c -= args.prm.erp * lm[2] / args.prm.dt;
          else if (d == 2) {
            float target = args.prm.erp * ct[CF_DEPTH] / args.prm.dt;
            if (args.prm.restitution > 0.f && jv < -args.prm.rest_threshold) target += -args.prm.restitution * jv;
            u_c -= target;
          }
        }
      } else {
        if (lane < CR) {
          const int c = lane;
          const bool is_lim = c >= C3;
          const float* ct = s_ct + (is_lim ? 0 : c / 3) * CT_WORDS;
          const float* lm = s_lim + 4 * (is_lim ? c - C3 : 0);
          const int d = c % 3;
          const int fo = (d == 0) ? CF_T1 : (d == 1 ? CF_T2 : CF_N);
          const f3 axd = mk(ct[fo], ct[fo + 1], ct[fo + 2]);
          const f3 pos = mk(ct[CF_POS], ct[CF_POS + 1], ct[CF_POS + 2]);
          const int i0 = is_lim ? __float_as_int(lm[0]) : bdof[__float_as_int(ct[CF_BODY])];
          const int m = i0 >= 0 ? ddepth[i0] : -1;
          float jv = 0.f;
          if (is_lim) {   // J = sign * e_dof
  #pragma unroll 1
            for (int t = 0; t < m; t++) s_Y[t * CP + c] = 0.f;
            s_Y[m * CP + c] = lm[1];
            jv = lm[1] * s_gv[i0];
          } else {
            if (floating) {
              f3 rc = cross(pos - O, axd);
              s_Y[0 * CP + c] = axd.x; s_Y[1 * CP + c] = axd.y; s_Y[2 * CP + c] = axd.z;
              s_Y[3 * CP + c] = rc.x; s_Y[4 * CP + c] = rc.y; s_Y[5 * CP + c] = rc.z;
              jv = axd.x * s_gv[0] + axd.y * s_gv[1] + axd.z * s_gv[2] + rc.x * s_gv[3] + rc.y * s_gv[4] + rc.z * s_gv[5];
            }
  #pragma unroll (UNR > 1 ? 2 : 1)
            for (int t = nbase; t <= m; t++) {
              const int a_t = danc[t * nvp + i0], j = dbody[a_t];
              f3 aj = mk(s_pose[(PF_A + 0) * nbp + j], s_pose[(PF_A + 1) * nbp + j], s_pose[(PF_A + 2) * nbp + j]);
              f3 col = aj;
              if (bodyi[BF_JTYPE * nbp + j] == 1) {
                f3 pj = mk(s_pose[(PF_P + 0) * nbp + j], s_pose[(PF_P + 1) * nbp + j], s_pose[(PF_P + 2) * nbp + j]);
                col = cross(aj, pos - pj);
              }
              float val = dot(col, axd);
              s_Y[t * CP + c] = val;
              jv += val * s_gv[a_t];
            }
          }
          float yz = 0.f;
          if constexpr (ST && SMAXDD + 1 <= 9) {
            // whole chain in registers (compile-time indices): 2 instructions per multiply-add instead of 4
            constexpr int DLc = SMAXDD + 1;
            float y[DLc];
  #pragma unroll
            for (int t = 0; t < DLc; t++) y[t] = (t <= m) ? s_Y[t * CP + c] : 0.f;
  #pragma unroll
            for (int sI = DLc - 1; sI >= 0; sI--) {
              if (sI <= m) {
                const int a_s = danc[sI * nvp + i0];
                const float ys = y[sI] * s_invd[a_s];
                y[sI] = ys;
                yz += ys * s_z[a_s];
  #pragma unroll
                for (int t = 0; t < sI; t++) y[t] -= s_L[a_s * DLP + t] * ys;
              }
            }
  #pragma unroll
            for (int t = 0; t < DLc; t++) if (t <= m) s_Y[t * CP + c] = y[t];
          } else {
  #pragma unroll 1
            for (int sI = m; sI >= 0; sI--) {
              const int a_s = danc[sI * nvp + i0];
              float y = s_Y[sI * CP + c] * s_invd[a_s];
              s_Y[sI * CP + c] = y;
              yz += y * s_z[a_s];
  #pragma unroll (UNR)
              for (int t = 0; t < sI; t++) s_Y[t * CP + c] -= s_L[a_s * DLP + t] * y;
            }
          }
          u_c = jv + args.prm.dt * yz;
          if (is_lim) u_c -= args.prm.erp * lm[2] / args.prm.dt;
          else if (d == 2) {
            float target = args.prm.erp * ct[CF_DEPTH] / args.prm.dt;
            if (args.prm.restitution > 0.f && jv < -args.prm.rest_threshold) target += -args.prm.restitution * jv;
            u_c -= target;
          }
        }
      }
      iters = 0; resid = 0.f; gs_status = RSB_SOLVER_CONVERGED;
      if (CR > 0) {
        __syncwarp();      // h / b / poses are dead from here: G overlays them
        // G = Y^T Y; rows a, b share ancestors exactly up to the depth of their bodies' LCA
        if constexpr (QUAD) {
          const int ng = 32 / CR;
          const int a = lane % CR, g = lane / CR;
          const int pa = __shfl_sync(FULL, row_lm, a);
          const int nit = (CR / 2 + ng) / ng;              // ceil((CR / 2 + 1) / ng): every lane runs the same trip count (warp-wide shuffle inside)
#pragma unroll 1
          for (int itr = 0; itr < nit; itr++) {
            const int dd = g + itr * ng;
            const bool active = g < ng && dd <= CR / 2;
            int bcol = a + dd; if (bcol >= CR) bcol -= CR;
            if (!active) bcol = 0;
            const int pb = __shfl_sync(FULL, row_lm, bcol);
            // same leg: the chains agree down to the shallower of the two; different legs (or a base row): the six base dofs only
            const int tmax = ((pa ^ pb) >> 4) == 0 ? min(pa & 15, pb & 15) : 5;
            if (active) {
              float sacc = 0.f;
#pragma unroll
              for (int t = 0; t < 9; t++) if (t <= tmax) sacc += s_Y[t * CP + a] * s_Y[t * CP + bcol];
              s_G[a * GP + bcol] = sacc; s_G[bcol * GP + a] = sacc;
            }
          }
        } else {
          {
            const int ng = 32 / CR;                   // CR <= 28 -> ng >= 1
            const int a = lane % CR, g = lane / CR;
            if (g < ng) {
              const int ba = a < C3 ? __float_as_int(s_ct[(a / 3) * CT_WORDS + CF_BODY]) : dbody[__float_as_int(s_lim[4 * (a - C3)])];
  #pragma unroll 1
              for (int dd = g; dd <= CR / 2; dd += ng) {
                int bcol = a + dd; if (bcol >= CR) bcol -= CR;
                const int bbody = bcol < C3 ? __float_as_int(s_ct[(bcol / 3) * CT_WORDS + CF_BODY]) : dbody[__float_as_int(s_lim[4 * (bcol - C3)])];
                const int tmax = lcad[ba * nbp + bbody];
                float sacc = 0.f;
  #pragma unroll (UNR)
                for (int t = 0; t <= tmax; t++) sacc += s_Y[t * CP + a] * s_Y[t * CP + bcol];
                s_G[a * GP + bcol] = sacc; s_G[bcol * GP + a] = sacc;
              }
            }
          }
        }
        __syncwarp();
        // per-contact constants: symmetric 3x3 block, friction and the block's inverse (lane i < K computes, all read)
        if (lane < K) {
          const int i3 = 3 * lane;
          float a = s_G[i3 * GP + i3], bq = s_G[i3 * GP + i3 + 1], cc = s_G[i3 * GP + i3 + 2];
          float d = s_G[(i3 + 1) * GP + i3 + 1], e = s_G[(i3 + 1) * GP + i3 + 2], f = s_G[(i3 + 2) * GP + i3 + 2];
          float c00 = d * f - e * e, c01 = cc * e - bq * f, c02 = bq * e - cc * d;
          float c11 = a * f - cc * cc, c12 = bq * cc - a * e, c22 = a * d - bq * bq;
          float id = 1.0f / (a * c00 + bq * c01 + cc * c02);
          float* o = s_u + CB_WORDS * lane;
          const float pm = ptsf[5 * H.nptp + __float_as_int(s_ct[lane * CT_WORDS + CF_PT])];
          o[0] = a; o[1] = bq; o[2] = cc; o[3] = d; o[4] = e; o[5] = f;
          o[6] = pm >= 0.f ? pm : args.prm.mu;     // per-collision-body friction (World::setMaterialPairProp analogue)
          o[8] = c00 * id; o[9] = c01 * id; o[10] = c02 * id; o[11] = c11 * id; o[12] = c12 * id; o[13] = c22 * id;
        }
        __syncwarp();
        if (args.prof && lane == 0) args.prof[((size_t)env * 4 + (sub & 3)) * 8 + 3] = (unsigned)clock64();
        // =========================== stage D: per-contact Gauss-Seidel ===========================
        const GsResult gs = gs_solve(s_prm, s_G, GP, s_u, s_hist, sec_c, SEC_STRIDE, lane, K, Lm, u_c);
        iters = gs.iters; resid = gs.resid; gs_status = gs.status;
        if (lane < CR) s_lam[lane] = gs.lam;
        __syncwarp();
      }
      __syncwarp();
      if (args.prof && lane == 0) args.prof[((size_t)env * 4 + (sub & 3)) * 8 + 4] = (unsigned)clock64();
      if (args.substep_barrier >= 3) asm volatile("bar.sync 1, %0;" ::"r"(bar_threads));
      // =========================== stage E: v+ = v + L^-1 (dt z + Y lam), integration ============
      if constexpr (QUAD) {
        // w_i = dt z_i + sum over the rows whose chain holds dof i of Y[depth i][row] lam_row, lane = dof
        const int i = min(lane, 17);
        const int legi = i >= 6 ? (i - 6) / 3 : 0, di = i >= 6 ? i - 3 * legi : i;
        float sacc = args.prm.dt * s_z[i];
#pragma unroll 1
        for (int k = 0; k < K; k++) {
          const int pr = __shfl_sync(FULL, row_lm, 3 * k);
          if (i < 6 || ((pr >> 4) == legi && (pr & 15) >= di))
            sacc += s_Y[di * CP + 3 * k] * s_lam[3 * k] + s_Y[di * CP + 3 * k + 1] * s_lam[3 * k + 1] + s_Y[di * CP + 3 * k + 2] * s_lam[3 * k + 2];
        }
#pragma unroll 1
        for (int l = 0; l < Lm; l++) {
          const int pr = __shfl_sync(FULL, row_lm, C3 + l);
          if (i < 6 || ((pr >> 4) == legi && (pr & 15) >= di)) sacc += s_Y[di * CP + C3 + l] * s_lam[C3 + l];
        }
        // x = L^-1 w, root to leaves: the base chain by shuffles, then the three joints of every leg by shuffles from the parent lanes
        float acc = lane < 6 ? sacc : 0.f;
#pragma unroll
        for (int t = 0; t < 6; t++) {
          const float xt = __shfl_sync(FULL, acc, t) * s_invd[t];
          if (lane > t && lane < 6) acc -= s_L[lane * QDLP + t] * xt;
          if (lane == t) acc = xt;
        }
        // acc (lanes 0..5) = x of the base dofs
        float legacc = sacc;
#pragma unroll
        for (int t = 0; t < 6; t++) legacc -= s_L[i * QDLP + t] * __shfl_sync(FULL, acc, t);
        const int j = i >= 6 ? di - 6 : 0;
        const float inv = s_invd[i];
        const float x0 = legacc * inv;                                            // joint 0 of a leg
        const float xa1 = __shfl_up_sync(FULL, x0, 1);
        const float x1 = (legacc - s_L[i * QDLP + 6] * xa1) * inv;               // joint 1: parent = joint 0
        const float xa2 = __shfl_up_sync(FULL, x0, 2), xh2 = __shfl_up_sync(FULL, x1, 1);
        const float x2 = (legacc - s_L[i * QDLP + 6] * xa2 - s_L[i * QDLP + 7] * xh2) * inv;   // joint 2: ancestors = joints 0, 1
        if (lane < 18) s_rhs[lane] = lane < 6 ? acc : (j == 0 ? x0 : (j == 1 ? x1 : x2));
        __syncwarp();
      } else {
  #pragma unroll 1
        for (int i = lane; i < nv; i += 32) {   // w = dt z + Y lam, gathered per dof over the contacts whose chain holds it
          float sacc = args.prm.dt * s_z[i];
          const int di = ddepth[i];
  #pragma unroll (UNR)
          for (int k = 0; k < K; k++) {
            const int i0 = bdof[__float_as_int(s_ct[k * CT_WORDS + CF_BODY])];
            if (i0 >= 0 && ddepth[i0] >= di && danc[di * nvp + i0] == i)
              sacc += s_Y[di * CP + 3 * k] * s_lam[3 * k] + s_Y[di * CP + 3 * k + 1] * s_lam[3 * k + 1] + s_Y[di * CP + 3 * k + 2] * s_lam[3 * k + 2];
          }
  #pragma unroll 1
          for (int l = 0; l < Lm; l++) {
            const int i0 = __float_as_int(s_lim[4 * l]);
            if (ddepth[i0] >= di && danc[di * nvp + i0] == i) sacc += s_Y[di * CP + C3 + l] * s_lam[C3 + l];
          }
          s_rhs[i] = sacc;
        }
        __syncwarp();
        if (floating) {   // x = L^-1 w, root to leaves: base chain by shuffles, then one tree level at a time
          float acc = lane < 6 ? s_rhs[lane] : 0.f;
  #pragma unroll 1
          for (int t = 0; t < 6; t++) {
            float xt = __shfl_sync(FULL, acc, t) * s_invd[t];
            if (lane > t && lane < 6) acc -= s_L[lane * DLP + t] * xt;
            if (lane == t) s_rhs[t] = xt;
          }
          __syncwarp();
        }
  #pragma unroll 1
        for (int lev = nbase; lev <= maxdd; lev++) {
          const int d0 = lvl[lev], nd = lvl[lev + 1] - d0;
          if (lane < nd) {
            const int i = lvldofs[d0 + lane];
            float acc = s_rhs[i];
            // base dofs are ancestors of every other dof and are their own index: no ancestor lookup
  #pragma unroll
            for (int t = 0; t < 6; t++) if (t < nbase) acc -= s_L[i * DLP + t] * s_rhs[t];
  #pragma unroll (UNR)
            for (int t = nbase; t < lev; t++) acc -= s_L[i * DLP + t] * s_rhs[danc[t * nvp + i]];
            s_rhs[i] = acc * s_invd[i];
          }
          __syncwarp();
        }
      }
#pragma unroll 1
      for (int i = lane; i < nv; i += 32) {
        const float v0 = s_gv[i], vp = v0 + s_rhs[i];
        s_gv[i] = vp;
        // generalized force applied over this step (implicit PD evaluated at q + dt v+, v+; the effort limit where it was hit): getGeneralizedForce()
        float ta = s_tau[i];
        const float kpi = args.use_pd ? kp[i] : 0.f, kdi = args.use_pd ? kd[i] : 0.f;
        const bool pd = kpi != 0.f || kdi != 0.f;
        const int qi = pd ? dofq[i] : 0;
        float te = ta;
        if (pd) te += kpi * (s_pt[qi] - s_gc[qi]) + kdi * (s_vt[i] - v0);
        if (s_sat[i] != 0.f) ta = copysignf(emax[i], te);
        else if (pd) ta += kpi * (s_pt[qi] - s_gc[qi] - args.prm.dt * vp) + kdi * (s_vt[i] - vp);
        s_b[i] = ta;
      }
      __syncwarp();
      if (floating) {
        if (lane < 3) s_gc[lane] += args.prm.dt * s_gv[lane];
        f3 wn = mk(s_gv[3], s_gv[4], s_gv[5]);
        float wnorm = sqrtf(dot(wn, wn)), ang = wnorm * args.prm.dt;
        float qw, qx, qy, qz;
        if (ang > 1e-10f) { float sh, ch; sincosf(0.5f * ang, &sh, &ch); float s = sh / wnorm; qw = ch; qx = s * wn.x; qy = s * wn.y; qz = s * wn.z; }
        else { qw = 1.f; qx = 0.5f * args.prm.dt * wn.x; qy = 0.5f * args.prm.dt * wn.y; qz = 0.5f * args.prm.dt * wn.z; }
        float pw = s_gc[3], px = s_gc[4], py = s_gc[5], pz = s_gc[6];
        float nw = qw * pw - qx * px - qy * py - qz * pz;
        float nx = qw * px + qx * pw + qy * pz - qz * py;
        float ny = qw * py - qx * pz + qy * pw + qz * px;
        float nz = qw * pz + qx * py - qy * px + qz * pw;
        float inv = 1.0f / sqrtf(nw * nw + nx * nx + ny * ny + nz * nz);
        __syncwarp();
        if (lane == 0) { s_gc[3] = nw * inv; s_gc[4] = nx * inv; s_gc[5] = ny * inv; s_gc[6] = nz * inv; }
      }
#pragma unroll 1
      for (int i = lane; i < nv; i += 32) {
        int qi = dofq[i];
        if (qi >= (floating ? 7 : 0)) s_gc[qi] += args.prm.dt * s_gv[i];
      }
      __syncwarp();
      if (args.prof && lane == 0) args.prof[((size_t)env * 4 + (sub & 3)) * 8 + 5] = (unsigned)clock64();
    }   // substeps

    if (args.gym_action) {
      // ENVIRONMENT::step() second half + isTerminalState() + reset(), same arithmetic as the stand-alone task kernel it replaces:
      // reward = torque_coeff |tau|^2 + forward_vel_coeff min(4, body-frame x velocity); any contact on a non-foot body ends the episode
      float qw = s_gc[3], qx = s_gc[4], qy = s_gc[5], qz = s_gc[6];
      const float inv = 1.0f / sqrtf(qw * qw + qx * qx + qy * qy + qz * qz);
      qw *= inv; qx *= inv; qy *= inv; qz *= inv;
      const float r00 = 1.f - 2.f * (qy * qy + qz * qz), r10 = 2.f * (qx * qy + qw * qz), r20 = 2.f * (qx * qz - qw * qy);
      const float vbx = r00 * s_gv[0] + r10 * s_gv[1] + r20 * s_gv[2];
      float t2 = 0.f;
#pragma unroll 1
      for (int i = lane; i < nv; i += 32) t2 += s_b[i] * s_b[i];          // s_b: generalized force applied in the last sub-step (stage E)
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) t2 += __shfl_xor_sync(FULL, t2, o);
      bool bad = false;
      if (lane < K) bad = ((args.gym.foot_mask >> __float_as_int(s_ct[lane * CT_WORDS + CF_BODY])) & 1u) == 0u;
      const bool term = __any_sync(FULL, bad);
      float r = args.gym.torque_coeff * t2 + args.gym.forward_vel_coeff * fminf(4.0f, vbx);
      __syncwarp();
      if (term) {
        r += args.gym.terminal_reward;
#pragma unroll 1
        for (int i = lane; i < nq; i += 32) { const float g0 = args.gym.gc_init[i]; s_gc[i] = g0; if (args.pt_store) args.pt_store[(size_t)env * args.gc_stride + i] = g0; }
#pragma unroll 1
        for (int i = lane; i < nv; i += 32) s_gv[i] = args.gym.gv_init[i];
      }
      if (lane == 0) { args.gym_reward[env] = r; args.gym_done[env] = term ? 1 : 0; }
      __syncwarp();
    }
    // ---- store state rows and contact records -----------------------------------------------------
    if (!(args.phase_mask & 1)) {
      float* g_gc = args.gc + (size_t)env * args.gc_stride;
      float* g_gv = args.gv + (size_t)env * args.gv_stride;
#pragma unroll 1
      for (int i = lane; i < nq; i += 32) g_gc[i] = s_gc[i];
#pragma unroll 1
      for (int i = lane; i < nv; i += 32) { g_gv[i] = s_gv[i]; args.tau_applied[(size_t)env * args.gv_stride + i] = s_b[i]; }
    }
    if (args.obs && floating) {   // VectorizedEnvironment::observe() fused into the step: [z, R^T e_z, q_j, R^T v, R^T w, qdot_j]
      float qw = s_gc[3], qx = s_gc[4], qy = s_gc[5], qz = s_gc[6];
      const float inv = 1.0f / sqrtf(qw * qw + qx * qx + qy * qy + qz * qz);
      qw *= inv; qx *= inv; qy *= inv; qz *= inv;
      float* o = args.obs + (size_t)env * args.ob_dim;
      const int nj = nq - 7;
      if (lane == 0) o[0] = s_gc[2];
      if (lane < 3) {   // same arithmetic as rsb_observe_kernel (aux_kernels.cuh)
        float c0, c1, c2;
        obs_rot_column(qw, qx, qy, qz, lane, c0, c1, c2);
        o[1 + lane] = c2;
        o[4 + nj + lane] = obs_dot3(c0, c1, c2, s_gv[0], s_gv[1], s_gv[2]);
        o[7 + nj + lane] = obs_dot3(c0, c1, c2, s_gv[3], s_gv[4], s_gv[5]);
      }
#pragma unroll 1
      for (int i = lane; i < nj; i += 32) { o[4 + i] = s_gc[7 + i]; o[10 + nj + i] = s_gv[6 + i]; }
      if (args.peer_world > 0) {   // fused all-gather: the finished row goes to every GPU of the job (this one included) over NVLink
        __syncwarp();
        const size_t row = ((size_t)args.peer_rank * args.num_envs + env) * args.ob_dim;
#pragma unroll 1
        for (int i = lane; i < args.ob_dim; i += 32) {
          const float v = o[i];                                          // re-read of this warp's own row (L2 hit), once for all peers
#pragma unroll 1
          for (int pr = 0; pr < args.peer_world; pr++) args.peer_obs[pr][row + i] = v;
        }
      }
    }
    if (args.phase_mask & 4) { __syncwarp(); continue; }   // kinematics only: contact records, iteration counts and flags of the last integrate() stay
    {   // failure detection: a non-finite coordinate or velocity marks the environment as diverged
      bool bad = false;
#pragma unroll 1
      for (int i = lane; i < nq; i += 32) bad |= !isfinite(s_gc[i]);
#pragma unroll 1
      for (int i = lane; i < nv; i += 32) bad |= !isfinite(s_gv[i]);
      const bool any_bad = __any_sync(FULL, bad);
      if (lane == 0) args.diverged[env] = any_bad ? 1 : 0;
    }
    if (lane == 0) { args.ncontacts[env] = K; args.iters[env] = iters; args.resid[env] = resid; args.solver_status[env] = gs_status; }
    if (lane < KMAX) {
      rsb_contact rc;
      int pt = -1;
      if (lane < K) {
        const float* ct = s_ct + lane * CT_WORDS;
        float lx = 0.f, ly = 0.f, lz = 0.f;
        if (!(args.phase_mask & 1)) { lx = s_lam[3 * lane]; ly = s_lam[3 * lane + 1]; lz = s_lam[3 * lane + 2]; }
        rc.local_body = __float_as_int(ct[CF_BODY]); rc.pair_index = __float_as_int(ct[CF_PAIR]);
        pt = __float_as_int(ct[CF_PT]);
#pragma unroll
        for (int k = 0; k < 3; k++) {
          rc.position[k] = ct[CF_POS + k]; rc.normal[k] = ct[CF_N + k];
          rc.impulse[k] = ct[CF_T1 + k] * lx + ct[CF_T2 + k] * ly + ct[CF_N + k] * lz;
        }
        rc.depth = ct[CF_DEPTH];
      } else {
        rc.local_body = -1; rc.pair_index = -1; rc.depth = 0.f;
#pragma unroll
        for (int k = 0; k < 3; k++) { rc.position[k] = 0.f; rc.normal[k] = 0.f; rc.impulse[k] = 0.f; }
      }
      args.contacts[(size_t)env * KMAX + lane] = rc;
      args.contact_pt[(size_t)env * KMAX + lane] = pt;
    }
    __syncwarp();
  }
  if (args.peer_world > 0 && args.obs) {
    // every row this CTA stored must be visible on the peers before they see the arrival count: the CTA barrier orders the warps'
    // stores before the signalling threads, whose release at system scope is cumulative over them (one fence per signalling
    // thread instead of one per thread of the CTA)
    __syncthreads();
    if ((int)threadIdx.x < args.peer_world)
      asm volatile("red.release.sys.global.add.u32 [%0], %1;" ::"l"(args.peer_flag[threadIdx.x] + args.peer_rank), "r"(1u) : "memory");
    if (args.peer_done) {
      // the arrival wait folded into the launch: the last CTA to finish stays until every rank's rows of this step have landed in
      // THIS GPU's buffer, so the launch completes exactly when the gathered rows do (no separate wait kernel, no launch gap).
      // Bounded: a dead peer traps instead of hanging the GPU.
      __shared__ int s_last;
      if (threadIdx.x == 0) {
        const unsigned d = atomicAdd(args.peer_done, 1u);
        s_last = d == gridDim.x - 1 ? 1 : 0;
        if (s_last) *args.peer_done = 0u;           // every CTA has counted itself: ready for the next launch
      }
      __syncthreads();
      if (s_last && (int)threadIdx.x < args.peer_world) {
        const unsigned* f = args.peer_flag[args.peer_rank] + threadIdx.x;
        const long long t0 = clock64();
        for (;;) {
          unsigned v;
          asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(f) : "memory");
          if ((int)(v - args.peer_expected) >= 0) break;
          if (clock64() - t0 > 20000000000ll) __trap();
        }
      }
    }
  }
}

}  // namespace rsb
