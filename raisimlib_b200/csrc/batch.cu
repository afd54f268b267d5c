// C-ABI implementation (include/rsb.h): batch memory, model-constant blob, kernel launches.
// No CPU fallback: every compute entry point launches the sm_100a kernel or fails loudly.
#include <cuda_runtime.h>

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include "model.hpp"
#include "step_kernel.cuh"
#include "aux_kernels.cuh"
#include "terrain_query.cuh"

using namespace rsb;

static thread_local std::string g_err;
static int fail(int code, const std::string& msg) { g_err = msg; return code; }
#define CK(call)                                                                                           \
  do {                                                                                                     \
    cudaError_t e_ = (call);                                                                               \
    if (e_ != cudaSuccess) return fail(RSB_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); \
  } while (0)

struct rsb_model { Model md; };

struct rsb_batch {
  const rsb_model* model = nullptr;
  int N = 0, device = 0;
  int nq = 0, nv = 0, nb = 0;
  int gc_stride = 0, gv_stride = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  rsb_params prm{};
  int control_mode = RSB_PD_PLUS_FEEDFORWARD_TORQUE;
  bool pd_set = false;
  const float* pt_bound = nullptr;   // caller-owned device buffer read in place of the internal PD-target rows
  int pt_bound_stride = 0;
  const float* vt_bound = nullptr;   // same for the velocity targets
  int vt_bound_stride = 0;
  bool pt_once = false, vt_once = false;   // zero-copy control step: the kernel copies the rows it read into pt / vt, then THAT binding ends
  // fused observation all-gather over NVLink peer memory (rsb_batch_set_observation_peers)
  int peer_world = 0, peer_rank = 0;
  float* peer_obs[MAX_PEERS][2] = {};     // [peer][buffer parity]: gathered-rows buffers, double-buffered by control step
  unsigned* peer_flag[MAX_PEERS] = {};    // [peer]: arrival counters [world]
  unsigned peer_epoch = 0;                // control steps signalled so far
  unsigned* peer_done = nullptr;          // device counter of finished CTAs (in-kernel arrival wait)
  bool kin_dirty = true;             // the getters' buffers (M, h, poses) do not describe the current state
  unsigned* prof = nullptr;          // rsb_internal_set_profile
  int* hmap_index = nullptr;         // terrain atlas: map index per environment
  float* ext = nullptr;              // [N][EXT_WORDS] external wrench rows; ext_active: rows hold a wrench for the next launch
  bool ext_active = false;
  // device buffers
  float *gc = nullptr, *gv = nullptr, *tau = nullptr, *pt = nullptr, *vt = nullptr, *tau_applied = nullptr;
  int *ncontacts = nullptr, *contact_pt = nullptr, *iters = nullptr, *diverged = nullptr;
  float* resid = nullptr;
  int* solver_status = nullptr;
  rsb_contact* contacts = nullptr;
  float *dbg_M = nullptr, *dbg_h = nullptr, *dbg_R = nullptr, *dbg_p = nullptr;
  float* hmap = nullptr;
  float* staging = nullptr;      // tight-row staging for host<->device repacking (staging_slice)
  size_t staging_words = 0, staging_cursor = 0;
  float* host_out = nullptr;     // results bound for host memory (and world rays in): every user synchronises before it returns
  size_t host_out_words = 0;
  uint32_t* blob = nullptr;
  std::vector<uint32_t> blob_host;
  BlobHeader hdr{};
  Dims dims{};
  WsLayout ws{};
  int spec = 0;                  // 0 generic, 1 quadruped-12 static dims, 2 humanoid-30 static dims
  int slots = 1;
  TerrainDesc ter{};
  std::vector<float> kp, kd;
  int wpc = 0, grid = 0;
  size_t smem_bytes = 0;
  int64_t launches = 0;
  // RaisimGym task state (rsb_batch_gym_*)
  float* gym_const = nullptr;     // device: gc_init | gv_init | action_mean | action_std
  GymConfig gym{};
  bool gym_ready = false;
  float *gym_action = nullptr, *gym_obs = nullptr, *gym_reward = nullptr;
  unsigned char* gym_done = nullptr;
  // terrain sensing (rsb_batch_height_scan / rsb_batch_ray_test)
  float2* hm_tiles = nullptr;        // per-tile height range of every map, kept beside the map (TqTiles)
  TqTiles tiles{};
  float* scan_pat = nullptr;         // device copies of the last height-scan / ray pattern, re-uploaded when the host arrays change
  float* ray_pat = nullptr;
  std::vector<float> scan_pat_host, ray_pat_host;
  size_t scan_pat_cap = 0, ray_pat_cap = 0;
};

static int round_up(int x, int m) { return (x + m - 1) / m * m; }

// ------------------------------------------------------------------ blob ------------------------
static void build_blob(rsb_batch* b) {
  const Model& md = b->model->md;
  BlobHeader& H = b->hdr;
  // dof tree: a floating base is a chain of 6 dofs; dof order is DFS pre-order so subtrees are contiguous
  const int nv = md.nv;
  std::vector<int> dparent(std::max(1, nv), -1), ddepth(std::max(1, nv), 0), dsub(std::max(1, nv), 1), dbody(std::max(1, nv), 0), bdof(md.nb, -1);
  const int nbase = md.floating ? 6 : 0;
  for (int k = 1; k < nbase; k++) dparent[k] = k - 1;
  if (md.floating) bdof[0] = 5;
  for (int i = 1; i < md.nb; i++) {
    bdof[i] = md.vidx[i]; dbody[md.vidx[i]] = i;
    dparent[md.vidx[i]] = bdof[md.parent[i]];
  }
  int maxdd = 0;
  for (int i = 0; i < nv; i++) { ddepth[i] = dparent[i] >= 0 ? ddepth[dparent[i]] + 1 : 0; maxdd = std::max(maxdd, ddepth[i]); }
  for (int i = nv - 1; i > 0; i--) if (dparent[i] >= 0) dsub[dparent[i]] += dsub[i];
  const int DL = maxdd + 1;
  std::vector<int> lvl(DL + 1, 0), lvldofs, entstart(DL + 1, 0), ent;
  for (int d = 0; d < DL; d++) {
    lvl[d] = (int)lvldofs.size(); entstart[d] = (int)ent.size();
    for (int i = 0; i < nv; i++) if (ddepth[i] == d) { lvldofs.push_back(i); for (int t = 0; t <= d; t++) ent.push_back(i | (t << 8)); }
  }
  lvl[DL] = (int)lvldofs.size(); entstart[DL] = (int)ent.size();
  b->dims = Dims{md.nb, md.nq, md.nv, md.floating, md.maxdepth, maxdd};
  H = make_blob_header(b->dims, md.npts(), (int)ent.size(), md.ncoll());
  {
    bool ident = true;
    for (int i = 1; i < md.nb; i++) for (int k = 0; k < 9; k++) if (std::fabs(md.jrot[9 * i + k] - ((k % 4 == 0) ? 1.0 : 0.0)) > 0.0) ident = false;
    int max_inner = 0;
    for (int i = 1; i < md.nb; i++) max_inner = std::max(max_inner, md.subtree[i] - 1);
    H.flags = (ident ? 1 : 0) | (max_inner << 8);
  }
  const int words = H.words;
  std::vector<uint32_t>& B = b->blob_host;
  B.assign(words, 0u);
  auto F = [&](int o, float v) { std::memcpy(&B[o], &v, 4); };
  auto I = [&](int o, int v) { std::memcpy(&B[o], &v, 4); };
  const int nbp = H.nbp;
  for (int i = 0; i < md.nb; i++) {
    I(H.off_body + BF_PARENT * nbp + i, md.parent[i]); I(H.off_body + BF_JTYPE * nbp + i, md.jtype[i]);
    I(H.off_body + BF_QIDX * nbp + i, md.qidx[i]); I(H.off_body + BF_VIDX * nbp + i, md.vidx[i]);
    I(H.off_body + BF_DEPTH * nbp + i, md.depth[i]); I(H.off_body + BF_SUBTREE * nbp + i, md.subtree[i]);
    for (int k = 0; k < 3; k++) F(H.off_body + (BF_JPOS + k) * nbp + i, (float)md.jpos[3 * i + k]);
    for (int k = 0; k < 9; k++) F(H.off_body + (BF_JROT + k) * nbp + i, (float)md.jrot[9 * i + k]);
    for (int k = 0; k < 3; k++) F(H.off_body + (BF_AXIS + k) * nbp + i, (float)md.axis[3 * i + k]);
    F(H.off_body + BF_MASS * nbp + i, (float)md.mass[i]);
    for (int k = 0; k < 3; k++) F(H.off_body + (BF_COM + k) * nbp + i, (float)md.com[3 * i + k]);
    for (int k = 0; k < 6; k++) F(H.off_body + (BF_INERTIA + k) * nbp + i, (float)md.inertia[6 * i + k]);
    F(H.off_body + BF_LO * nbp + i, (float)std::max(-3.0e38, md.jlimit[2 * i])); F(H.off_body + BF_HI * nbp + i, (float)std::min(3.0e38, md.jlimit[2 * i + 1]));
    // ancestor at depth d (d = 1..depth[i]) stored at anc[(d-1)*nbp + i]
    for (int d = 0; d < std::max(1, md.maxdepth); d++) I(H.off_anc + d * nbp + i, -1);
    for (int j = i; md.parent[j] >= 0; j = md.parent[j]) I(H.off_anc + (md.depth[j] - 1) * nbp + i, j);
  }
  for (int k = 0; k < md.npts(); k++) {
    I(H.off_pts + 0 * H.nptp + k, md.pt_body[k]);
    for (int q = 0; q < 3; q++) F(H.off_pts + (1 + q) * H.nptp + k, (float)md.pt_pos[3 * k + q]);
    F(H.off_pts + 4 * H.nptp + k, (float)md.pt_rad[k]);
    F(H.off_pts + 5 * H.nptp + k, -1.0f);
    I(H.off_pts + 6 * H.nptp + k, md.pt_type[k]);
    for (int q = 0; q < 3; q++) F(H.off_pts + (7 + q) * H.nptp + k, (float)md.pt_pos2[3 * k + q]);
    I(H.off_pts + 10 * H.nptp + k, md.pt_coll[k]);
    // bounding sphere of the candidate for the height cull of stage B: the sphere itself / the rim circle, the whole capsule, the whole box
    double cc[3] = {md.pt_pos[3 * k], md.pt_pos[3 * k + 1], md.pt_pos[3 * k + 2]}, cr = md.pt_rad[k];
    if (md.pt_type[k] == FT_SEGMENT) {
      double hl = 0;
      for (int q = 0; q < 3; q++) { cc[q] = 0.5 * (md.pt_pos[3 * k + q] + md.pt_pos2[3 * k + q]); const double d = md.pt_pos2[3 * k + q] - md.pt_pos[3 * k + q]; hl += d * d; }
      cr = md.pt_rad[k] + 0.5 * std::sqrt(hl);
    } else if (md.pt_type[k] == FT_BOXFACE) {
      const double* sz = &md.csize[3 * md.pt_coll[k]];
      cr = std::sqrt(sz[0] * sz[0] + sz[1] * sz[1] + sz[2] * sz[2]);
    }
    if (bdof[md.pt_body[k]] < 0) cr = -3.0e38;         // welded to the world: cannot collide
    for (int q = 0; q < 3; q++) F(H.off_pts + (11 + q) * H.nptp + k, (float)cc[q]);
    F(H.off_pts + 14 * H.nptp + k, (float)(cr * 1.0001 + 1e-6));   // float32 rounding of the product must never cull a touching candidate
  }
  for (int c = 0; c < md.ncoll(); c++) {   // collision-body table (box features): half extents, body-frame position and rotation
    for (int q = 0; q < 3; q++) { F(H.off_coll + COLL_WORDS * c + q, (float)md.csize[3 * c + q]); F(H.off_coll + COLL_WORDS * c + 3 + q, (float)md.cpos[3 * c + q]); }
    for (int q = 0; q < 9; q++) F(H.off_coll + COLL_WORDS * c + 6 + q, (float)md.crot[9 * c + q]);
  }
  for (int i = 0; i < md.nv; i++) {
    F(H.off_gain + i, b->kp[i]); F(H.off_gain + H.nvp + i, b->kd[i]); F(H.off_gain + 2 * H.nvp + i, 3.0e38f);
    I(H.off_dofq + i, -1);
  }
  for (int i = 1; i < md.nb; i++) F(H.off_gain + 2 * H.nvp + md.vidx[i], (float)std::min(md.jeffort[i], 3.0e38));   // actuator effort limit per dof
  for (int i = 1; i < md.nb; i++) I(H.off_dofq + md.vidx[i], md.qidx[i]);
  for (int i = 0; i < nv; i++) {
    I(H.off_ddepth + i, ddepth[i]); I(H.off_dsub + i, dsub[i]); I(H.off_dbody + i, dbody[i]);
    int a = i;
    for (int t = ddepth[i]; t >= 0; t--) { I(H.off_danc + t * H.nvp + i, a); a = dparent[a]; }
  }
  for (int i = 0; i < md.nb; i++) I(H.off_bdof + i, bdof[i]);
  for (int d = 0; d <= DL; d++) { I(H.off_lvl + d, lvl[d]); I(H.off_entstart + d, entstart[d]); }
  for (size_t k = 0; k < lvldofs.size(); k++) I(H.off_lvldofs + (int)k, lvldofs[k]);
  for (size_t k = 0; k < ent.size(); k++) I(H.off_ent + (int)k, ent[k]);
  {   // depth (in the dof tree) of the lowest common ancestor dof of two bodies; -1 when they share none
    int8_t* tab = reinterpret_cast<int8_t*>(&B[H.off_lcad]);
    for (int a = 0; a < md.nb; a++) for (int c = 0; c < md.nb; c++) {
      int x = a, y = c;
      while (x != y) { if (md.depth[x] >= md.depth[y]) x = md.parent[x]; else y = md.parent[y]; }
      tab[a * H.nbp + c] = (int8_t)(bdof[x] >= 0 ? ddepth[bdof[x]] : -1);
    }
  }
  for (int r = 0; r < NROUNDS; r++) {
    double width = 2.0 * M_PI / std::pow((double)NSEC, r);
    for (int k = 0; k <= NSEC; k++) {
      F(H.off_sec + r * SEC_STRIDE + k, (float)std::cos(width * k / NSEC));
      F(H.off_sec + NROUNDS * SEC_STRIDE + r * SEC_STRIDE + k, (float)std::sin(width * k / NSEC));
    }
  }
  std::memcpy(B.data(), &H, sizeof(H));
}

// ------------------------------------------------------------------ launches --------------------
// static specialisations: every 12-joint quadruped (ANYmal, A1, Go1, ...) shares (13,19,18,floating,3,8);
// the Atlas-like humanoid is (31,37,36,floating,10,15).  Anything else takes the generic kernel.
constexpr Dims kQuad12{13, 19, 18, 1, 3, 8};
constexpr Dims kHumanoid30{31, 37, 36, 1, 10, 15};
static bool same_dims(const Dims& a, const Dims& b) {
  return a.nb == b.nb && a.nq == b.nq && a.nv == b.nv && a.floating == b.floating && a.maxdepth == b.maxdepth && a.maxdd == b.maxdd;
}

template <int WPC, int SLOTS, int NB, int NQ, int NV, int FL, int MD, int MDD>
static cudaError_t launch_step(const StepArgs& a, int grid, size_t smem, cudaStream_t s) {
  auto kern = rsb_step_kernel<WPC, SLOTS, NB, NQ, NV, FL, MD, MDD>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  kern<<<grid, WPC * 32, smem, s>>>(a);
  return cudaGetLastError();
}

extern "C" int rsb_batch_ob_dim(const rsb_batch* b);

static int pick_config(rsb_batch* b) {
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, b->device));
  if (prop.major < 10) return fail(RSB_ERR_UNSUPPORTED, "raisimlib_b200 needs an sm_100a (B200) device; found sm_" + std::to_string(prop.major) + std::to_string(prop.minor));
  const size_t budget = prop.sharedMemPerBlockOptin;   // 227 KB on B200
  const size_t blob_bytes = (size_t)b->blob_host.size() * 4;
  const size_t per_warp = (size_t)b->ws.words * 4;
  const int sms = prop.multiProcessorCount;
  b->slots = b->model->md.npts() > 32 ? 2 : 1;
  // the quadruped instance has the topology compiled in (floating base + 4 serial chains of 3 joints in DFS order): check it
  bool quad_topology = same_dims(b->dims, kQuad12);
  if (quad_topology) {
    const Model& md = b->model->md;
    for (int leg = 0; leg < 4; leg++)
      for (int j = 0; j < 3; j++) {
        const int body = 1 + 3 * leg + j;
        if (md.parent[body] != (j == 0 ? 0 : body - 1) || md.vidx[body] != 5 + body || md.qidx[body] != 6 + body) quad_topology = false;
        if (md.jtype[body] != 1 && md.jtype[body] != 2) quad_topology = false;
      }
  }
  b->spec = quad_topology ? 1 : (same_dims(b->dims, kHumanoid30) ? 2 : 0);
  // Warps per CTA (= resident environments per CTA).  A round of w resident warps per SM costs ~ max(13, w): latency-bound up to a
  // dozen warps (32 k cycles per sub-step), issue-bound beyond (2.5 k cycles per warp; profiles/).  Choose the option with the
  // smallest rounds x cost, ties to the larger CTA (one sub-step barrier group, one copy of
  // the model block).  4096 ANYmal-like environments: 28 (one round).  4096 Atlas-like ones, whose 10.9 KB workspaces allow 16 per
  // SM: 14 (two balanced rounds: 0.98 ms per launch) rather than 16 (a full round and a 73 % one: 1.29 ms).
  static const int options[] = {28, 16, 14, 8, 4, 1};
  int best = 0; long best_cost = 0;
  for (int w : options) {
    const size_t cta_bytes = blob_bytes + (size_t)w * per_warp + 1024;
    if (cta_bytes > budget) continue;
    const int ctas = (w == 14 && 2 * cta_bytes <= (size_t)prop.sharedMemPerMultiprocessor) ? 2 : 1;   // 14-warp CTAs are compiled for two per SM
    const long resident = (long)sms * w * ctas;
    const long rounds = (b->N + resident - 1) / resident;
    const long cost = rounds * std::max(13L, (long)w * ctas);
    if (best == 0 || cost < best_cost) { best = w; best_cost = cost; }
  }
  if (best == 0) return fail(RSB_ERR_UNSUPPORTED, "model too large for one warp's shared-memory workspace");
  b->wpc = best;
  b->grid = std::min((b->N + best - 1) / best, best == 14 ? 2 * sms : sms);
  b->smem_bytes = blob_bytes + (size_t)best * per_warp;
  return RSB_OK;
}

template <int WPC>
static cudaError_t dispatch_spec(const rsb_batch* b, const StepArgs& a) {
  if (b->spec == 1 && b->slots == 1) return launch_step<WPC, 1, 13, 19, 18, 1, 3, 8>(a, b->grid, b->smem_bytes, b->stream);
  if (b->spec == 1) return launch_step<WPC, 2, 13, 19, 18, 1, 3, 8>(a, b->grid, b->smem_bytes, b->stream);
  if (b->spec == 2) return launch_step<WPC, 2, 31, 37, 36, 1, 10, 15>(a, b->grid, b->smem_bytes, b->stream);
  if (b->slots == 1) return launch_step<WPC, 1, 0, 0, 0, 0, 0, 0>(a, b->grid, b->smem_bytes, b->stream);
  return launch_step<WPC, 2, 0, 0, 0, 0, 0, 0>(a, b->grid, b->smem_bytes, b->stream);
}

struct GymLaunch { const float* action; float* reward; unsigned char* done; };   // rsb_batch_gym_step: the task fused into the step launch

static int do_launch(rsb_batch* b, int substeps, int phase_mask, bool debug, float* obs_dev = nullptr, bool peers = false, const GymLaunch* gym = nullptr) {
  StepArgs a{};
  a.num_envs = b->N; a.substeps = substeps;
  a.gc_stride = b->gc_stride; a.gv_stride = b->gv_stride;
  a.gc = b->gc; a.gv = b->gv; a.tau = b->tau;
  a.use_pd = (b->control_mode == RSB_PD_PLUS_FEEDFORWARD_TORQUE && b->pd_set) ? 1 : 0;
  a.ptarget = b->pt_bound ? b->pt_bound : b->pt; a.pt_stride = b->pt_bound ? b->pt_bound_stride : b->gc_stride;
  a.vtarget = b->vt_bound ? b->vt_bound : b->vt; a.vt_stride = b->vt_bound ? b->vt_bound_stride : b->gv_stride;
  a.pt_store = (b->pt_once && b->pt_bound) ? b->pt : nullptr;
  a.vt_store = (b->vt_once && b->vt_bound) ? b->vt : nullptr;
  a.prm = b->prm; a.ter = b->ter; a.ws = b->ws;
  a.blob_words = (int)b->blob_host.size(); a.blob = b->blob;
  a.tau_applied = b->tau_applied;
  a.ncontacts = b->ncontacts; a.contacts = b->contacts; a.contact_pt = b->contact_pt; a.iters = b->iters; a.diverged = b->diverged; a.resid = b->resid; a.solver_status = b->solver_status;
  if (debug) { a.dbg_M = b->dbg_M; a.dbg_h = b->dbg_h; a.dbg_R = b->dbg_R; a.dbg_p = b->dbg_p; }
  a.phase_mask = phase_mask; a.prof = b->prof;
  a.ext = b->ext_active ? b->ext : nullptr;
  a.obs = obs_dev; a.ob_dim = rsb_batch_ob_dim(b);
  if (gym) {       // targets come from the action rows and are kept in the batch's own rows; terminated environments get their reset target there too
    a.gym_action = gym->action; a.gym = b->gym; a.gym_reward = gym->reward; a.gym_done = gym->done;
    a.ptarget = b->pt; a.pt_stride = b->gc_stride; a.pt_store = b->pt;
  }
  if (peers && b->peer_world > 0 && obs_dev && phase_mask == 0) {
    a.peer_world = b->peer_world; a.peer_rank = b->peer_rank;
    for (int p = 0; p < b->peer_world; p++) { a.peer_obs[p] = b->peer_obs[p][b->peer_epoch & 1]; a.peer_flag[p] = b->peer_flag[p]; }
    b->peer_epoch++;
    a.peer_expected = b->peer_epoch * (unsigned)b->grid; a.peer_done = b->peer_done;
  }
  {
    const char* e = getenv("RSB_SUBSTEP_BARRIER");
    const int level = e ? atoi(e) : 1;
    a.substep_barrier = ((size_t)b->grid * b->wpc >= (size_t)b->N && phase_mask == 0) ? level : 0;
  }
  cudaError_t e;
  switch (b->wpc) {
    case 28: e = dispatch_spec<28>(b, a); break;
    case 16: e = dispatch_spec<16>(b, a); break;
    case 14: e = dispatch_spec<14>(b, a); break;
    case 8: e = dispatch_spec<8>(b, a); break;
    case 4: e = dispatch_spec<4>(b, a); break;
    default: e = dispatch_spec<1>(b, a); break;
  }
  if (e != cudaSuccess) return fail(RSB_ERR_CUDA, std::string("step kernel launch: ") + cudaGetErrorString(e));
  b->launches++;
  if (!(phase_mask & 1)) b->kin_dirty = !debug;   // the state advanced: M, h and poses are stale unless this launch refreshed them
  else if (debug) b->kin_dirty = false;
  if (phase_mask == 0 || (phase_mask & 2)) b->ext_active = false;   // an external wrench lasts for one integrate() call (upstream semantics)
  return RSB_OK;
}

// grows a batch-owned device buffer to at least `count` elements; work already on the stream may still use the old one
template <class T>
static int grow(rsb_batch* b, T*& buf, size_t& cap, size_t count) {
  if (cap >= count) return RSB_OK;
  if (buf) { CK(cudaStreamSynchronize(b->stream)); cudaFree(buf); buf = nullptr; cap = 0; }
  CK(cudaMalloc((void**)&buf, count * sizeof(T)));
  cap = count;
  return RSB_OK;
}
// the next `words` of the staging ring, or null (error recorded).  The ring is reused by back-to-back calls on the same stream:
// stream order keeps them apart.
static float* staging_slice(rsb_batch* b, size_t words) {
  if (grow(b, b->staging, b->staging_words, (size_t)b->N * 64 + 64)) return nullptr;
  float* st = b->staging + b->staging_cursor;
  b->staging_cursor = (b->staging_cursor + words + 31) / 32 * 32;
  if (b->staging_cursor + (size_t)b->N * 40 > b->staging_words) b->staging_cursor = 0;
  return st;
}
// device memory -> the caller's buffer (null: nothing to copy).  RSB_HOST returns with the copy complete; RSB_DEVICE stays
// stream-ordered.
static int read_back(rsb_batch* b, void* dst, const void* src, size_t bytes, int where) {
  if (dst && bytes) CK(cudaMemcpyAsync(dst, src, bytes, where == RSB_HOST ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice, b->stream));
  if (where == RSB_HOST) CK(cudaStreamSynchronize(b->stream));
  return RSB_OK;
}
// device-side alias of a pinned, mapped host allocation (cudaHostAlloc / cudaHostRegister / torch pin_memory); null otherwise
static const float* mapped_alias(const void* host) {
  cudaPointerAttributes at{};
  if (cudaPointerGetAttributes(&at, host) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  if (at.type == cudaMemoryTypeHost && at.devicePointer) return static_cast<const float*>(at.devicePointer);
  return nullptr;
}
// rows: tight [n][w] <-> padded [n][stride].  Host buffers go through one CONTIGUOUS PCIe copy into a
// device staging area and are (un)padded on the device: pitched H2D/D2H copies of 76-byte rows are slow.
static int copy_rows_in(rsb_batch* b, float* dst, int stride, const float* src, int w, int env_begin, int n, int where) {
  if (!src || n == 0) return RSB_OK;
  const float* dsrc = src;
  if (where == RSB_HOST) {
    float* st = staging_slice(b, (size_t)n * w);
    if (!st) return RSB_ERR_CUDA;
    CK(cudaMemcpyAsync(st, src, (size_t)n * w * 4, cudaMemcpyHostToDevice, b->stream));
    dsrc = st;
  }
  CK(cudaMemcpy2DAsync(dst + (size_t)env_begin * stride, (size_t)stride * 4, dsrc, (size_t)w * 4, (size_t)w * 4, n, cudaMemcpyDeviceToDevice, b->stream));
  return RSB_OK;
}
static int copy_rows_out(rsb_batch* b, float* dst, const float* src, int stride, int w, int env_begin, int n, int where) {
  float* rows = dst;
  if (dst && n > 0) {
    if (where == RSB_HOST && !(rows = staging_slice(b, (size_t)n * w))) return RSB_ERR_CUDA;
    CK(cudaMemcpy2DAsync(rows, (size_t)w * 4, src + (size_t)env_begin * stride, (size_t)stride * 4, (size_t)w * 4, n, cudaMemcpyDeviceToDevice, b->stream));
  }
  return where == RSB_HOST ? read_back(b, dst, rows, (size_t)n * w * 4, RSB_HOST) : RSB_OK;
}
// coarse grid of the ray test (terrain_query.cuh): [min, max] over the vertices of every TQ_TILE x TQ_TILE-cell tile of every map
static int build_tiles(rsb_batch* b, int count, int xs, int ys, const float* h) {
  const int nx = (xs - 1 + TQ_TILE - 1) / TQ_TILE, ny = (ys - 1 + TQ_TILE - 1) / TQ_TILE;
  std::vector<float2> mm((size_t)count * nx * ny);
  float lo = h[0], hi = h[0];
  for (int m = 0; m < count; m++)
    for (int ty = 0; ty < ny; ty++)
      for (int tx = 0; tx < nx; tx++) {
        const float* H = h + (size_t)m * xs * ys;
        float a = 3.0e38f, c = -3.0e38f;
        for (int iy = ty * TQ_TILE; iy <= std::min((ty + 1) * TQ_TILE, ys - 1); iy++)
          for (int ix = tx * TQ_TILE; ix <= std::min((tx + 1) * TQ_TILE, xs - 1); ix++) { a = std::min(a, H[(size_t)iy * xs + ix]); c = std::max(c, H[(size_t)iy * xs + ix]); }
        mm[((size_t)m * ny + ty) * nx + tx] = make_float2(a, c);
        lo = std::min(lo, a); hi = std::max(hi, c);
      }
  CK(cudaMalloc((void**)&b->hm_tiles, mm.size() * sizeof(float2)));
  CK(cudaMemcpy(b->hm_tiles, mm.data(), mm.size() * sizeof(float2), cudaMemcpyHostToDevice));
  b->tiles = TqTiles{b->hm_tiles, nx, ny, lo, hi};
  return RSB_OK;
}
// `count` same-sized height maps back to back and the map of every environment, or (map_of_env null) one map shared by all
static int install_heightmaps(rsb_batch* b, int count, int xs, int ys, float x_size, float y_size, float cx, float cy, const float* h,
                              const int32_t* map_of_env) {
  CK(cudaSetDevice(b->device));
  CK(cudaStreamSynchronize(b->stream));
  if (b->hmap) { cudaFree(b->hmap); b->hmap = nullptr; }
  if (b->hmap_index) { cudaFree(b->hmap_index); b->hmap_index = nullptr; }
  if (b->hm_tiles) { cudaFree(b->hm_tiles); b->hm_tiles = nullptr; }
  b->ter = TerrainDesc{};               // nothing may point at the freed maps if an allocation below fails
  const size_t words = (size_t)count * xs * ys;
  CK(cudaMalloc((void**)&b->hmap, words * 4));
  CK(cudaMemcpy(b->hmap, h, words * 4, cudaMemcpyHostToDevice));
  int rc = build_tiles(b, count, xs, ys, h); if (rc) return rc;
  TerrainDesc t{};
  if (map_of_env) {
    CK(cudaMalloc((void**)&b->hmap_index, (size_t)b->N * 4));
    CK(cudaMemcpy(b->hmap_index, map_of_env, (size_t)b->N * 4, cudaMemcpyHostToDevice));
    t.env_map = b->hmap_index; t.map_words = xs * ys;
  }
  t.type = 2; t.xs = xs; t.ys = ys;
  t.dx = x_size / (float)(xs - 1); t.dy = y_size / (float)(ys - 1); t.inv_dx = 1.0f / t.dx; t.inv_dy = 1.0f / t.dy;
  t.x0 = cx - 0.5f * x_size; t.y0 = cy - 0.5f * y_size;
  t.xmax = (float)(xs - 1); t.ymax = (float)(ys - 1);
  t.h = b->hmap;
  t.hmax = h[0];
  for (size_t i = 1; i < words; i++) t.hmax = std::max(t.hmax, h[i]);
  b->ter = t;
  return RSB_OK;
}
// a parsed model, once it fits the kernels (one lane per body, MAX_PT_SLOTS candidate slots per lane); parse errors become RSB_ERR_PARSE
static int adopt_model(Model (*load)(const std::string&), const char* path, rsb_model** out) {
  if (!path || !out) return fail(RSB_ERR_INVALID, "null argument");
  try {
    std::unique_ptr<rsb_model> m(new rsb_model);      // a parse error thrown below must not leak the half-built model
    m->md = load(path);
    if (m->md.nb > 32) return fail(RSB_ERR_UNSUPPORTED, "more than 32 movable bodies (one lane per body)");
    if (m->md.npts() > 32 * MAX_PT_SLOTS) return fail(RSB_ERR_UNSUPPORTED, "more than 64 candidate contact points");
    *out = m.release();
    return RSB_OK;
  } catch (const std::exception& e) { return fail(RSB_ERR_PARSE, e.what()); }
}
static int check_range(const rsb_batch* b, int env_begin, int env_count) {
  if (!b) return fail(RSB_ERR_INVALID, "null batch");
  if (env_begin < 0 || env_count < 0 || env_begin + env_count > b->N) return fail(RSB_ERR_INVALID, "environment range out of bounds");
  return RSB_OK;
}

extern "C" {

const char* rsb_last_error(void) { return g_err.c_str(); }
int rsb_version(void) { return 100; }

int rsb_params_default(rsb_params* p) {
  if (!p) return fail(RSB_ERR_INVALID, "null params");
  p->dt = 0.0025f; p->gravity[0] = 0.f; p->gravity[1] = 0.f; p->gravity[2] = -9.81f; p->erp = 0.f;
  p->alpha_init = 1.f; p->alpha_min = 1.f; p->alpha_decay = 1.f; p->max_iter = 150; p->threshold = 1e-6f;
  p->mu = 0.8f; p->restitution = 0.f; p->rest_threshold = 0.01f; p->stall_window = 8; p->stall_ratio = 0.5f; p->joint_limits = 1;
  p->accel_m = 2; p->accel_start = 6; p->stall_reg = 0.02f;
  return RSB_OK;
}

// ---- model ---------------------------------------------------------------------------------------
int rsb_model_create_from_urdf(const char* path_or_xml, rsb_model** out) { return adopt_model(load_urdf, path_or_xml, out); }
int rsb_model_save(const rsb_model* m, const char* path) {
  if (!m || !path) return fail(RSB_ERR_INVALID, "null argument");
  try { save_model(m->md, path); return RSB_OK; } catch (const std::exception& e) { return fail(RSB_ERR_PARSE, e.what()); }
}
int rsb_model_load(const char* path, rsb_model** out) { return adopt_model(load_model, path, out); }
void rsb_model_destroy(rsb_model* m) { delete m; }
int rsb_model_dims(const rsb_model* m, int* nq, int* nv, int* nb, int* ncoll, int* npts) {
  if (!m) return fail(RSB_ERR_INVALID, "null model");
  if (nq) *nq = m->md.nq; if (nv) *nv = m->md.nv; if (nb) *nb = m->md.nb; if (ncoll) *ncoll = m->md.ncoll(); if (npts) *npts = m->md.npts();
  return RSB_OK;
}
int rsb_model_get_tables(const rsb_model* m, rsb_model_tables* t) {
  if (!m || !t) return fail(RSB_ERR_INVALID, "null argument");
  const Model& d = m->md;
  t->nb = d.nb; t->nq = d.nq; t->nv = d.nv; t->floating = d.floating; t->ncoll = d.ncoll(); t->npts = d.npts();
  t->parent = d.parent.data(); t->jtype = d.jtype.data(); t->qidx = d.qidx.data(); t->vidx = d.vidx.data(); t->depth = d.depth.data();
  t->jpos = d.jpos.data(); t->jrot = d.jrot.data(); t->axis = d.axis.data(); t->mass = d.mass.data(); t->com = d.com.data();
  t->inertia = d.inertia.data(); t->jlimit = d.jlimit.data();
  t->cbody = d.cbody.data(); t->ctype = d.ctype.data(); t->csize = d.csize.data(); t->cpos = d.cpos.data(); t->crot = d.crot.data();
  t->pt_body = d.pt_body.data(); t->pt_coll = d.pt_coll.data(); t->pt_feat = d.pt_feat.data(); t->pt_pos = d.pt_pos.data(); t->pt_rad = d.pt_rad.data();
  t->pt_type = d.pt_type.data(); t->pt_pos2 = d.pt_pos2.data(); t->jeffort = d.jeffort.data();
  return RSB_OK;
}
int rsb_model_body_index(const rsb_model* m, const char* name) {
  if (!m || !name) return fail(RSB_ERR_INVALID, "null argument");
  for (int i = 0; i < m->md.nb; i++) if (m->md.body_names[i] == name) return i;
  for (const Frame& f : m->md.frames) if (f.name == name) return f.body;   // a link merged through a fixed joint
  return fail(RSB_ERR_INVALID, std::string("no body named '") + name + "'");
}
// collision bodies are named after the link that carries them, upstream style "LINK/k" for the k-th one ("LINK" = "LINK/0")
int rsb_model_collision_index(const rsb_model* m, const char* name) {
  if (!m || !name) return fail(RSB_ERR_INVALID, "null argument");
  std::string link = name; int which = 0;
  const size_t slash = link.rfind('/');
  if (slash != std::string::npos) { which = std::atoi(link.c_str() + slash + 1); link.resize(slash); }
  int seen = 0;
  for (int c = 0; c < m->md.ncoll(); c++) if (m->md.coll_names[c] == link) { if (seen == which) return c; seen++; }
  return fail(RSB_ERR_INVALID, std::string("no collision body named '") + name + "'");
}
const char* rsb_model_body_name(const rsb_model* m, int body) { return (m && body >= 0 && body < m->md.nb) ? m->md.body_names[body].c_str() : nullptr; }
const char* rsb_model_joint_name(const rsb_model* m, int body) { return (m && body >= 0 && body < m->md.nb) ? m->md.joint_names[body].c_str() : nullptr; }
int rsb_model_frame_index(const rsb_model* m, const char* name) {
  if (!m || !name) return fail(RSB_ERR_INVALID, "null argument");
  for (size_t i = 0; i < m->md.frames.size(); i++) if (m->md.frames[i].name == name) return (int)i;
  for (size_t i = 0; i < m->md.frames.size(); i++) if (!m->md.frames[i].joint.empty() && m->md.frames[i].joint == name) return (int)i;   // joint-name alias
  return fail(RSB_ERR_INVALID, std::string("no frame named '") + name + "'");
}
int rsb_model_frame(const rsb_model* m, int frame, int* body, double pos[3], double rot[9]) {
  if (!m || frame < 0 || frame >= (int)m->md.frames.size()) return fail(RSB_ERR_INVALID, "bad frame index");
  const Frame& f = m->md.frames[frame];
  if (body) *body = f.body;
  if (pos) for (int k = 0; k < 3; k++) pos[k] = f.pos[k];
  if (rot) for (int k = 0; k < 9; k++) rot[k] = f.rot[k];
  return RSB_OK;
}

// ---- batch ---------------------------------------------------------------------------------------
int rsb_batch_create(const rsb_model* m, int num_envs, int device, rsb_batch** out) {
  if (!m || !out || num_envs <= 0) return fail(RSB_ERR_INVALID, "bad arguments to rsb_batch_create");
  int ndev = 0;
  cudaError_t e0 = cudaGetDeviceCount(&ndev);
  if (e0 != cudaSuccess || ndev == 0) return fail(RSB_ERR_CUDA, "no CUDA device: raisimlib_b200 has no CPU fallback");
  if (device < 0 || device >= ndev) return fail(RSB_ERR_INVALID, "device index out of range");
  CK(cudaSetDevice(device));
  rsb_batch* b = new rsb_batch;
  b->model = m; b->N = num_envs; b->device = device;
  const Model& md = m->md;
  b->nq = md.nq; b->nv = md.nv; b->nb = md.nb;
  b->gc_stride = round_up(std::max(1, md.nq), 8); b->gv_stride = round_up(std::max(1, md.nv), 8);   // 32-byte sector-aligned rows
  rsb_params_default(&b->prm);
  b->kp.assign(std::max(1, md.nv), 0.f); b->kd.assign(std::max(1, md.nv), 0.f);
  build_blob(b);
  b->ws = make_ws_layout(b->dims);
  int rc = pick_config(b);
  if (rc != RSB_OK) { delete b; return rc; }
  size_t N = (size_t)num_envs;
  auto alloc = [&](void** p, size_t bytes) { cudaError_t e = cudaMalloc(p, std::max<size_t>(bytes, 16)); if (e == cudaSuccess) e = cudaMemset(*p, 0, std::max<size_t>(bytes, 16)); return e; };
  cudaError_t e = cudaSuccess;
  if (e == cudaSuccess) e = alloc((void**)&b->gc, N * b->gc_stride * 4);
  if (e == cudaSuccess) e = alloc((void**)&b->gv, N * b->gv_stride * 4);
  if (e == cudaSuccess) e = alloc((void**)&b->tau, N * b->gv_stride * 4);
  if (e == cudaSuccess) e = alloc((void**)&b->pt, N * b->gc_stride * 4);
  if (e == cudaSuccess) e = alloc((void**)&b->vt, N * b->gv_stride * 4);
  if (e == cudaSuccess) e = alloc((void**)&b->tau_applied, N * b->gv_stride * 4);
  if (e == cudaSuccess) e = alloc((void**)&b->ncontacts, N * 4);
  if (e == cudaSuccess) e = alloc((void**)&b->contact_pt, N * KMAX * 4);
  if (e == cudaSuccess) e = alloc((void**)&b->iters, N * 4);
  if (e == cudaSuccess) e = alloc((void**)&b->diverged, N * 4);
  if (e == cudaSuccess) e = alloc((void**)&b->resid, N * 4);
  if (e == cudaSuccess) e = alloc((void**)&b->solver_status, N * 4);
  if (e == cudaSuccess) e = alloc((void**)&b->contacts, N * KMAX * sizeof(rsb_contact));
  if (e == cudaSuccess) e = alloc((void**)&b->blob, b->blob_host.size() * 4);
  if (e == cudaSuccess) e = cudaMemcpy(b->blob, b->blob_host.data(), b->blob_host.size() * 4, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&b->stream, cudaStreamNonBlocking);
  if (e != cudaSuccess) { std::string msg = cudaGetErrorString(e); rsb_batch_destroy(b); return fail(RSB_ERR_CUDA, "rsb_batch_create: " + msg); }
  b->own_stream = true;
  // identity quaternion so that a fresh batch is a valid state
  if (md.floating) {
    std::vector<float> q0((size_t)N * b->gc_stride, 0.f);
    for (size_t i = 0; i < N; i++) q0[i * b->gc_stride + 3] = 1.f;
    cudaMemcpy(b->gc, q0.data(), q0.size() * 4, cudaMemcpyHostToDevice);
  }
  *out = b;
  return RSB_OK;
}

void rsb_batch_destroy(rsb_batch* b) {
  if (!b) return;
  cudaSetDevice(b->device);
  if (b->stream) cudaStreamSynchronize(b->stream);
  for (void* p : {(void*)b->solver_status, (void*)b->resid, (void*)b->diverged, (void*)b->tau_applied, (void*)b->gc, (void*)b->gv, (void*)b->tau, (void*)b->pt, (void*)b->vt, (void*)b->ncontacts, (void*)b->contact_pt, (void*)b->iters,
                  (void*)b->contacts, (void*)b->dbg_M, (void*)b->dbg_h, (void*)b->dbg_R, (void*)b->dbg_p, (void*)b->hmap, (void*)b->staging, (void*)b->host_out, (void*)b->blob, (void*)b->gym_const, (void*)b->gym_action,
                  (void*)b->gym_obs, (void*)b->gym_reward, (void*)b->gym_done, (void*)b->ext, (void*)b->hmap_index, (void*)b->peer_done,
                  (void*)b->hm_tiles, (void*)b->scan_pat, (void*)b->ray_pat})
    if (p) cudaFree(p);
  if (b->own_stream && b->stream) cudaStreamDestroy(b->stream);
  delete b;
}

int rsb_batch_set_stream(rsb_batch* b, void* s) {
  if (!b) return fail(RSB_ERR_INVALID, "null batch");
  CK(cudaStreamSynchronize(b->stream));
  if (b->own_stream) { cudaStreamDestroy(b->stream); b->own_stream = false; }
  b->stream = (cudaStream_t)s;
  return RSB_OK;
}
int rsb_batch_sync(rsb_batch* b) {
  if (!b) return fail(RSB_ERR_INVALID, "null batch");
  CK(cudaStreamSynchronize(b->stream));
  return RSB_OK;
}
int rsb_batch_num_envs(const rsb_batch* b) { return b ? b->N : 0; }

int rsb_batch_set_ground(rsb_batch* b, float z) {
  if (!b) return fail(RSB_ERR_INVALID, "null batch");
  b->ter = TerrainDesc{}; b->ter.type = 1; b->ter.ground_z = z;
  return RSB_OK;
}
int rsb_batch_clear_terrain(rsb_batch* b) {
  if (!b) return fail(RSB_ERR_INVALID, "null batch");
  b->ter = TerrainDesc{};
  return RSB_OK;
}
int rsb_batch_set_heightmap(rsb_batch* b, int xs, int ys, float x_size, float y_size, float cx, float cy, const float* h) {
  if (!b || !h || xs < 2 || ys < 2 || !(x_size > 0) || !(y_size > 0)) return fail(RSB_ERR_INVALID, "bad height map");
  return install_heightmaps(b, 1, xs, ys, x_size, y_size, cx, cy, h, nullptr);
}
// terrain atlas (SURVEY 8f N3 "per-env distinct terrains"): `count` same-sized height maps back to back and one map
// index per environment; every environment collides with its own map, everything else is as rsb_batch_set_heightmap
int rsb_batch_set_heightmaps(rsb_batch* b, int count, int xs, int ys, float x_size, float y_size, float cx, float cy, const float* h,
                             const int32_t* map_of_env) {
  if (!b || !h || !map_of_env || count < 1 || xs < 2 || ys < 2 || !(x_size > 0) || !(y_size > 0)) return fail(RSB_ERR_INVALID, "bad height-map atlas");
  if ((size_t)count * xs * ys > ((size_t)1 << 30)) return fail(RSB_ERR_INVALID, "height-map atlas too large");
  for (int e = 0; e < b->N; e++) if (map_of_env[e] < 0 || map_of_env[e] >= count) return fail(RSB_ERR_INVALID, "height-map index out of range");
  return install_heightmaps(b, count, xs, ys, x_size, y_size, cx, cy, h, map_of_env);
}
int rsb_batch_set_params(rsb_batch* b, const rsb_params* p) {
  if (!b || !p) return fail(RSB_ERR_INVALID, "null argument");
  if (!(p->dt > 0) || p->max_iter < 1 || !(p->mu >= 0)) return fail(RSB_ERR_INVALID, "invalid params");
  if (p->accel_m != 0 && p->accel_m != 2) return fail(RSB_ERR_INVALID, "accel_m must be 0 (plain sweeps) or 2");
  if (p->accel_m == 2 && p->accel_start < 3) return fail(RSB_ERR_INVALID, "accel_start must be at least 3");
  if (!(p->stall_reg >= 0.f)) return fail(RSB_ERR_INVALID, "stall_reg must be >= 0");
  b->prm = *p;
  return RSB_OK;
}
int rsb_batch_get_params(const rsb_batch* b, rsb_params* p) {
  if (!b || !p) return fail(RSB_ERR_INVALID, "null argument");
  *p = b->prm;
  return RSB_OK;
}

int rsb_batch_set_state(rsb_batch* b, const float* gc, const float* gv, int env_begin, int env_count, int where) {
  int rc = check_range(b, env_begin, env_count); if (rc) return rc;
  b->kin_dirty = true;
  rc = copy_rows_in(b, b->gc, b->gc_stride, gc, b->nq, env_begin, env_count, where); if (rc) return rc;
  return copy_rows_in(b, b->gv, b->gv_stride, gv, b->nv, env_begin, env_count, where);
}
int rsb_batch_get_state(rsb_batch* b, float* gc, float* gv, int env_begin, int env_count, int where) {
  int rc = check_range(b, env_begin, env_count); if (rc) return rc;
  rc = copy_rows_out(b, gc, b->gc, b->gc_stride, b->nq, env_begin, env_count, where); if (rc) return rc;
  return copy_rows_out(b, gv, b->gv, b->gv_stride, b->nv, env_begin, env_count, where);
}
int rsb_batch_set_pd_gains(rsb_batch* b, const float* kp, const float* kd) {
  if (!b || !kp || !kd) return fail(RSB_ERR_INVALID, "null argument");
  const Model& md = b->model->md;
  for (int i = 0; i < md.nv; i++) { b->kp[i] = kp[i]; b->kd[i] = kd[i]; }
  if (md.floating) for (int i = 0; i < 6; i++) { b->kp[i] = 0.f; b->kd[i] = 0.f; }   // the base is not actuated
  for (int i = 0; i < md.nv; i++) {
    std::memcpy(&b->blob_host[b->hdr.off_gain + i], &b->kp[i], 4);
    std::memcpy(&b->blob_host[b->hdr.off_gain + b->hdr.nvp + i], &b->kd[i], 4);
  }
  CK(cudaMemcpyAsync(b->blob + b->hdr.off_gain, b->blob_host.data() + b->hdr.off_gain, (size_t)2 * b->hdr.nvp * 4, cudaMemcpyHostToDevice, b->stream));
  CK(cudaStreamSynchronize(b->stream));
  b->pd_set = true;
  return RSB_OK;
}
// friction coefficient of one collision body against the terrain (mu < 0 restores the default material):
// the per-body half of World::setMaterialPairProp / CollisionDefinition::setMaterial
int rsb_batch_set_collision_friction(rsb_batch* b, int collision_body, float mu) {
  if (!b) return fail(RSB_ERR_INVALID, "null batch");
  const Model& md = b->model->md;
  if (collision_body < 0 || collision_body >= md.ncoll()) return fail(RSB_ERR_INVALID, "collision body index out of range");
  const BlobHeader& H = b->hdr;
  for (int k = 0; k < md.npts(); k++) if (md.pt_coll[k] == collision_body) std::memcpy(&b->blob_host[H.off_pts + 5 * H.nptp + k], &mu, 4);
  CK(cudaMemcpyAsync(b->blob + H.off_pts + 5 * H.nptp, b->blob_host.data() + H.off_pts + 5 * H.nptp, (size_t)H.nptp * 4, cudaMemcpyHostToDevice, b->stream));
  CK(cudaStreamSynchronize(b->stream));
  return RSB_OK;
}
int rsb_batch_set_pd_target(rsb_batch* b, const float* ptarget, const float* vtarget, int env_begin, int env_count, int where) {
  int rc = check_range(b, env_begin, env_count); if (rc) return rc;
  if (ptarget) b->pt_bound = nullptr;     // copying targets in ends a zero-copy binding
  rc = copy_rows_in(b, b->pt, b->gc_stride, ptarget, b->nq, env_begin, env_count, where); if (rc) return rc;
  return copy_rows_in(b, b->vt, b->gv_stride, vtarget, b->nv, env_begin, env_count, where);
}
int rsb_batch_bind_pd_target(rsb_batch* b, const float* ptarget_device, int row_stride) {
  if (!b) return fail(RSB_ERR_INVALID, "null batch");
  if (ptarget_device && row_stride < b->nq) return fail(RSB_ERR_INVALID, "row stride smaller than nq");
  b->pt_bound = ptarget_device; b->pt_bound_stride = row_stride;
  return RSB_OK;
}
int rsb_batch_set_generalized_force(rsb_batch* b, const float* tau, int env_begin, int env_count, int where) {
  int rc = check_range(b, env_begin, env_count); if (rc) return rc;
  return copy_rows_in(b, b->tau, b->gv_stride, tau, b->nv, env_begin, env_count, where);
}
int rsb_batch_get_generalized_force(rsb_batch* b, float* tau, int env_begin, int env_count, int where) {
  int rc = check_range(b, env_begin, env_count); if (rc) return rc;
  return copy_rows_out(b, tau, b->tau_applied, b->gv_stride, b->nv, env_begin, env_count, where);
}
// ArticulatedSystem::setExternalForce / setExternalTorque for a range of environments: one wrench per environment,
// acting on `body` at `point_body` (body frame; null = body origin), world-frame force / torque rows (null = zero).
// It acts during the next integrate() / control-step call (all of its fused sub-steps) and is cleared afterwards.
int rsb_batch_set_external_wrench(rsb_batch* b, int body, const float* force, const float* torque, const float* point_body, int env_begin, int env_count, int where) {
  int rc = check_range(b, env_begin, env_count); if (rc) return rc;
  if (body < 0 || body >= b->nb) return fail(RSB_ERR_INVALID, "external wrench: body index out of range");
  if (env_count == 0) return RSB_OK;
  CK(cudaSetDevice(b->device));
  if (!b->ext) CK(cudaMalloc((void**)&b->ext, (size_t)b->N * EXT_WORDS * 4));
  if (!b->ext_active) {   // rows of an earlier call are stale: body = -1 everywhere
    CK(cudaMemsetAsync(b->ext, 0xff, (size_t)b->N * EXT_WORDS * 4, b->stream));
    b->ext_active = true;
  }
  const float *df = force, *dtq = torque;
  if (where == RSB_HOST && (force || torque)) {
    float* st = staging_slice(b, (size_t)env_count * 6);
    if (!st) return RSB_ERR_CUDA;
    if (force) { CK(cudaMemcpyAsync(st, force, (size_t)env_count * 12, cudaMemcpyHostToDevice, b->stream)); df = st; }
    if (torque) { CK(cudaMemcpyAsync(st + (size_t)env_count * 3, torque, (size_t)env_count * 12, cudaMemcpyHostToDevice, b->stream)); dtq = st + (size_t)env_count * 3; }
  }
  const float px = point_body ? point_body[0] : 0.f, py = point_body ? point_body[1] : 0.f, pz = point_body ? point_body[2] : 0.f;
  const int threads = 128, blocks = (env_count + threads - 1) / threads;
  rsb_ext_pack_kernel<<<blocks, threads, 0, b->stream>>>(b->ext + (size_t)env_begin * EXT_WORDS, body, df, dtq, px, py, pz, env_count);
  CK(cudaGetLastError());
  return RSB_OK;
}
int rsb_batch_set_control_mode(rsb_batch* b, int mode) {
  if (!b || (mode != RSB_FORCE_AND_TORQUE && mode != RSB_PD_PLUS_FEEDFORWARD_TORQUE)) return fail(RSB_ERR_INVALID, "bad control mode");
  b->control_mode = mode;
  return RSB_OK;
}

static int ensure_debug(rsb_batch* b) {
  if (b->dbg_M) return RSB_OK;
  size_t N = (size_t)b->N;
  CK(cudaMalloc((void**)&b->dbg_M, std::max<size_t>(16, N * b->nv * b->nv * 4)));
  CK(cudaMalloc((void**)&b->dbg_h, std::max<size_t>(16, N * b->nv * 4)));
  CK(cudaMalloc((void**)&b->dbg_R, N * b->nb * 9 * 4));
  CK(cudaMalloc((void**)&b->dbg_p, N * b->nb * 3 * 4));
  return RSB_OK;
}

int rsb_batch_integrate1(rsb_batch* b) {
  if (!b) return fail(RSB_ERR_INVALID, "null batch");
  CK(cudaSetDevice(b->device));
  int rc = ensure_debug(b); if (rc) return rc;
  return do_launch(b, 1, 1, true);
}
int rsb_batch_update_kinematics(rsb_batch* b) {
  if (!b) return fail(RSB_ERR_INVALID, "null batch");
  CK(cudaSetDevice(b->device));
  int rc = ensure_debug(b); if (rc) return rc;
  return do_launch(b, 1, 1 | 4, true);      // stage A + the getters' buffers; contact records of the last integrate() untouched
}
// lazy getters: refresh M, h and the poses when the state changed through this API since they were last computed
static int ensure_kinematics(rsb_batch* b) {
  if (b->dbg_M && !b->kin_dirty) return RSB_OK;
  return rsb_batch_update_kinematics(b);
}
int rsb_batch_integrate2(rsb_batch* b) {
  if (!b) return fail(RSB_ERR_INVALID, "null batch");
  CK(cudaSetDevice(b->device));
  // state is unchanged since integrate1(), so the fused step recomputes stage A-B on-chip and goes on;
  // generalized forces / PD targets set between integrate1() and integrate2() are honoured
  return do_launch(b, 1, 0, b->dbg_M != nullptr);
}
int rsb_batch_integrate(rsb_batch* b, int substeps) {
  if (!b || substeps < 1) return fail(RSB_ERR_INVALID, "bad arguments to rsb_batch_integrate");
  CK(cudaSetDevice(b->device));
  return do_launch(b, substeps, 0, false);
}

int rsb_batch_get_mass_matrix(rsb_batch* b, int env_begin, int env_count, float* out, int where) {
  int rc = check_range(b, env_begin, env_count); if (rc) return rc;
  if (!out) return fail(RSB_ERR_INVALID, "null output buffer");
  if (env_count == 0) return RSB_OK;
  rc = ensure_kinematics(b); if (rc) return rc;
  const size_t w = (size_t)b->nv * b->nv;
  return read_back(b, out, b->dbg_M + env_begin * w, env_count * w * 4, where);
}
int rsb_batch_get_nonlinearities(rsb_batch* b, int env_begin, int env_count, float* out, int where) {
  int rc = check_range(b, env_begin, env_count); if (rc) return rc;
  if (!out) return fail(RSB_ERR_INVALID, "null output buffer");
  if (env_count == 0) return RSB_OK;
  rc = ensure_kinematics(b); if (rc) return rc;
  return read_back(b, out, b->dbg_h + (size_t)env_begin * b->nv, (size_t)env_count * b->nv * 4, where);
}
int rsb_batch_get_body_poses(rsb_batch* b, int env_begin, int env_count, float* rot, float* pos, int where) {
  int rc = check_range(b, env_begin, env_count); if (rc) return rc;
  if (env_count == 0) return RSB_OK;
  rc = ensure_kinematics(b); if (rc) return rc;
  rc = read_back(b, rot, b->dbg_R + (size_t)env_begin * b->nb * 9, (size_t)env_count * b->nb * 9 * 4, where); if (rc) return rc;
  return read_back(b, pos, b->dbg_p + (size_t)env_begin * b->nb * 3, (size_t)env_count * b->nb * 3 * 4, where);
}
int rsb_batch_get_contacts(rsb_batch* b, rsb_contact* out, int32_t* counts, int env_begin, int env_count, int where) {
  int rc = check_range(b, env_begin, env_count); if (rc) return rc;
  rc = read_back(b, out, b->contacts + (size_t)env_begin * KMAX, (size_t)env_count * KMAX * sizeof(rsb_contact), where); if (rc) return rc;
  return read_back(b, counts, b->ncontacts + env_begin, (size_t)env_count * 4, where);
}
int rsb_batch_get_contact_points(rsb_batch* b, int32_t* pt, int env_begin, int env_count, int where) {
  int rc = check_range(b, env_begin, env_count); if (rc) return rc;
  if (!pt) return fail(RSB_ERR_INVALID, "null output buffer");
  return read_back(b, pt, b->contact_pt + (size_t)env_begin * KMAX, (size_t)env_count * KMAX * 4, where);
}
int rsb_batch_get_solver_iterations(rsb_batch* b, int32_t* it, int env_begin, int env_count, int where) {
  int rc = check_range(b, env_begin, env_count); if (rc) return rc;
  if (!it) return fail(RSB_ERR_INVALID, "null output buffer");
  return read_back(b, it, b->iters + env_begin, (size_t)env_count * 4, where);
}
int rsb_batch_get_solver_status(rsb_batch* b, int32_t* status, int env_begin, int env_count, int where) {
  int rc = check_range(b, env_begin, env_count); if (rc) return rc;
  if (!status) return fail(RSB_ERR_INVALID, "null output buffer");
  return read_back(b, status, b->solver_status + env_begin, (size_t)env_count * 4, where);
}
int rsb_batch_get_solver_residual(rsb_batch* b, float* resid, int env_begin, int env_count, int where) {
  int rc = check_range(b, env_begin, env_count); if (rc) return rc;
  if (!resid) return fail(RSB_ERR_INVALID, "null output buffer");
  return read_back(b, resid, b->resid + env_begin, (size_t)env_count * 4, where);
}
int rsb_batch_get_diverged(rsb_batch* b, int32_t* flags, int env_begin, int env_count, int where) {
  int rc = check_range(b, env_begin, env_count); if (rc) return rc;
  if (!flags) return fail(RSB_ERR_INVALID, "null output buffer");
  return read_back(b, flags, b->diverged + env_begin, (size_t)env_count * 4, where);
}
int rsb_batch_device_ptrs(rsb_batch* b, rsb_device_view* v) {
  if (!b || !v) return fail(RSB_ERR_INVALID, "null argument");
  v->num_envs = b->N; v->nq = b->nq; v->nv = b->nv; v->gc_stride = b->gc_stride; v->gv_stride = b->gv_stride;
  v->gc = b->gc; v->gv = b->gv; v->tau_ff = b->tau; v->ptarget = b->pt; v->vtarget = b->vt;
  v->ncontacts = b->ncontacts; v->contacts = b->contacts;
  return RSB_OK;
}
int64_t rsb_batch_launch_count(const rsb_batch* b) { return b ? b->launches : 0; }

int rsb_batch_ob_dim(const rsb_batch* b) {
  if (!b) return 0;
  return b->model->md.floating ? (b->nq + b->nv - 3) : (b->nq + b->nv);
}
static int observe_impl(rsb_batch* b, float* obs, int env_begin, int env_count, int where) {
  const int od = rsb_batch_ob_dim(b);
  float* dst = obs;
  if (where == RSB_HOST) {
    int rc = grow(b, b->host_out, b->host_out_words, (size_t)b->N * od); if (rc) return rc;
    dst = b->host_out;
  }
  int threads = 128, blocks = (env_count * 32 + threads - 1) / threads;
  rsb_observe_kernel<<<blocks, threads, 0, b->stream>>>(b->gc + (size_t)env_begin * b->gc_stride, b->gv + (size_t)env_begin * b->gv_stride,
                                                         b->gc_stride, b->gv_stride, b->nq, b->nv, b->model->md.floating, env_count, dst, od);
  CK(cudaGetLastError());
  b->launches++;
  return where == RSB_HOST ? read_back(b, obs, dst, (size_t)env_count * od * 4, RSB_HOST) : RSB_OK;
}
int rsb_batch_observe(rsb_batch* b, float* obs, int env_begin, int env_count, int where) {
  int rc = check_range(b, env_begin, env_count); if (rc) return rc;
  if (!obs) return fail(RSB_ERR_INVALID, "null obs");
  if (env_count == 0) return RSB_OK;
  CK(cudaSetDevice(b->device));
  return observe_impl(b, obs, env_begin, env_count, where);
}

// VectorizedEnvironment::step() for the whole batch in ONE call: PD targets in, `substeps` fused
// World::integrate() calls, observation rows out.  Host buffers should be pinned (cudaHostAlloc /
// torch pin_memory) so that the copies overlap; the call returns after the observations have landed.
int rsb_batch_control_step(rsb_batch* b, const float* ptarget, const float* vtarget, int where_in, int substeps, float* obs, int where_out) {
  if (!b || substeps < 1) return fail(RSB_ERR_INVALID, "bad arguments to rsb_batch_control_step");
  CK(cudaSetDevice(b->device));
  // Host buffers in pinned (page-locked, mapped) memory are read and written IN PLACE by the step kernel over PCIe:
  // no staging copy, no separate H2D / D2H operations on the stream.  Pageable buffers take the staged path.
  int rc = RSB_OK;
  const float* pt_alias = (ptarget && where_in == RSB_HOST) ? mapped_alias(ptarget) : nullptr;
  const float* vt_alias = (vtarget && where_in == RSB_HOST) ? mapped_alias(vtarget) : nullptr;
  const bool pd_mode = b->control_mode == RSB_PD_PLUS_FEEDFORWARD_TORQUE && b->pd_set;
  // one-shot bindings end with this call; a persistent rsb_batch_bind_pd_target() binding the call did not replace survives it
  struct Unbind { rsb_batch* b; ~Unbind() { if (b->pt_once) { b->pt_bound = nullptr; b->pt_once = false; } if (b->vt_once) { b->vt_bound = nullptr; b->vt_once = false; } } } unbind{b};
  if (ptarget) {
    b->pt_bound = nullptr;
    if (pt_alias && pd_mode) { b->pt_bound = pt_alias; b->pt_bound_stride = b->nq; b->pt_once = true; }
    else { rc = copy_rows_in(b, b->pt, b->gc_stride, ptarget, b->nq, 0, b->N, where_in); if (rc) return rc; }
  }
  if (vtarget) {
    b->vt_bound = nullptr;
    if (vt_alias && pd_mode) { b->vt_bound = vt_alias; b->vt_bound_stride = b->nv; b->vt_once = true; }
    else { rc = copy_rows_in(b, b->vt, b->gv_stride, vtarget, b->nv, 0, b->N, where_in); if (rc) return rc; }
  }
  const bool bound_once = b->pt_once || b->vt_once;
  if (!obs || !b->model->md.floating) {
    rc = do_launch(b, substeps, 0, false); if (rc) return rc;
    if (obs) rc = observe_impl(b, obs, 0, b->N, where_out);
    if (bound_once) CK(cudaStreamSynchronize(b->stream));   // the caller may reuse its pinned target buffer on return
    return rc;
  }
  // observation rows are written by the step kernel itself (no separate observe launch): into the caller's device rows, straight
  // into its pinned host buffer as each environment finishes, or (pageable host memory) into host_out and then one copy
  float* dst = where_out == RSB_HOST ? const_cast<float*>(mapped_alias(obs)) : obs;
  const bool staged = !dst;
  const size_t obs_words = (size_t)b->N * rsb_batch_ob_dim(b);
  if (staged) {
    rc = grow(b, b->host_out, b->host_out_words, obs_words); if (rc) return rc;
    dst = b->host_out;
  }
  rc = do_launch(b, substeps, 0, false, dst, where_out == RSB_DEVICE); if (rc) return rc;
  if (staged) return read_back(b, obs, dst, obs_words * 4, RSB_HOST);
  if (where_out == RSB_HOST || bound_once) CK(cudaStreamSynchronize(b->stream));
  return RSB_OK;
}

// ---- terrain sensing: height scans and ray tests (terrain_query.cuh) ----
// frame records of a pattern (TQ_FRAME_WORDS each); *needs_kin: some frame's pose comes from the getters' pose buffers
static int pack_frames(const rsb_batch* b, const int32_t* frames, int num_frames, std::vector<float>& pat, bool* needs_kin) {
  const Model& md = b->model->md;
  *needs_kin = false;
  for (int f = 0; f < num_frames; f++) {
    if (frames[f] < 0 || frames[f] >= (int)md.frames.size()) return fail(RSB_ERR_INVALID, "bad frame index " + std::to_string(frames[f]));
    const Frame& fr = md.frames[frames[f]];
    float w[TQ_FRAME_WORDS] = {};
    std::memcpy(&w[0], &fr.body, 4);
    for (int k = 0; k < 3; k++) w[1 + k] = (float)fr.pos[k];
    for (int k = 0; k < 9; k++) w[4 + k] = (float)fr.rot[k];
    pat.insert(pat.end(), w, w + TQ_FRAME_WORDS);
    if (fr.body != 0 || !md.floating) *needs_kin = true;
  }
  return RSB_OK;
}
// device copy of a small host pattern; uploaded only when it differs from the last one (stream order keeps earlier readers safe)
static int upload_pattern(rsb_batch* b, const std::vector<float>& pat, std::vector<float>& last, float*& dev, size_t& cap) {
  if (dev && pat.size() == last.size() && std::memcmp(pat.data(), last.data(), pat.size() * 4) == 0) return RSB_OK;
  last.clear();            // a failed allocation or copy below must not leave a stale match behind
  int rc = grow(b, dev, cap, pat.size()); if (rc) return rc;
  CK(cudaMemcpyAsync(dev, pat.data(), pat.size() * 4, cudaMemcpyHostToDevice, b->stream));
  last = pat;
  return RSB_OK;
}
static TqPose tq_pose(const rsb_batch* b) { return TqPose{b->gc, b->gc_stride, b->dbg_R, b->dbg_p, b->nb, b->model->md.floating}; }

int rsb_batch_height_scan(rsb_batch* b, const int32_t* frames, int num_frames, const float* points_xy, int num_points,
                          float* out, int out_stride, int env_begin, int env_count, int where) {
  int rc = check_range(b, env_begin, env_count); if (rc) return rc;
  if (!frames || !points_xy || !out) return fail(RSB_ERR_INVALID, "height scan: null argument");
  if (num_frames < 1 || num_points < 1) return fail(RSB_ERR_INVALID, "height scan: num_frames and num_points must be >= 1");
  if ((long long)num_frames * num_points > (1 << 24)) return fail(RSB_ERR_INVALID, "height scan: more than 2^24 samples per environment");
  if (out_stride < num_frames * num_points) return fail(RSB_ERR_INVALID, "height scan: out_stride " + std::to_string(out_stride) + " < num_frames * num_points = " + std::to_string(num_frames * num_points));
  if (b->ter.type == 0) return fail(RSB_ERR_INVALID, "height scan: no terrain set (rsb_batch_set_ground / rsb_batch_set_heightmap)");
  std::vector<float> pat;
  bool needs_kin = false;
  rc = pack_frames(b, frames, num_frames, pat, &needs_kin); if (rc) return rc;
  for (int k = 0; k < 2 * num_points; k++) if (!std::isfinite(points_xy[k])) return fail(RSB_ERR_INVALID, "height scan: non-finite point");
  if (env_count == 0) return RSB_OK;
  CK(cudaSetDevice(b->device));
  pat.insert(pat.end(), points_xy, points_xy + 2 * (size_t)num_points);
  rc = upload_pattern(b, pat, b->scan_pat_host, b->scan_pat, b->scan_pat_cap); if (rc) return rc;
  if (needs_kin) { rc = ensure_kinematics(b); if (rc) return rc; }
  const int per_env = num_frames * num_points;
  float* dst = out; int stride = out_stride;
  if (where == RSB_HOST) { rc = grow(b, b->host_out, b->host_out_words, (size_t)env_count * per_env); if (rc) return rc; dst = b->host_out; stride = per_env; }
  const long long total = (long long)env_count * num_frames * ((num_points + TQ_SCAN_PPT - 1) / TQ_SCAN_PPT);
  rsb_height_scan_kernel<<<(unsigned)((total + 255) / 256), 256, 0, b->stream>>>(b->ter, tq_pose(b), b->scan_pat, num_frames, num_points, env_begin, env_count, dst, stride);
  CK(cudaGetLastError());
  b->launches++;
  if (where == RSB_HOST) {
    CK(cudaMemcpy2DAsync(out, (size_t)out_stride * 4, dst, (size_t)per_env * 4, (size_t)per_env * 4, env_count, cudaMemcpyDeviceToHost, b->stream));
    CK(cudaStreamSynchronize(b->stream));
  }
  return RSB_OK;
}

int rsb_batch_ray_test(rsb_batch* b, const int32_t* frames, int num_frames, const float* origins, const float* dirs, int num_rays,
                       float length, rsb_ray_hit* out, int env_begin, int env_count, int where) {
  int rc = check_range(b, env_begin, env_count); if (rc) return rc;
  if (!origins || !dirs || !out || (num_frames > 0 && !frames)) return fail(RSB_ERR_INVALID, "ray test: null argument");
  if (num_frames < 0 || num_rays < 1) return fail(RSB_ERR_INVALID, "ray test: num_frames must be >= 0 and num_rays >= 1");
  if ((long long)std::max(num_frames, 1) * num_rays > (1 << 24)) return fail(RSB_ERR_INVALID, "ray test: more than 2^24 rays per environment");
  if (!(length > 0.f) || !std::isfinite(length)) return fail(RSB_ERR_INVALID, "ray test: length must be finite and > 0");
  const bool host_rays = num_frames > 0 || where == RSB_HOST;
  const size_t nray_words = (size_t)3 * num_rays * (num_frames > 0 ? 1 : (size_t)env_count);
  if (host_rays)
    for (size_t r = 0; r < nray_words; r += 3) {
      const double n2 = (double)dirs[r] * dirs[r] + (double)dirs[r + 1] * dirs[r + 1] + (double)dirs[r + 2] * dirs[r + 2];
      if (!(n2 > 0.0) || !std::isfinite(n2)) return fail(RSB_ERR_INVALID, "ray test: zero or non-finite ray direction");
    }
  std::vector<float> pat;
  bool needs_kin = false;
  rc = pack_frames(b, frames, num_frames, pat, &needs_kin); if (rc) return rc;
  if (env_count == 0) return RSB_OK;
  CK(cudaSetDevice(b->device));
  const float *org = origins, *dir = dirs;
  const size_t out_bytes = (size_t)env_count * std::max(num_frames, 1) * num_rays * sizeof(rsb_ray_hit);
  const size_t in_words = (num_frames == 0 && where == RSB_HOST) ? 2 * nray_words : 0;
  rc = grow(b, b->host_out, b->host_out_words, in_words + (where == RSB_HOST ? out_bytes / 4 : 0)); if (rc) return rc;
  if (num_frames > 0) {
    pat.insert(pat.end(), origins, origins + 3 * (size_t)num_rays);
    for (int r = 0; r < num_rays; r++) {     // directions are normalised here, in double
      const double n = std::sqrt((double)dirs[3 * r] * dirs[3 * r] + (double)dirs[3 * r + 1] * dirs[3 * r + 1] + (double)dirs[3 * r + 2] * dirs[3 * r + 2]);
      for (int k = 0; k < 3; k++) pat.push_back((float)(dirs[3 * r + k] / n));
    }
    rc = upload_pattern(b, pat, b->ray_pat_host, b->ray_pat, b->ray_pat_cap); if (rc) return rc;
    if (needs_kin) { rc = ensure_kinematics(b); if (rc) return rc; }
    org = dir = nullptr;
  } else if (where == RSB_HOST) {
    float* st = b->host_out;
    CK(cudaMemcpyAsync(st, origins, nray_words * 4, cudaMemcpyHostToDevice, b->stream));
    CK(cudaMemcpyAsync(st + nray_words, dirs, nray_words * 4, cudaMemcpyHostToDevice, b->stream));
    org = st; dir = st + nray_words;
  }
  rsb_ray_hit* dst = where == RSB_HOST ? reinterpret_cast<rsb_ray_hit*>(b->host_out + in_words) : out;
  const long long total = (long long)env_count * std::max(num_frames, 1) * num_rays;
  rsb_ray_test_kernel<<<(unsigned)((total + 255) / 256), 256, 0, b->stream>>>(b->ter, b->tiles, tq_pose(b), b->ray_pat, num_frames, org, dir, num_rays, length,
                                                                            env_begin, env_count, dst);
  CK(cudaGetLastError());
  b->launches++;
  return where == RSB_HOST ? read_back(b, out, dst, out_bytes, RSB_HOST) : RSB_OK;
}

// ---- RaisimGym ANYmal task (SURVEY 8f N1): VectorizedEnvironment::{reset, step, observe} for the whole batch ----
int rsb_batch_gym_configure(rsb_batch* b, const float* gc_init, const float* gv_init, const float* action_mean, const float* action_std,
                            const int32_t* foot_bodies, int n_foot, float torque_coeff, float forward_vel_coeff, float terminal_reward) {
  if (!b || !gc_init || !gv_init || !action_mean || !action_std || (n_foot > 0 && !foot_bodies)) return fail(RSB_ERR_INVALID, "null argument");
  if (!b->model->md.floating) return fail(RSB_ERR_UNSUPPORTED, "the gym task needs a floating-base robot");
  CK(cudaSetDevice(b->device));
  const int nq = b->nq, nv = b->nv, nj = nq - 7;
  std::vector<float> h((size_t)nq + nv + 2 * nj);
  std::memcpy(h.data(), gc_init, nq * 4); std::memcpy(h.data() + nq, gv_init, nv * 4);
  std::memcpy(h.data() + nq + nv, action_mean, nj * 4); std::memcpy(h.data() + nq + nv + nj, action_std, nj * 4);
  // every buffer under its own check: a retry after a failed allocation finishes the set instead of skipping it
  if (!b->gym_const) CK(cudaMalloc((void**)&b->gym_const, h.size() * 4));
  if (!b->gym_action) CK(cudaMalloc((void**)&b->gym_action, (size_t)b->N * nj * 4));
  if (!b->gym_obs) CK(cudaMalloc((void**)&b->gym_obs, (size_t)b->N * rsb_batch_ob_dim(b) * 4));
  if (!b->gym_reward) CK(cudaMalloc((void**)&b->gym_reward, (size_t)b->N * 4));
  if (!b->gym_done) CK(cudaMalloc((void**)&b->gym_done, (size_t)b->N));
  CK(cudaMemcpyAsync(b->gym_const, h.data(), h.size() * 4, cudaMemcpyHostToDevice, b->stream));
  CK(cudaStreamSynchronize(b->stream));
  b->gym.gc_init = b->gym_const; b->gym.gv_init = b->gym_const + nq; b->gym.action_mean = b->gym_const + nq + nv; b->gym.action_std = b->gym_const + nq + nv + nj;
  b->gym.foot_mask = 0;
  for (int i = 0; i < n_foot; i++) {
    if (foot_bodies[i] < 0 || foot_bodies[i] >= b->nb) return fail(RSB_ERR_INVALID, "foot body index out of range");
    b->gym.foot_mask |= 1u << foot_bodies[i];
  }
  b->gym.torque_coeff = torque_coeff; b->gym.forward_vel_coeff = forward_vel_coeff; b->gym.terminal_reward = terminal_reward;
  b->gym_ready = true;
  return RSB_OK;
}

// ENVIRONMENT::reset() for every environment: state and PD target back to the initial configuration
int rsb_batch_gym_reset(rsb_batch* b) {
  if (!b || !b->gym_ready) return fail(RSB_ERR_INVALID, "call rsb_batch_gym_configure() first");
  CK(cudaSetDevice(b->device));
  int threads = 128, blocks = (b->N * 32 + threads - 1) / threads;
  rsb_gym_reset_kernel<<<blocks, threads, 0, b->stream>>>(b->gc, b->gv, b->pt, b->vt, b->gym, b->gc_stride, b->gv_stride, b->nq, b->nv, b->N);
  CK(cudaGetLastError());
  b->kin_dirty = true;
  b->launches++;
  return RSB_OK;
}

// VectorizedEnvironment::step(action, reward, done) + observe(ob): action rows [N][nq-7] in; `substeps` fused
// World::integrate() calls; reward [N], done [N] (uint8) and observation rows [N][ob_dim] out.
int rsb_batch_gym_step(rsb_batch* b, const float* action, int where_in, int substeps, float* obs, float* reward, unsigned char* done, int where_out) {
  if (!b || !b->gym_ready) return fail(RSB_ERR_INVALID, "call rsb_batch_gym_configure() first");
  if (!action || substeps < 1) return fail(RSB_ERR_INVALID, "bad arguments to rsb_batch_gym_step");
  CK(cudaSetDevice(b->device));
  const int nj = b->nq - 7, od = rsb_batch_ob_dim(b);
  b->pt_bound = nullptr;              // the task writes its own PD-target rows
  // pinned host buffers are read / written in place by the task kernels (see rsb_batch_control_step)
  const float* act = action;
  if (where_in == RSB_HOST) {
    act = mapped_alias(action);
    if (!act) {
      CK(cudaMemcpyAsync(b->gym_action, action, (size_t)b->N * nj * 4, cudaMemcpyHostToDevice, b->stream));
      act = b->gym_action;
    }
  }
  const bool host_out = where_out == RSB_HOST;
  float* a_obs = (host_out && obs) ? const_cast<float*>(mapped_alias(obs)) : nullptr;
  float* a_rew = (host_out && reward) ? const_cast<float*>(mapped_alias(reward)) : nullptr;
  unsigned char* a_done = (host_out && done) ? reinterpret_cast<unsigned char*>(const_cast<float*>(mapped_alias(done))) : nullptr;
  float* d_obs = a_obs ? a_obs : (host_out || !obs) ? b->gym_obs : obs;
  float* d_rew = a_rew ? a_rew : (host_out || !reward) ? b->gym_reward : reward;
  unsigned char* d_done = a_done ? a_done : (host_out || !done) ? b->gym_done : done;
  // ONE launch: action rows -> PD targets, `substeps` x World::integrate(), reward, isTerminalState(), reset() of the terminated
  // environments and the observation rows of the resulting state (the task used to be an action kernel and a post kernel around the step)
  if (!(b->control_mode == RSB_PD_PLUS_FEEDFORWARD_TORQUE && b->pd_set)) return fail(RSB_ERR_INVALID, "the gym task drives the robot through PD targets: call rsb_batch_set_pd_gains() first");
  const GymLaunch gl{act, d_rew, d_done};
  int rc = do_launch(b, substeps, 0, false, d_obs, false, &gl); if (rc) return rc;
  if (where_out == RSB_HOST) {
    if (obs && !a_obs) CK(cudaMemcpyAsync(obs, d_obs, (size_t)b->N * od * 4, cudaMemcpyDeviceToHost, b->stream));
    if (reward && !a_rew) CK(cudaMemcpyAsync(reward, d_rew, (size_t)b->N * 4, cudaMemcpyDeviceToHost, b->stream));
    if (done && !a_done) CK(cudaMemcpyAsync(done, d_done, (size_t)b->N, cudaMemcpyDeviceToHost, b->stream));
    CK(cudaStreamSynchronize(b->stream));
  } else if (where_in == RSB_HOST && act != b->gym_action) {
    CK(cudaStreamSynchronize(b->stream));   // the action rows were read in place from pinned host memory: the caller may reuse them on return
  }
  return RSB_OK;
}

// ---- fused observation all-gather over NVLink peer memory (SURVEY 8e; one process per GPU or one process for all) ----
// Buffers that other processes map: plain cudaMalloc memory + a CUDA IPC handle (64 bytes) to ship over any host channel.
int rsb_peer_buffer_create(int device, size_t bytes, void** dev_ptr, unsigned char* handle64) {
  if (!dev_ptr || bytes == 0) return fail(RSB_ERR_INVALID, "bad arguments to rsb_peer_buffer_create");
  CK(cudaSetDevice(device));
  void* p = nullptr;
  CK(cudaMalloc(&p, bytes));
  cudaError_t e = cudaMemset(p, 0, bytes);
  if (e == cudaSuccess && handle64) {
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle is 64 bytes");
    cudaIpcMemHandle_t h;
    e = cudaIpcGetMemHandle(&h, p);
    if (e == cudaSuccess) std::memcpy(handle64, &h, 64);
  }
  if (e != cudaSuccess) { cudaFree(p); return fail(RSB_ERR_CUDA, std::string("rsb_peer_buffer_create: ") + cudaGetErrorString(e)); }
  *dev_ptr = p;
  return RSB_OK;
}
int rsb_peer_buffer_open(int device, const unsigned char* handle64, void** dev_ptr) {
  if (!dev_ptr || !handle64) return fail(RSB_ERR_INVALID, "null argument");
  CK(cudaSetDevice(device));
  cudaIpcMemHandle_t h;
  std::memcpy(&h, handle64, 64);
  CK(cudaIpcOpenMemHandle(dev_ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return RSB_OK;
}
int rsb_peer_buffer_close(void* dev_ptr) { if (dev_ptr) CK(cudaIpcCloseMemHandle(dev_ptr)); return RSB_OK; }
int rsb_peer_buffer_destroy(void* dev_ptr) { if (dev_ptr) CK(cudaFree(dev_ptr)); return RSB_OK; }

// obs_all[2 * world]: for every rank r, its two gathered-rows buffers (parity 0, 1), each [world * num_envs][ob_dim] float32, as
// device pointers valid in THIS process (own allocations, IPC mappings, or peer-enabled pointers of other devices of this process);
// flags[world]: rank r's arrival counters, unsigned[world], zero-initialised.  From now on every control step that returns
// observation rows on the device also stores them into the buffer (step parity) of every rank and bumps flags[r][rank] once
// per finished CTA.  world = 0 switches the fused gather off.  Every rank must run the same num_envs.
int rsb_batch_set_observation_peers(rsb_batch* b, int world, int rank, void* const* obs_all, void* const* flags) {
  if (!b) return fail(RSB_ERR_INVALID, "null batch");
  if (world == 0) { b->peer_world = 0; return RSB_OK; }
  if (world < 1 || world > MAX_PEERS || rank < 0 || rank >= world || !obs_all || !flags) return fail(RSB_ERR_INVALID, "bad arguments to rsb_batch_set_observation_peers");
  if (!b->model->md.floating) return fail(RSB_ERR_UNSUPPORTED, "fused observation rows need a floating-base robot");
  for (int p = 0; p < world; p++) if (!obs_all[2 * p] || !obs_all[2 * p + 1] || !flags[p]) return fail(RSB_ERR_INVALID, "null peer buffer");
  CK(cudaSetDevice(b->device));
  CK(cudaStreamSynchronize(b->stream));
  b->peer_world = 0;                    // a failure below leaves the gather off
  if (!b->peer_done) CK(cudaMalloc(&b->peer_done, sizeof(unsigned)));
  CK(cudaMemsetAsync(b->peer_done, 0, sizeof(unsigned), b->stream));
  for (int p = 0; p < world; p++) { b->peer_obs[p][0] = (float*)obs_all[2 * p]; b->peer_obs[p][1] = (float*)obs_all[2 * p + 1]; b->peer_flag[p] = (unsigned*)flags[p]; }
  b->peer_world = world; b->peer_rank = rank; b->peer_epoch = 0;
  return RSB_OK;
}
// *buffer_parity (optional) = which of this rank's two buffers holds the rows of the LAST control step of every rank.  The arrival
// wait itself is part of that control step's launch (its last CTA stays until every rank's rows have landed), so in stream order
// after the step the rows are complete and nothing is enqueued here.
int rsb_batch_wait_observation_peers(rsb_batch* b, int* buffer_parity) {
  if (!b || b->peer_world <= 0 || b->peer_epoch == 0) return fail(RSB_ERR_INVALID, "no fused observation gather in flight");
  if (buffer_parity) *buffer_parity = (int)((b->peer_epoch - 1) & 1);
  return RSB_OK;
}

// ---- hooks for comm.cu -----------------------------------------------------------------------------
int rsb_internal_batch_info(rsb_batch* b, int* device, void** stream, int* num_envs) {
  if (!b) return fail(RSB_ERR_INVALID, "null batch");
  if (device) *device = b->device;
  if (stream) *stream = (void*)b->stream;
  if (num_envs) *num_envs = b->N;
  return RSB_OK;
}
// profiling hook (tools/balance_probe.py): device buffer [num_envs][4][8] of SM-clock stamps, or null to switch off
int rsb_internal_set_profile(rsb_batch* b, unsigned* dev) { if (!b) return -1; b->prof = dev; return 0; }
void rsb_internal_set_error(const char* msg) { g_err = msg ? msg : ""; }

}  // extern "C"
