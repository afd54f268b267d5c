// raisim::World / raisim::ArticulatedSystem / raisim::Contact -- header-only facade over the C-ABI
// (include/rsb.h).  Keeps the reference's API surface for the hot path so RaisimGym-style
// ENVIRONMENT code compiles against it (SURVEY.md 8b lists the upstream signatures, [RECALL]:
// include/raisim/World.hpp, object/ArticulatedSystem/ArticulatedSystem.hpp, contact/Contact.hpp;
// none of them is in the reference snapshot).
//
// Design inversion: the batch lives UNDER World.  A raisim::BatchedWorld owns N environments of
// SoA state on one GPU; raisim::World and raisim::ArticulatedSystem are thin per-environment VIEWS
// {batch, env index}.  A World constructed standalone owns a batch of one (config 1 semantics).
// VectorizedEnvironment.hpp issues ONE batched launch per control step instead of N OpenMP iterations.
//
// Errors: the reference aborts through RSFATAL; here every failing C-ABI call throws
// std::runtime_error with rsb_last_error() (define RAISIM_B200_ABORT_ON_ERROR to abort instead).
// Units and conventions are the reference's: gc = [xyz | qw qx qy qz | joints], gv = [v | w | joint rates].
#pragma once
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <functional>
#include <map>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include "../rsb.h"
#include "math.hpp"

namespace raisim {

using CollisionGroup = unsigned long;

inline void rsbCheck(int rc, const char* what) {
  if (rc >= 0) return;
#ifdef RAISIM_B200_ABORT_ON_ERROR
  std::fprintf(stderr, "[RSFATAL] %s: %s\n", what, rsb_last_error());
  std::abort();
#else
  throw std::runtime_error(std::string(what) + ": " + rsb_last_error());
#endif
}

namespace ControlMode {
enum Type : int { FORCE_AND_TORQUE = RSB_FORCE_AND_TORQUE, PD_PLUS_FEEDFORWARD_TORQUE = RSB_PD_PLUS_FEEDFORWARD_TORQUE };
}

// contact::Contact read-back (ArticulatedSystem::getContacts())
class Contact {
 public:
  explicit Contact(const rsb_contact& c) : c_(c) {}
  size_t getlocalBodyIndex() const { return size_t(c_.local_body); }
  size_t getPairObjectIndex() const { return 0; }            // the terrain is object 0 of the world
  int getPairContactIndexInPairObject() const { return c_.pair_index; }
  Vec<3> getPosition() const { return {c_.position[0], c_.position[1], c_.position[2]}; }
  Vec<3> getNormal() const { return {c_.normal[0], c_.normal[1], c_.normal[2]}; }
  Vec<3> getImpulse() const { return {c_.impulse[0], c_.impulse[1], c_.impulse[2]}; }   // world frame, on the robot
  double getDepth() const { return c_.depth; }
  // Rows t1, t2, n of the contact frame (DESIGN.md section 2: t1 = normalise(e_x - (e_x . n) n), e_y when |n_x| >= 0.9; t2 = n x t1), so
  // that frame^T * (impulse in the contact frame) = world-frame impulse, the product user code forms with upstream's frame.
  Mat<3, 3> getContactFrame() const {
    const double n[3] = {c_.normal[0], c_.normal[1], c_.normal[2]};
    const int a = std::fabs(n[0]) < 0.9 ? 0 : 1;
    double t1[3] = {-n[a] * n[0], -n[a] * n[1], -n[a] * n[2]};
    t1[a] += 1.0;
    const double inv = 1.0 / std::sqrt(t1[0] * t1[0] + t1[1] * t1[1] + t1[2] * t1[2]);
    for (double& x : t1) x *= inv;
    const double t2[3] = {n[1] * t1[2] - n[2] * t1[1], n[2] * t1[0] - n[0] * t1[2], n[0] * t1[1] - n[1] * t1[0]};
    Mat<3, 3> F;
    for (int j = 0; j < 3; j++) { F(0, j) = t1[j]; F(1, j) = t2[j]; F(2, j) = n[j]; }
    return F;
  }
  Vec<3> getImpulseInContactFrame() const {       // (tangential 1, tangential 2, normal): what the solver iterates on
    const Mat<3, 3> F = getContactFrame();
    Vec<3> l;
    for (int i = 0; i < 3; i++) l[i] = F(i, 0) * c_.impulse[0] + F(i, 1) * c_.impulse[1] + F(i, 2) * c_.impulse[2];
    return l;
  }
  bool isObjectA() const { return true; }
  bool skip() const { return false; }
 private:
  rsb_contact c_;
};

// Lock-step execution of N unmodified per-environment programs on one batch (VectorizedEnvironment<ENVIRONMENT>).
// Every environment holds World / ArticulatedSystem VIEWS of the same BatchedWorld.  Their setters and getters work on host
// mirrors of the batch rows, and World::integrate() only counts: the first access that needs the result (getState, getContacts,
// setPdTarget after an integrate ...) suspends that environment until every environment has reached the same point; then the
// dirty rows go up in one copy each, ONE launch integrates the counted sub-steps of every environment (the usual RaisimGym loop
// `for (i < control_dt / simulation_dt) world_->integrate();` becomes a single fused launch), and the mirrors are refilled lazily,
// one copy per array and control step.
struct LockStep {
  rsb_batch* batch = nullptr;
  int n = 0, nq = 0, nv = 0;
  std::vector<float> gc, gv, pt, vt, tau, tauApplied;
  std::vector<rsb_contact> contacts;
  std::vector<int32_t> ncontacts;
  std::vector<int> pending;                 // World::integrate() calls not executed yet, per environment
  bool stateValid = false, stateDirty = false, ptDirty = false, vtDirty = false, tauDirty = false, tauAppliedValid = false, contactsValid = false;
  long launches = 0;
  std::function<void(int)> suspend;         // installed by the scheduler: park the calling environment until the batch was flushed

  void init(rsb_batch* b, int n_, int nq_, int nv_) {
    batch = b; n = n_; nq = nq_; nv = nv_;
    gc.assign(size_t(n) * nq, 0.f); gv.assign(size_t(n) * nv, 0.f); pt.assign(size_t(n) * nq, 0.f); vt.assign(size_t(n) * nv, 0.f);
    tau.assign(size_t(n) * nv, 0.f); tauApplied.assign(size_t(n) * nv, 0.f); contacts.resize(size_t(n) * RSB_KMAX); ncontacts.assign(n, 0);
    pending.assign(n, 0);
  }
  // an environment is about to read or write the world: whatever it integrated before must have happened
  void sync(int env) {
    if (pending[env] == 0) return;
    if (!suspend) throw std::runtime_error("World: state access with integrate() calls pending outside VectorizedEnvironment::step()");
    suspend(env);
  }
  void needState() {
    if (stateValid) return;
    rsbCheck(rsb_batch_get_state(batch, gc.data(), gv.data(), 0, n, RSB_HOST), "getState");
    stateValid = true;
  }
  void needTauApplied() {
    if (tauAppliedValid) return;
    rsbCheck(rsb_batch_get_generalized_force(batch, tauApplied.data(), 0, n, RSB_HOST), "getGeneralizedForce");
    tauAppliedValid = true;
  }
  void needContacts() {
    if (contactsValid) return;
    rsbCheck(rsb_batch_get_contacts(batch, contacts.data(), ncontacts.data(), 0, n, RSB_HOST), "getContacts");
    contactsValid = true;
  }
  // every environment is parked (or finished) with the same number of integrate() calls pending: upload, one launch, invalidate
  void flush() {
    int k = 0;
    for (int e = 0; e < n; e++) k = pending[e] > k ? pending[e] : k;
    if (k == 0) return;
    for (int e = 0; e < n; e++)
      if (pending[e] != k) throw std::runtime_error("VectorizedEnvironment: environments disagree on the number of World::integrate() calls between two state accesses");
    if (stateDirty) rsbCheck(rsb_batch_set_state(batch, gc.data(), gv.data(), 0, n, RSB_HOST), "setState");
    if (ptDirty || vtDirty) rsbCheck(rsb_batch_set_pd_target(batch, ptDirty ? pt.data() : nullptr, vtDirty ? vt.data() : nullptr, 0, n, RSB_HOST), "setPdTarget");
    if (tauDirty) rsbCheck(rsb_batch_set_generalized_force(batch, tau.data(), 0, n, RSB_HOST), "setGeneralizedForce");
    stateDirty = ptDirty = vtDirty = tauDirty = false;
    rsbCheck(rsb_batch_integrate(batch, k), "integrate");
    launches++;
    for (int& p : pending) p = 0;
    stateValid = tauAppliedValid = contactsValid = false;
  }
  // rows written outside a step (reset(), init()): push them before anything else reads the device
  void pushWrites() {
    if (stateDirty) rsbCheck(rsb_batch_set_state(batch, gc.data(), gv.data(), 0, n, RSB_HOST), "setState");
    if (ptDirty || vtDirty) rsbCheck(rsb_batch_set_pd_target(batch, ptDirty ? pt.data() : nullptr, vtDirty ? vt.data() : nullptr, 0, n, RSB_HOST), "setPdTarget");
    if (tauDirty) rsbCheck(rsb_batch_set_generalized_force(batch, tau.data(), 0, n, RSB_HOST), "setGeneralizedForce");
    stateDirty = ptDirty = vtDirty = tauDirty = false;
  }
};

// One GPU batch of N identical worlds (new; the reference has no equivalent -- its batching is the
// OpenMP loop of VectorizedEnvironment).
class BatchedWorld {
 public:
  BatchedWorld(const std::string& urdfPathOrXml, int numEnvs, int device = 0) {
    rsbCheck(rsb_model_create_from_urdf(urdfPathOrXml.c_str(), &model_), "addArticulatedSystem");
    rsbCheck(rsb_batch_create(model_, numEnvs, device, &batch_), "BatchedWorld");
    rsbCheck(rsb_model_dims(model_, &nq_, &nv_, &nb_, nullptr, nullptr), "dims");
    n_ = numEnvs;
  }
  ~BatchedWorld() { if (batch_) rsb_batch_destroy(batch_); if (model_) rsb_model_destroy(model_); }
  BatchedWorld(const BatchedWorld&) = delete;
  BatchedWorld& operator=(const BatchedWorld&) = delete;
  rsb_batch* batch() const { return batch_; }
  rsb_model* model() const { return model_; }
  int numEnvs() const { return n_; }
  int nq() const { return nq_; }
  int nv() const { return nv_; }
  int nb() const { return nb_; }
  rsb_params params() const { rsb_params p; rsbCheck(rsb_batch_get_params(batch_, &p), "getParams"); return p; }
  void setParams(const rsb_params& p) { rsbCheck(rsb_batch_set_params(batch_, &p), "setParams"); }
  void integrate(int substeps = 1) { rsbCheck(rsb_batch_integrate(batch_, substeps), "integrate"); worldTime_ += substeps * params().dt; }
  void integrate1() { rsbCheck(rsb_batch_integrate1(batch_), "integrate1"); }
  void integrate2() { rsbCheck(rsb_batch_integrate2(batch_), "integrate2"); worldTime_ += params().dt; }
  double worldTime() const { return worldTime_; }
  void advanceTime(double t) { worldTime_ += t; }
  // lock-step mode (VectorizedEnvironment<ENVIRONMENT>): per-environment views work on host mirrors, integrate() is deferred
  LockStep* lockStep() { return ls_.get(); }
  void enableLockStep() { if (!ls_) { ls_.reset(new LockStep); ls_->init(batch_, n_, nq_, nv_); } }
  const std::string& urdf() const { return urdf_; }
  void rememberUrdf(const std::string& u) { urdf_ = u; }
 private:
  std::unique_ptr<LockStep> ls_;
  std::string urdf_;
  rsb_model* model_ = nullptr;
  rsb_batch* batch_ = nullptr;
  int n_ = 0, nq_ = 0, nv_ = 0, nb_ = 0;
  double worldTime_ = 0;
};

// raisim::Ground / raisim::HeightMap ([RECALL] object/terrain/Ground.hpp, HeightMap.hpp): host-side descriptions of the terrain the
// batch collides with -- what user code queries when it places a robot (getHeight) or builds height scans
class Ground {
 public:
  double getHeight(double /*x*/ = 0, double /*y*/ = 0) const { return z_; }
  void setHeight(double z) { z_ = z; }
 private:
  double z_ = 0;
};
class HeightMap {
 public:
  void set(size_t xs, size_t ys, double xSize, double ySize, double cx, double cy, std::vector<double> h) {
    xs_ = xs; ys_ = ys; xSize_ = xSize; ySize_ = ySize; cx_ = cx; cy_ = cy; h_ = std::move(h);
  }
  size_t getXSamples() const { return xs_; }
  size_t getYSamples() const { return ys_; }
  double getXSize() const { return xSize_; }
  double getYSize() const { return ySize_; }
  double getCenterX() const { return cx_; }
  double getCenterY() const { return cy_; }
  const std::vector<double>& getHeightVector() const { return h_; }
  // height of the collision surface at (x, y): the triangle of the cell beneath the point, two triangles per cell split along the
  // P00-P11 diagonal exactly as the narrow phase does (DESIGN.md section 2); outside the map: the nearest border point
  double getHeight(double x, double y) const {
    if (xs_ < 2 || ys_ < 2) return 0.0;
    const double dx = xSize_ / double(xs_ - 1), dy = ySize_ / double(ys_ - 1);
    double gx = (x - (cx_ - 0.5 * xSize_)) / dx, gy = (y - (cy_ - 0.5 * ySize_)) / dy;
    gx = std::fmin(std::fmax(gx, 0.0), double(xs_ - 1)); gy = std::fmin(std::fmax(gy, 0.0), double(ys_ - 1));
    size_t ix = size_t(gx), iy = size_t(gy);
    if (ix > xs_ - 2) ix = xs_ - 2;
    if (iy > ys_ - 2) iy = ys_ - 2;
    const double fx = gx - double(ix), fy = gy - double(iy);
    const double h00 = h_[iy * xs_ + ix], h10 = h_[iy * xs_ + ix + 1], h01 = h_[(iy + 1) * xs_ + ix], h11 = h_[(iy + 1) * xs_ + ix + 1];
    return fx >= fy ? h00 + (h10 - h00) * fx + (h11 - h10) * fy : h00 + (h11 - h01) * fx + (h01 - h00) * fy;
  }
 private:
  size_t xs_ = 0, ys_ = 0;
  double xSize_ = 0, ySize_ = 0, cx_ = 0, cy_ = 0;
  std::vector<double> h_;
};

// World::rayTest() result ([RECALL] upstream RayCollisionList / RayCollisionItem).  Rays see the terrain only (Ground / HeightMap), so a
// list holds at most one item: the closest hit.  getNormal(), getDistance() and getPairIndex() are extensions of this facade.
class RayCollisionItem {
 public:
  explicit RayCollisionItem(const rsb_ray_hit& h) : h_(h) {}
  Vec<3> getPosition() const { return {h_.position[0], h_.position[1], h_.position[2]}; }
  Vec<3> getNormal() const { return {h_.normal[0], h_.normal[1], h_.normal[2]}; }       // unit normal of the triangle hit, +z side
  double getDistance() const { return h_.distance; }                                       // along the unit direction
  int getPairIndex() const { return h_.pair_index; }                                       // 0 = Ground, 2*cell+tri on a HeightMap
  size_t getObjectIndex() const { return 0; }                                              // the terrain is object 0 of the world
 private:
  rsb_ray_hit h_;
};
class RayCollisionList {
 public:
  size_t size() const { return items_.size(); }
  const RayCollisionItem& operator[](size_t i) const { return items_[i]; }
  std::vector<RayCollisionItem>::const_iterator begin() const { return items_.begin(); }
  std::vector<RayCollisionItem>::const_iterator end() const { return items_.end(); }
  void clear() { items_.clear(); }
  void push(const rsb_ray_hit& h) { items_.emplace_back(h); }
 private:
  std::vector<RayCollisionItem> items_;
};

// ArticulatedSystem::getSparseJacobian(): the non-zero columns of a 3 x dof Jacobian (the ancestors' dofs only)
class SparseJacobian {
 public:
  size_t size = 0;             // number of non-zero columns
  std::vector<size_t> idx;     // their generalized-velocity indices, ascending
  MatDyn v;                    // 3 x size
  void resize(size_t cols) { size = cols; idx.assign(cols, 0); v.resize(3, cols); }
};

// ArticulatedSystem::setIntegrationScheme ([RECALL] ArticulatedSystem.hpp)
enum class IntegrationScheme : int { TRAPEZOID = 0, SEMI_IMPLICIT, EULER, RUNGE_KUTTA_4 };

// raisim::TerrainProperties ([RECALL] include/raisim/object/terrain/HeightMap.hpp)
struct TerrainProperties {
  double frequency = 0.1, xSize = 10.0, ySize = 10.0, zScale = 2.0, fractalLacunarity = 2.0, fractalGain = 0.5, stepSize = 0.0, heightOffset = 0.0;
  size_t xSamples = 100, ySamples = 100, fractalOctaves = 5;
  std::uint32_t seed = 1;
};

// raisim::ArticulatedSystem -- a view of one environment's robot
class ArticulatedSystem {
 public:
  ArticulatedSystem(BatchedWorld* w, int env) : w_(w), env_(env) {}
  // upstream addArticulatedSystem(urdf, resDir, jointOrder): the order of the joints in gc / gv as the caller wants it.  The batch keeps
  // its depth-first order; this view permutes on the way in and out (base coordinates first, as always).
  void setJointOrder(const std::vector<std::string>& jointOrder) {
    qmap_.clear(); vmap_.clear();
    if (jointOrder.empty()) return;
    rsb_model_tables t; rsbCheck(rsb_model_get_tables(w_->model(), &t), "getTables");
    const int nj = t.nb - 1, q0 = t.floating ? 7 : 0, v0 = t.floating ? 6 : 0;
    if (int(jointOrder.size()) != nj) throw std::runtime_error("addArticulatedSystem: jointOrder must name every movable joint exactly once");
    qmap_.resize(size_t(t.nq)); vmap_.resize(size_t(t.nv));
    for (int i = 0; i < q0; i++) qmap_[i] = i;
    for (int i = 0; i < v0; i++) vmap_[i] = i;
    std::vector<bool> seen(size_t(t.nb), false);
    for (int k = 0; k < nj; k++) {
      int body = -1;
      for (int b = 1; b < t.nb; b++) if (jointOrder[k] == rsb_model_joint_name(w_->model(), b)) body = b;
      if (body < 0 || seen[body]) throw std::runtime_error("addArticulatedSystem: jointOrder names an unknown joint or one joint twice: '" + jointOrder[k] + "'");
      seen[body] = true;
      qmap_[q0 + k] = t.qidx[body]; vmap_[v0 + k] = t.vidx[body];
    }
  }
  size_t getGeneralizedCoordinateDim() const { return size_t(w_->nq()); }
  size_t getDOF() const { return size_t(w_->nv()); }
  void setName(const std::string& n) { name_ = n; }
  const std::string& getName() const { return name_; }

  void getState(VecDyn& gc, VecDyn& gv) const {
    if (LockStep* ls = w_->lockStep()) {
      ls->sync(env_); ls->needState();
      gc.resize(size_t(ls->nq)); gv.resize(size_t(ls->nv));
      for (int i = 0; i < ls->nq; i++) gc[i] = ls->gc[size_t(env_) * ls->nq + qi(i)];
      for (int i = 0; i < ls->nv; i++) gv[i] = ls->gv[size_t(env_) * ls->nv + vi(i)];
      return;
    }
    std::vector<float> q(w_->nq()), v(w_->nv());
    rsbCheck(rsb_batch_get_state(w_->batch(), q.data(), v.data(), env_, 1, RSB_HOST), "getState");
    gc.resize(q.size()); gv.resize(v.size());
    for (size_t i = 0; i < q.size(); i++) gc[i] = q[qi(i)];
    for (size_t i = 0; i < v.size(); i++) gv[i] = v[vi(i)];
  }
  VecDyn getGeneralizedCoordinate() const { VecDyn q, v; getState(q, v); return q; }
  VecDyn getGeneralizedVelocity() const { VecDyn q, v; getState(q, v); return v; }
  template <class VQ, class VV> void setState(const VQ& gc, const VV& gv) {
    if (LockStep* ls = w_->lockStep()) {
      ls->sync(env_); ls->needState();           // the other environments' rows of the mirror must be current before the whole array goes up
      for (int i = 0; i < ls->nq; i++) ls->gc[size_t(env_) * ls->nq + qi(i)] = float(gc[i]);
      for (int i = 0; i < ls->nv; i++) ls->gv[size_t(env_) * ls->nv + vi(i)] = float(gv[i]);
      ls->stateDirty = true;
      return;
    }
    std::vector<float> q(w_->nq()), v(w_->nv());
    for (size_t i = 0; i < q.size(); i++) q[qi(i)] = float(gc[i]);
    for (size_t i = 0; i < v.size(); i++) v[vi(i)] = float(gv[i]);
    rsbCheck(rsb_batch_set_state(w_->batch(), q.data(), v.data(), env_, 1, RSB_HOST), "setState");
  }
  template <class VQ> void setGeneralizedCoordinate(const VQ& gc) {
    if (LockStep* ls = w_->lockStep()) {
      ls->sync(env_); ls->needState();
      for (int i = 0; i < ls->nq; i++) ls->gc[size_t(env_) * ls->nq + qi(i)] = float(gc[i]);
      ls->stateDirty = true;
      return;
    }
    std::vector<float> q(w_->nq());
    for (size_t i = 0; i < q.size(); i++) q[qi(i)] = float(gc[i]);
    rsbCheck(rsb_batch_set_state(w_->batch(), q.data(), nullptr, env_, 1, RSB_HOST), "setGeneralizedCoordinate");
  }
  template <class VV> void setGeneralizedVelocity(const VV& gv) {
    if (LockStep* ls = w_->lockStep()) {
      ls->sync(env_); ls->needState();
      for (int i = 0; i < ls->nv; i++) ls->gv[size_t(env_) * ls->nv + vi(i)] = float(gv[i]);
      ls->stateDirty = true;
      return;
    }
    std::vector<float> v(w_->nv());
    for (size_t i = 0; i < v.size(); i++) v[vi(i)] = float(gv[i]);
    rsbCheck(rsb_batch_set_state(w_->batch(), nullptr, v.data(), env_, 1, RSB_HOST), "setGeneralizedVelocity");
  }
  template <class VV> void setGeneralizedForce(const VV& tau) {
    if (LockStep* ls = w_->lockStep()) {
      ls->sync(env_);
      for (int i = 0; i < ls->nv; i++) ls->tau[size_t(env_) * ls->nv + vi(i)] = float(tau[i]);
      ls->tauDirty = true;
      return;
    }
    std::vector<float> t(w_->nv());
    for (size_t i = 0; i < t.size(); i++) t[vi(i)] = float(tau[i]);
    rsbCheck(rsb_batch_set_generalized_force(w_->batch(), t.data(), env_, 1, RSB_HOST), "setGeneralizedForce");
  }
  // gains are shared by every environment of the batch (they are per-robot-model constants in RaisimGym)
  template <class VV> void setPdGains(const VV& p, const VV& d) {
    std::vector<float> kp(w_->nv()), kd(w_->nv());
    for (size_t i = 0; i < kp.size(); i++) { kp[vi(i)] = float(p[i]); kd[vi(i)] = float(d[i]); }
    rsbCheck(rsb_batch_set_pd_gains(w_->batch(), kp.data(), kd.data()), "setPdGains");
  }
  template <class VQ, class VV> void setPdTarget(const VQ& posTarget, const VV& velTarget) {
    if (LockStep* ls = w_->lockStep()) {
      ls->sync(env_);
      for (int i = 0; i < ls->nq; i++) ls->pt[size_t(env_) * ls->nq + qi(i)] = float(posTarget[i]);
      for (int i = 0; i < ls->nv; i++) ls->vt[size_t(env_) * ls->nv + vi(i)] = float(velTarget[i]);
      ls->ptDirty = ls->vtDirty = true;
      return;
    }
    std::vector<float> q(w_->nq()), v(w_->nv());
    for (size_t i = 0; i < q.size(); i++) q[qi(i)] = float(posTarget[i]);
    for (size_t i = 0; i < v.size(); i++) v[vi(i)] = float(velTarget[i]);
    rsbCheck(rsb_batch_set_pd_target(w_->batch(), q.data(), v.data(), env_, 1, RSB_HOST), "setPdTarget");
  }
  void setControlMode(ControlMode::Type m) { rsbCheck(rsb_batch_set_control_mode(w_->batch(), int(m)), "setControlMode"); }

  // lazy getters: always describe the current state (the C-ABI refreshes M, h and the poses when the state changed)
  MatDyn getMassMatrix() const {
    const int nv = w_->nv();
    std::vector<float> m(size_t(nv) * nv);
    rsbCheck(rsb_batch_get_mass_matrix(w_->batch(), env_, 1, m.data(), RSB_HOST), "getMassMatrix");
    MatDyn M; M.resize(nv, nv);
    for (int i = 0; i < nv; i++) for (int j = 0; j < nv; j++) M(i, j) = m[vi(size_t(i)) * size_t(nv) + vi(size_t(j))];   // the caller's dof order (jointOrder)
    return M;
  }
  // M^-1 from the lazy M getter (dense Cholesky on the host: a convenience getter, not the hot path -- the kernel
  // never forms M^-1, it keeps the branch-sparse factor on chip)
  MatDyn getInverseMassMatrix() const {
    MatDyn M = getMassMatrix();
    const int n = int(M.rows());
    std::vector<double> L(size_t(n) * n, 0.0);
    for (int j = 0; j < n; j++) {
      double s = M(j, j);
      for (int k = 0; k < j; k++) s -= L[j * n + k] * L[j * n + k];
      const double d = std::sqrt(s);
      L[j * n + j] = d;
      for (int i = j + 1; i < n; i++) {
        double t = M(i, j);
        for (int k = 0; k < j; k++) t -= L[i * n + k] * L[j * n + k];
        L[i * n + j] = t / d;
      }
    }
    MatDyn Minv; Minv.resize(n, n);
    std::vector<double> x(n);
    for (int c = 0; c < n; c++) {
      for (int i = 0; i < n; i++) { double s = (i == c) ? 1.0 : 0.0; for (int k = 0; k < i; k++) s -= L[i * n + k] * x[k]; x[i] = s / L[i * n + i]; }
      for (int i = n - 1; i >= 0; i--) { double s = x[i]; for (int k = i + 1; k < n; k++) s -= L[k * n + i] * x[k]; x[i] = s / L[i * n + i]; }
      for (int i = 0; i < n; i++) Minv(i, c) = x[i];
    }
    return Minv;
  }
  VecDyn getGeneralizedForce() const {
    if (LockStep* ls = w_->lockStep()) {
      ls->sync(env_); ls->needTauApplied();
      VecDyn r(size_t(ls->nv));
      for (int i = 0; i < ls->nv; i++) r[i] = ls->tauApplied[size_t(env_) * ls->nv + vi(i)];
      return r;
    }
    std::vector<float> t(w_->nv());
    rsbCheck(rsb_batch_get_generalized_force(w_->batch(), t.data(), env_, 1, RSB_HOST), "getGeneralizedForce");
    VecDyn r(t.size());
    for (size_t i = 0; i < t.size(); i++) r[i] = t[vi(i)];
    return r;
  }
  // upstream: setExternalForce(localIdx, force) acts at the body COM, setExternalForce(localIdx, pos_in_body, force) at a
  // point fixed in the body, setExternalTorque(localIdx, torque); world frame, valid for the next integrate() only.
  // One wrench (force + torque on the same body) per environment.
  void setExternalForce(size_t localIdx, const Vec<3>& force) {
    rsb_model_tables t; rsbCheck(rsb_model_get_tables(w_->model(), &t), "getTables");
    Vec<3> c{t.com[localIdx * 3], t.com[localIdx * 3 + 1], t.com[localIdx * 3 + 2]};
    setExternalForce(localIdx, c, force);
  }
  void setExternalForce(size_t localIdx, const Vec<3>& posInBody, const Vec<3>& force) {
    if (extBody_ >= 0 && extBody_ != int(localIdx)) throw std::runtime_error("setExternalForce: one external wrench per environment (force and torque must act on the same body)");
    extBody_ = int(localIdx); extHasForce_ = true;
    for (int k = 0; k < 3; k++) { extF_[k] = float(force[k]); extP_[k] = float(posInBody[k]); }
    pushWrench();
  }
  void setExternalTorque(size_t localIdx, const Vec<3>& torque) {
    if (extBody_ >= 0 && extBody_ != int(localIdx)) throw std::runtime_error("setExternalTorque: one external wrench per environment (force and torque must act on the same body)");
    extBody_ = int(localIdx);
    for (int k = 0; k < 3; k++) extT_[k] = float(torque[k]);
    pushWrench();
  }
  void clearExternalWrench() { extBody_ = -1; extHasForce_ = false; for (int k = 0; k < 3; k++) extF_[k] = extT_[k] = extP_[k] = 0.f; }   // called by World::integrate()
  // upstream: robot->getCollisionBody("LF_FOOT/0").setMaterial("rubber"); world.setMaterialPairProp("rubber", "default", mu, ...)
  class CollisionBodyRef {
   public:
    CollisionBodyRef(ArticulatedSystem* a, size_t idx) : a_(a), idx_(idx) {}
    void setMaterial(const std::string& name) { a_->collisionMaterial_[idx_] = name; a_->materialsDirty_ = true; }
    const std::string& getMaterial() const { static const std::string d = "default"; auto it = a_->collisionMaterial_.find(idx_); return it == a_->collisionMaterial_.end() ? d : it->second; }
    size_t index() const { return idx_; }
   private:
    ArticulatedSystem* a_; size_t idx_;
  };
  CollisionBodyRef getCollisionBody(const std::string& name) {
    int i = rsb_model_collision_index(w_->model(), name.c_str());
    rsbCheck(i, "getCollisionBody");
    return CollisionBodyRef(this, size_t(i));
  }
  const std::map<size_t, std::string>& collisionMaterials() const { return collisionMaterial_; }
  bool materialsDirty() const { return materialsDirty_; }
  void materialsApplied() { materialsDirty_ = false; }
  // friction of one collision body against the terrain (upstream: getCollisionBody(name).setMaterial + setMaterialPairProp)
  void setCollisionBodyFriction(size_t collisionBodyIdx, double mu) {
    rsbCheck(rsb_batch_set_collision_friction(w_->batch(), int(collisionBodyIdx), float(mu)), "setCollisionBodyFriction");
  }
  VecDyn getNonlinearities() const {
    std::vector<float> h(w_->nv());
    rsbCheck(rsb_batch_get_nonlinearities(w_->batch(), env_, 1, h.data(), RSB_HOST), "getNonlinearities");
    VecDyn r(h.size());
    for (size_t i = 0; i < h.size(); i++) r[i] = h[vi(i)];
    return r;
  }
  size_t getBodyIdx(const std::string& name) const {
    int i = rsb_model_body_index(w_->model(), name.c_str());
    rsbCheck(i, "getBodyIdx");
    return size_t(i);
  }
  size_t getFrameIdxByName(const std::string& name) const {
    int i = rsb_model_frame_index(w_->model(), name.c_str());
    rsbCheck(i, "getFrameIdxByName");
    return size_t(i);
  }
  void getPosition(size_t bodyIdx, const Vec<3>& pointInBody, Vec<3>& out) const {
    std::vector<float> R(size_t(w_->nb()) * 9), p(size_t(w_->nb()) * 3);
    rsbCheck(rsb_batch_get_body_poses(w_->batch(), env_, 1, R.data(), p.data(), RSB_HOST), "getPosition");
    for (int r = 0; r < 3; r++) out[r] = p[bodyIdx * 3 + r] + R[bodyIdx * 9 + 3 * r] * pointInBody[0] + R[bodyIdx * 9 + 3 * r + 1] * pointInBody[1] + R[bodyIdx * 9 + 3 * r + 2] * pointInBody[2];
  }
  // ---- kinematic getters (host algebra on body poses the kernel computes for the current state) ----
  // upstream: getBodyPosition/Orientation, getFramePosition/Orientation/Velocity/AngularVelocity,
  // getVelocity/getAngularVelocity(bodyIdx), getDenseJacobian(bodyIdx, point_W, J), getDenseRotationalJacobian,
  // getDenseFrameJacobian / getDenseFrameRotationalJacobian ([RECALL] ArticulatedSystem.hpp; SURVEY.md 8b)
  void getBodyPosition(size_t bodyIdx, Vec<3>& out) const { Poses P = poses(); for (int r = 0; r < 3; r++) out[r] = P.p[bodyIdx * 3 + r]; }
  void getBodyOrientation(size_t bodyIdx, Mat<3, 3>& out) const {
    Poses P = poses();
    for (int r = 0; r < 3; r++) for (int c = 0; c < 3; c++) out(r, c) = P.R[bodyIdx * 9 + 3 * r + c];
  }
  void getBasePosition(Vec<3>& out) const { getBodyPosition(0, out); }
  void getBaseOrientation(Mat<3, 3>& out) const { getBodyOrientation(0, out); }
  void getFramePosition(size_t frameIdx, Vec<3>& out) const { Poses P = poses(); FrameW f = frameWorld(P, frameIdx); out = f.pos; }
  void getFrameOrientation(size_t frameIdx, Mat<3, 3>& out) const { Poses P = poses(); FrameW f = frameWorld(P, frameIdx); out = f.rot; }
  void getDenseJacobian(size_t bodyIdx, const Vec<3>& point_W, MatDyn& J) const { Poses P = poses(); jacobian(P, bodyIdx, point_W, &J, nullptr); }
  void getDenseRotationalJacobian(size_t bodyIdx, MatDyn& J) const { Poses P = poses(); jacobian(P, bodyIdx, Vec<3>{0, 0, 0}, nullptr, &J); }
  void getDenseFrameJacobian(size_t frameIdx, MatDyn& J) const { Poses P = poses(); FrameW f = frameWorld(P, frameIdx); jacobian(P, size_t(f.body), f.pos, &J, nullptr); }
  void getDenseFrameRotationalJacobian(size_t frameIdx, MatDyn& J) const { Poses P = poses(); FrameW f = frameWorld(P, frameIdx); jacobian(P, size_t(f.body), f.pos, nullptr, &J); }
  void getVelocity(size_t bodyIdx, const Vec<3>& point_W, Vec<3>& out) const {
    Poses P = poses(); MatDyn J; jacobian(P, bodyIdx, point_W, &J, nullptr); mulGv(J, out);
  }
  void getVelocity(size_t bodyIdx, Vec<3>& out) const { Vec<3> o; getBodyPosition(bodyIdx, o); getVelocity(bodyIdx, o, out); }
  void getAngularVelocity(size_t bodyIdx, Vec<3>& out) const { Poses P = poses(); MatDyn J; jacobian(P, bodyIdx, Vec<3>{0, 0, 0}, nullptr, &J); mulGv(J, out); }
  void getFrameVelocity(size_t frameIdx, Vec<3>& out) const { MatDyn J; getDenseFrameJacobian(frameIdx, J); mulGv(J, out); }
  void getFrameAngularVelocity(size_t frameIdx, Vec<3>& out) const { MatDyn J; getDenseFrameRotationalJacobian(frameIdx, J); mulGv(J, out); }

  // ---- model queries and whole-body quantities (host algebra on the model tables, the poses and M of the current state;
  //      upstream names, [RECALL] ArticulatedSystem.hpp) --------------------------------------------------------------
  std::vector<std::string> getBodyNames() const {
    std::vector<std::string> r;
    for (int b = 0; b < w_->nb(); b++) r.emplace_back(rsb_model_body_name(w_->model(), b));
    return r;
  }
  // movable joints in the order of the generalized coordinates the caller sees (jointOrder if one was given)
  std::vector<std::string> getMovableJointNames() const {
    const rsb_model_tables t = tables();
    const int q0 = t.floating ? 7 : 0;
    std::vector<std::string> r(size_t(t.nq - q0));
    for (int k = 0; k < t.nq - q0; k++)
      for (int b = 1; b < t.nb; b++) if (t.qidx[b] == int(qi(size_t(q0 + k)))) r[size_t(k)] = rsb_model_joint_name(w_->model(), b);
    return r;
  }
  // [lower, upper] per generalized velocity index (URDF <limit lower upper>; the base dofs and unlimited joints: -/+ 1e30 as parsed)
  std::vector<Vec<2>> getJointLimits() const {
    const rsb_model_tables t = tables();
    std::vector<Vec<2>> r(size_t(t.nv));
    for (int i = 0; i < t.nv; i++) { r[size_t(i)][0] = -1e30; r[size_t(i)][1] = 1e30; }
    for (int i = 0; i < t.nv; i++)
      for (int b = 1; b < t.nb; b++) if (t.vidx[b] == int(vi(size_t(i)))) { r[size_t(i)][0] = t.jlimit[2 * b]; r[size_t(i)][1] = t.jlimit[2 * b + 1]; }
    return r;
  }
  // actuator effort limits per generalized velocity index (URDF <limit effort>; none: 1e30); the step kernel saturates the commanded torque there
  VecDyn getActuationUpperLimits() const {
    const rsb_model_tables t = tables();
    VecDyn r(size_t(t.nv));
    for (int i = 0; i < t.nv; i++) {
      r[size_t(i)] = 1e30;
      for (int b = 1; b < t.nb; b++) if (t.vidx[b] == int(vi(size_t(i)))) r[size_t(i)] = t.jeffort[b];
    }
    return r;
  }
  VecDyn getActuationLowerLimits() const { VecDyn r = getActuationUpperLimits(); for (size_t i = 0; i < r.size(); i++) r[i] = -r[i]; return r; }
  double getMass(size_t localIdx) const { return tables().mass[localIdx]; }
  double getTotalMass() const { const rsb_model_tables t = tables(); double m = 0; for (int b = 0; b < t.nb; b++) m += t.mass[b]; return m; }
  std::vector<Vec<3>> getBodyCOM_B() const {
    const rsb_model_tables t = tables();
    std::vector<Vec<3>> r(size_t(t.nb));
    for (int b = 0; b < t.nb; b++) for (int k = 0; k < 3; k++) r[size_t(b)][size_t(k)] = t.com[3 * b + k];
    return r;
  }
  std::vector<Vec<3>> getBodyCOM_W() const {
    const rsb_model_tables t = tables(); const Poses P = poses();
    std::vector<Vec<3>> r(size_t(t.nb));
    for (int b = 0; b < t.nb; b++) r[size_t(b)] = comWorld(t, P, b);
    return r;
  }
  Vec<3> getCOM() const {      // centre of mass of the whole robot, world frame
    const rsb_model_tables t = tables(); const Poses P = poses();
    Vec<3> c; double m = 0;
    for (int b = 0; b < t.nb; b++) { const Vec<3> cb = comWorld(t, P, b); for (int k = 0; k < 3; k++) c[size_t(k)] += t.mass[b] * cb[size_t(k)]; m += t.mass[b]; }
    for (int k = 0; k < 3; k++) c[size_t(k)] /= m;
    return c;
  }
  VecDyn getGeneralizedMomentum() const {      // M gv (M from the kernel's CRBA)
    const MatDyn M = getMassMatrix(); const VecDyn gv = getGeneralizedVelocity();
    VecDyn r(size_t(M.rows()));
    for (size_t i = 0; i < M.rows(); i++) { double s = 0; for (size_t j = 0; j < M.cols(); j++) s += M(i, j) * gv[j]; r[i] = s; }
    return r;
  }
  double getKineticEnergy() const {
    const MatDyn M = getMassMatrix(); const VecDyn gv = getGeneralizedVelocity();
    double e = 0;
    for (size_t i = 0; i < M.rows(); i++) for (size_t j = 0; j < M.cols(); j++) e += 0.5 * gv[i] * M(i, j) * gv[j];
    return e;
  }
  double getPotentialEnergy(const Vec<3>& gravity) const {
    const rsb_model_tables t = tables(); const Poses P = poses();
    double e = 0;
    for (int b = 0; b < t.nb; b++) { const Vec<3> c = comWorld(t, P, b); e -= t.mass[b] * (gravity[0] * c[0] + gravity[1] * c[1] + gravity[2] * c[2]); }
    return e;
  }
  double getEnergy(const Vec<3>& gravity) const { return getKineticEnergy() + getPotentialEnergy(gravity); }
  Vec<3> getLinearMomentum() const {           // sum of m_b v_com,b through the body Jacobians
    const rsb_model_tables t = tables(); const Poses P = poses(); const VecDyn gv = getGeneralizedVelocity();
    Vec<3> p;
    for (int b = 0; b < t.nb; b++) {
      MatDyn J; jacobian(P, size_t(b), comWorld(t, P, b), &J, nullptr);
      for (int r = 0; r < 3; r++) { double s = 0; for (size_t c = 0; c < J.cols(); c++) s += J(size_t(r), c) * gv[c]; p[size_t(r)] += t.mass[b] * s; }
    }
    return p;
  }
  void getSparseJacobian(size_t bodyIdx, const Vec<3>& point_W, SparseJacobian& J) const {
    const rsb_model_tables t = tables(); const Poses P = poses();
    MatDyn D; jacobian(P, bodyIdx, point_W, &D, nullptr);
    std::vector<size_t> cols;        // dofs of the chain root .. body, in the caller's order
    for (int i = int(bodyIdx); i >= 0; i = t.parent[i]) {
      const int nd = t.jtype[i] == 3 ? 6 : (t.jtype[i] == 1 || t.jtype[i] == 2 ? 1 : 0);
      for (int k = 0; k < nd; k++) cols.push_back(vinv(size_t(t.vidx[i] + k)));
    }
    std::sort(cols.begin(), cols.end());
    J.resize(cols.size());
    for (size_t k = 0; k < cols.size(); k++) { J.idx[k] = cols[k]; for (size_t r = 0; r < 3; r++) J.v(r, k) = D(r, cols[k]); }
  }
  // base pose setters (floating base): the other coordinates stay as they are
  void setBasePos(const Vec<3>& pos) {
    VecDyn gc = getGeneralizedCoordinate();
    if (gc.size() < 7 || !tables().floating) throw std::runtime_error("setBasePos: the robot has a fixed base");
    for (size_t k = 0; k < 3; k++) gc[k] = pos[k];
    setGeneralizedCoordinate(gc);
  }
  void setBaseOrientation(const Vec<4>& quat) {
    VecDyn gc = getGeneralizedCoordinate();
    if (gc.size() < 7 || !tables().floating) throw std::runtime_error("setBaseOrientation: the robot has a fixed base");
    const double n = std::sqrt(quat[0] * quat[0] + quat[1] * quat[1] + quat[2] * quat[2] + quat[3] * quat[3]);
    for (size_t k = 0; k < 4; k++) gc[3 + k] = quat[k] / n;
    setGeneralizedCoordinate(gc);
  }
  void setBaseOrientation(const Mat<3, 3>& rot) { Vec<4> q; rotMatToQuat(rot, q); setBaseOrientation(q); }
  // upstream's separate target / gain setters: the other half keeps its last value
  template <class VQ> void setPTarget(const VQ& posTarget) {
    lastP_.resize(size_t(w_->nq())); for (size_t i = 0; i < lastP_.size(); i++) lastP_[i] = posTarget[i];
    if (lastD_.size() != size_t(w_->nv())) lastD_.resize(size_t(w_->nv()));
    setPdTarget(lastP_, lastD_);
  }
  template <class VV> void setDTarget(const VV& velTarget) {
    lastD_.resize(size_t(w_->nv())); for (size_t i = 0; i < lastD_.size(); i++) lastD_[i] = velTarget[i];
    if (lastP_.size() != size_t(w_->nq())) lastP_ = getGeneralizedCoordinate();     // no position target given yet: hold the current pose
    setPdTarget(lastP_, lastD_);
  }
  template <class VV> void setPGains(const VV& p) {
    kpLast_.resize(size_t(w_->nv())); for (size_t i = 0; i < kpLast_.size(); i++) kpLast_[i] = p[i];
    if (kdLast_.size() != kpLast_.size()) kdLast_.resize(kpLast_.size());
    setPdGains(kpLast_, kdLast_);
  }
  template <class VV> void setDGains(const VV& d) {
    kdLast_.resize(size_t(w_->nv())); for (size_t i = 0; i < kdLast_.size(); i++) kdLast_[i] = d[i];
    if (kpLast_.size() != kdLast_.size()) kpLast_.resize(kdLast_.size());
    setPdGains(kpLast_, kdLast_);
  }
  // The batch integrates semi-implicitly (DESIGN.md section 2: v+ from the implicit PD / contact solve, then q+ = q (+) dt v+);
  // asking for another scheme fails loudly instead of silently integrating differently from what the caller expects.
  void setIntegrationScheme(IntegrationScheme scheme) {
    if (scheme != IntegrationScheme::SEMI_IMPLICIT) throw std::runtime_error("setIntegrationScheme: only IntegrationScheme::SEMI_IMPLICIT is implemented by the batched step");
  }

  std::vector<Contact>& getContacts() {
    if (LockStep* ls = w_->lockStep()) {
      ls->sync(env_); ls->needContacts();
      contacts_.clear();
      for (int i = 0; i < ls->ncontacts[env_]; i++) contacts_.emplace_back(ls->contacts[size_t(env_) * RSB_KMAX + i]);
      return contacts_;
    }
    rsb_contact c[RSB_KMAX]; int32_t n = 0;
    rsbCheck(rsb_batch_get_contacts(w_->batch(), c, &n, env_, 1, RSB_HOST), "getContacts");
    contacts_.clear();
    for (int i = 0; i < n; i++) contacts_.emplace_back(c[i]);
    return contacts_;
  }
  int env() const { return env_; }
 private:
  void pushWrench() {
    rsbCheck(rsb_batch_set_external_wrench(w_->batch(), extBody_, extF_, extT_, extP_, env_, 1, RSB_HOST), "setExternalForce");
  }
  std::map<size_t, std::string> collisionMaterial_;   // collision body -> material name (absent = "default")
  bool materialsDirty_ = false;
  int extBody_ = -1; bool extHasForce_ = false;
  float extF_[3] = {0, 0, 0}, extT_[3] = {0, 0, 0}, extP_[3] = {0, 0, 0};
  struct Poses { std::vector<float> R, p; };
  struct FrameW { int body; Vec<3> pos; Mat<3, 3> rot; };
  Poses poses() const {
    Poses P; P.R.resize(size_t(w_->nb()) * 9); P.p.resize(size_t(w_->nb()) * 3);
    if (LockStep* ls = w_->lockStep()) { ls->sync(env_); ls->pushWrites(); }
    // the C-ABI getter is lazy: it runs a kinematics-only pass when the state changed (upstream's updateKinematics()); the contact
    // records and impulses of the last integrate() stay valid across kinematic getters, as upstream's getContacts() does
    rsbCheck(rsb_batch_get_body_poses(w_->batch(), env_, 1, P.R.data(), P.p.data(), RSB_HOST), "getBodyPoses");
    return P;
  }
  FrameW frameWorld(const Poses& P, size_t frameIdx) const {
    FrameW f; double pos[3], rot[9];
    rsbCheck(rsb_model_frame(w_->model(), int(frameIdx), &f.body, pos, rot), "getFrame");
    const float* R = &P.R[size_t(f.body) * 9];
    for (int r = 0; r < 3; r++) {
      f.pos[r] = P.p[size_t(f.body) * 3 + r] + R[3 * r] * pos[0] + R[3 * r + 1] * pos[1] + R[3 * r + 2] * pos[2];
      for (int c = 0; c < 3; c++) f.rot(r, c) = R[3 * r] * rot[c] + R[3 * r + 1] * rot[3 + c] + R[3 * r + 2] * rot[6 + c];
    }
    return f;
  }
  // geometric Jacobians of a world point attached to `body`: v_point = Jp gv, omega_body = Jr gv
  void jacobian(const Poses& P, size_t body, const Vec<3>& pt, MatDyn* Jp, MatDyn* Jr) const {
    rsb_model_tables t; rsbCheck(rsb_model_get_tables(w_->model(), &t), "getTables");
    if (Jp) Jp->resize(3, size_t(t.nv));
    if (Jr) Jr->resize(3, size_t(t.nv));
    for (int i = int(body); i >= 0; i = t.parent[i]) {
      const float* R = &P.R[size_t(i) * 9]; const float* o = &P.p[size_t(i) * 3];
      const double r[3] = {pt[0] - o[0], pt[1] - o[1], pt[2] - o[2]};
      if (t.jtype[i] == 3) {          // floating base: [v_world | omega_world]
        if (Jp) {
          for (int k = 0; k < 3; k++) (*Jp)(k, k) = 1.0;
          (*Jp)(0, 4) = r[2]; (*Jp)(0, 5) = -r[1]; (*Jp)(1, 3) = -r[2]; (*Jp)(1, 5) = r[0]; (*Jp)(2, 3) = r[1]; (*Jp)(2, 4) = -r[0];   // -[r]x
        }
        if (Jr) for (int k = 0; k < 3; k++) (*Jr)(k, 3 + k) = 1.0;
      } else if (t.jtype[i] == 1 || t.jtype[i] == 2) {
        const double* ab = &t.axis[size_t(i) * 3];
        double a[3];
        for (int k = 0; k < 3; k++) a[k] = R[3 * k] * ab[0] + R[3 * k + 1] * ab[1] + R[3 * k + 2] * ab[2];
        const size_t c = vinv(size_t(t.vidx[i]));      // column in the caller's dof order (jointOrder)
        if (t.jtype[i] == 1) {
          if (Jp) { (*Jp)(0, c) = a[1] * r[2] - a[2] * r[1]; (*Jp)(1, c) = a[2] * r[0] - a[0] * r[2]; (*Jp)(2, c) = a[0] * r[1] - a[1] * r[0]; }
          if (Jr) for (int k = 0; k < 3; k++) (*Jr)(k, c) = a[k];
        } else if (Jp) for (int k = 0; k < 3; k++) (*Jp)(k, c) = a[k];
      }
    }
  }
  void mulGv(const MatDyn& J, Vec<3>& out) const {
    VecDyn gv = getGeneralizedVelocity();
    for (int r = 0; r < 3; r++) { double s = 0; for (size_t c = 0; c < J.cols(); c++) s += J(r, c) * gv[c]; out[r] = s; }
  }
  size_t qi(size_t i) const { return qmap_.empty() ? i : size_t(qmap_[i]); }     // caller's coordinate index -> the batch's
  size_t vi(size_t i) const { return vmap_.empty() ? i : size_t(vmap_[i]); }
  size_t vinv(size_t batchIdx) const {                                            // the batch's velocity index -> the caller's
    if (vmap_.empty()) return batchIdx;
    for (size_t i = 0; i < vmap_.size(); i++) if (size_t(vmap_[i]) == batchIdx) return i;
    return batchIdx;
  }
  rsb_model_tables tables() const { rsb_model_tables t; rsbCheck(rsb_model_get_tables(w_->model(), &t), "getTables"); return t; }
  Vec<3> comWorld(const rsb_model_tables& t, const Poses& P, int b) const {
    const float* R = &P.R[size_t(b) * 9]; const float* o = &P.p[size_t(b) * 3]; const double* c = &t.com[size_t(b) * 3];
    Vec<3> r;
    for (int k = 0; k < 3; k++) r[size_t(k)] = o[k] + R[3 * k] * c[0] + R[3 * k + 1] * c[1] + R[3 * k + 2] * c[2];
    return r;
  }
  VecDyn lastP_, lastD_, kpLast_, kdLast_;
  std::vector<int> qmap_, vmap_;
  BatchedWorld* w_;
  int env_;
  std::string name_;
  std::vector<Contact> contacts_;
};

// raisim::World -- standalone it owns a batch of one environment; as a view it forwards to a shared batch
// While a VectorizedEnvironment<ENVIRONMENT> constructs its environments, every `raisim::World` they create becomes a view of
// ONE shared batch instead of a batch of one: environment i's World is view i; the first addArticulatedSystem() creates the
// batch (num_envs environments of that URDF, lock-step mode), the others attach to it.
struct BatchContext {
  int numEnvs = 0, device = 0, envIndex = 0;
  std::unique_ptr<BatchedWorld> batch;
  static BatchContext*& current() { static thread_local BatchContext* c = nullptr; return c; }
};

class World {
 public:
  World() { if (BatchContext* c = BatchContext::current()) { ctx_ = c; env_ = c->envIndex; } }
  World(BatchedWorld* shared, int env) : w_(shared), env_(env) { robot_.reset(new ArticulatedSystem(w_, env_)); }
  static void setActivationKey(const std::string&) {}          // licence check of the reference: not a capability

  ArticulatedSystem* addArticulatedSystem(const std::string& urdfPathOrXml, const std::string& = "", const std::vector<std::string>& jointOrder = {},
                                          CollisionGroup = 1, CollisionGroup = CollisionGroup(-1)) {
    if (w_) throw std::runtime_error("addArticulatedSystem: this World is a view of a BatchedWorld (one robot per environment)");
    if (ctx_) {   // environment of a VectorizedEnvironment: attach to (or create) the shared batch
      if (!ctx_->batch) {
        ctx_->batch.reset(new BatchedWorld(urdfPathOrXml, ctx_->numEnvs, ctx_->device));
        ctx_->batch->rememberUrdf(urdfPathOrXml);
        ctx_->batch->enableLockStep();
      } else if (ctx_->batch->urdf() != urdfPathOrXml) throw std::runtime_error("VectorizedEnvironment: every environment must load the same robot description");
      w_ = ctx_->batch.get();
      rsb_params p = w_->params();
      p.dt = float(dt_); p.gravity[0] = float(g_[0]); p.gravity[1] = float(g_[1]); p.gravity[2] = float(g_[2]);
      w_->setParams(p);
      if (haveGround_) rsbCheck(rsb_batch_set_ground(w_->batch(), float(groundZ_)), "addGround");
      robot_.reset(new ArticulatedSystem(w_, env_));
      robot_->setJointOrder(jointOrder);
      return robot_.get();
    }
    owned_.reset(new BatchedWorld(urdfPathOrXml, 1));
    w_ = owned_.get(); env_ = 0;
    rsb_params p = w_->params();
    p.dt = float(dt_); p.gravity[0] = float(g_[0]); p.gravity[1] = float(g_[1]); p.gravity[2] = float(g_[2]);
    w_->setParams(p);
    if (haveGround_) rsbCheck(rsb_batch_set_ground(w_->batch(), float(groundZ_)), "addGround");
    robot_.reset(new ArticulatedSystem(w_, 0));
    robot_->setJointOrder(jointOrder);
    return robot_.get();
  }
  Ground* addGround(double zHeight = 0.0, const std::string& material = "default", CollisionGroup = CollisionGroup(-1)) {
    haveGround_ = true; groundZ_ = zHeight; terrainMaterial_ = material; ground_.setHeight(zHeight);
    if (robot_) applyMaterials(true);
    if (w_) rsbCheck(rsb_batch_set_ground(w_->batch(), float(zHeight)), "addGround");
    return &ground_;
  }
  HeightMap* addHeightMap(size_t xSamples, size_t ySamples, double xSize, double ySize, double centerX, double centerY,
                          const std::vector<double>& height, const std::string& = "default", CollisionGroup = 1, CollisionGroup = CollisionGroup(-1)) {
    need();
    std::vector<float> h(height.begin(), height.end());
    rsbCheck(rsb_batch_set_heightmap(w_->batch(), int(xSamples), int(ySamples), float(xSize), float(ySize), float(centerX), float(centerY), h.data()), "addHeightMap");
    hm_.set(xSamples, ySamples, xSize, ySize, centerX, centerY, std::vector<double>(h.begin(), h.end()));   // what the batch collides with (float32 heights)
    return &hm_;
  }
  HeightMap* addHeightMap(double centerX, double centerY, const TerrainProperties& tp, const std::string& = "default", CollisionGroup = 1,
                          CollisionGroup = CollisionGroup(-1)) {
    need();
    rsb_terrain_properties p{int(tp.xSamples), int(tp.ySamples), tp.xSize, tp.ySize, tp.frequency, tp.zScale, int(tp.fractalOctaves), tp.fractalLacunarity,
                             tp.fractalGain, tp.stepSize, tp.heightOffset, tp.seed};
    std::vector<float> h(tp.xSamples * tp.ySamples);
    rsbCheck(rsb_terrain_generate(&p, h.data()), "TerrainGenerator");
    rsbCheck(rsb_batch_set_heightmap(w_->batch(), int(tp.xSamples), int(tp.ySamples), float(tp.xSize), float(tp.ySize), float(centerX), float(centerY), h.data()), "addHeightMap");
    hm_.set(tp.xSamples, tp.ySamples, tp.xSize, tp.ySize, centerX, centerY, std::vector<double>(h.begin(), h.end()));
    return &hm_;
  }
  // height-map files (upstream overloads of the same name; [RECALL] formats, see include/rsb.h)
  HeightMap* addHeightMap(const std::string& raisimHeightMapFileName, double centerX, double centerY, const std::string& = "default",
                          CollisionGroup = 1, CollisionGroup = CollisionGroup(-1)) {
    need();
    int xs = 0, ys = 0; double sx = 0, sy = 0;
    rsbCheck(rsb_heightmap_read_text(raisimHeightMapFileName.c_str(), &xs, &ys, &sx, &sy, nullptr, 0), "addHeightMap");
    std::vector<float> h(size_t(xs) * ys);
    rsbCheck(rsb_heightmap_read_text(raisimHeightMapFileName.c_str(), &xs, &ys, &sx, &sy, h.data(), int(h.size())), "addHeightMap");
    rsbCheck(rsb_batch_set_heightmap(w_->batch(), xs, ys, float(sx), float(sy), float(centerX), float(centerY), h.data()), "addHeightMap");
    hm_.set(size_t(xs), size_t(ys), sx, sy, centerX, centerY, std::vector<double>(h.begin(), h.end()));
    return &hm_;
  }
  HeightMap* addHeightMap(const std::string& pngFileName, double centerX, double centerY, double xSize, double ySize, double heightScale,
                          double heightOffset, const std::string& = "default", CollisionGroup = 1, CollisionGroup = CollisionGroup(-1)) {
    need();
    int xs = 0, ys = 0;
    rsbCheck(rsb_heightmap_read_png(pngFileName.c_str(), heightScale, heightOffset, &xs, &ys, nullptr, 0), "addHeightMap");
    std::vector<float> h(size_t(xs) * ys);
    rsbCheck(rsb_heightmap_read_png(pngFileName.c_str(), heightScale, heightOffset, &xs, &ys, h.data(), int(h.size())), "addHeightMap");
    rsbCheck(rsb_batch_set_heightmap(w_->batch(), xs, ys, float(xSize), float(ySize), float(centerX), float(centerY), h.data()), "addHeightMap");
    hm_.set(size_t(xs), size_t(ys), xSize, ySize, centerX, centerY, std::vector<double>(h.begin(), h.end()));
    return &hm_;
  }
  void setTimeStep(double dt) { dt_ = dt; if (w_) { rsb_params p = w_->params(); p.dt = float(dt); w_->setParams(p); } }
  double getTimeStep() const { return dt_; }
  void setGravity(const Vec<3>& g) { g_ = g; if (w_) { rsb_params p = w_->params(); for (int k = 0; k < 3; k++) p.gravity[k] = float(g[k]); w_->setParams(p); } }
  void setERP(double erp, double = 0) { need(); rsb_params p = w_->params(); p.erp = float(erp); w_->setParams(p); }
  void setContactSolverParam(double alpha_init, double alpha_min, double alpha_decay, int maxIter, double threshold) {
    need(); rsb_params p = w_->params();
    p.alpha_init = float(alpha_init); p.alpha_min = float(alpha_min); p.alpha_decay = float(alpha_decay); p.max_iter = maxIter; p.threshold = float(threshold);
    w_->setParams(p);
  }
  void setDefaultMaterial(double friction, double restitution, double resThreshold) {
    need(); rsb_params p = w_->params(); p.mu = float(friction); p.restitution = float(restitution); p.rest_threshold = float(resThreshold); w_->setParams(p);
  }
  // named material pairs: friction of (collision-body material, terrain material); restitution is global (setDefaultMaterial)
  void setMaterialPairProp(const std::string& m1, const std::string& m2, double friction, double /*restitution*/ = 0, double /*resThreshold*/ = 0) {
    pairFriction_[m1 < m2 ? std::make_pair(m1, m2) : std::make_pair(m2, m1)] = friction;
    if (robot_) applyMaterials(true);
  }
  struct ContactSolverView {            // World::getContactSolver().getLoopCounter()
    const World* w;
    int getLoopCounter() const { int32_t it = 0; rsbCheck(rsb_batch_get_solver_iterations(w->w_->batch(), &it, w->env_, 1, RSB_HOST), "getLoopCounter"); return it; }
  };
  ContactSolverView getContactSolver() const { need(); return ContactSolverView{this}; }
  // upstream World::rayTest: the first crossing of start + t * direction / |direction|, t in [0, length], with this environment's terrain.
  // The robot is not hit (objectId / localId / mask select among objects upstream; the terrain is the only one here).  Only the closest
  // hit exists on this path: closestOnly = false is refused.  The terrain is static, so inside a VectorizedEnvironment this costs no
  // lock-step flush; one launch on the batch's stream and one 32-byte read-back.
  const RayCollisionList& rayTest(const Vec<3>& start, const Vec<3>& direction, double length, bool closestOnly = true, size_t /*objectId*/ = size_t(-10),
                                  size_t /*localId*/ = size_t(-10), CollisionGroup /*collisionMask*/ = CollisionGroup(-1)) {
    if (!closestOnly) throw std::runtime_error("rayTest: only closestOnly = true is implemented (rays see the terrain only: one hit at most)");
    need();
    const float o[3] = {float(start[0]), float(start[1]), float(start[2])}, d[3] = {float(direction[0]), float(direction[1]), float(direction[2])};
    rsb_ray_hit h;
    rsbCheck(rsb_batch_ray_test(w_->batch(), nullptr, 0, o, d, 1, float(length), &h, env_, 1, RSB_HOST), "rayTest");
    rays_.clear();
    if (h.pair_index >= 0) rays_.push(h);
    return rays_;
  }
  ArticulatedSystem* getObject(const std::string& name) { return (robot_ && robot_->getName() == name) ? robot_.get() : nullptr; }
  // object-object and self collisions are not part of this path (robot vs terrain only): nothing to ignore
  void ignoreCollisionBetween(size_t, size_t, size_t, size_t) {}
  // one World::integrate() of THIS environment's batch.  Views of a shared batch must not call this
  // per environment -- the vectorized wrapper steps the whole batch once (see VectorizedEnvironment.hpp).
  void integrate() {
    need();
    if (LockStep* ls = w_->lockStep()) {   // deferred: counted now, executed for every environment at once when the result is first needed
      ls->pending[env_]++;
      if (env_ == 0) w_->advanceTime(w_->params().dt);
      return;
    }
    applyMaterials(false); w_->integrate(1); if (robot_) robot_->clearExternalWrench();
  }
  void integrate1() { need(); applyMaterials(false); w_->integrate1(); }
  void integrate2() { need(); w_->integrate2(); if (robot_) robot_->clearExternalWrench(); }
  double getWorldTime() const { return w_ ? w_->worldTime() : 0.0; }
  ArticulatedSystem* getRobot() { return robot_.get(); }
  BatchedWorld* batched() { return w_; }
 private:
  void need() const { if (!w_) throw std::runtime_error("World: call addArticulatedSystem() first (the batch is created with the robot)"); }
  void applyMaterials(bool force) {
    if (!robot_ || (!force && !robot_->materialsDirty())) return;
    for (const auto& kv : robot_->collisionMaterials()) {
      const std::string& a = kv.second; const std::string& b = terrainMaterial_;
      auto it = pairFriction_.find(a < b ? std::make_pair(a, b) : std::make_pair(b, a));
      robot_->setCollisionBodyFriction(kv.first, it == pairFriction_.end() ? -1.0 : it->second);   // < 0: default material
    }
    robot_->materialsApplied();
  }
  std::map<std::pair<std::string, std::string>, double> pairFriction_;
  std::string terrainMaterial_ = "default";
  std::unique_ptr<BatchedWorld> owned_;
  BatchedWorld* w_ = nullptr;
  BatchContext* ctx_ = nullptr;
  int env_ = 0;
  std::unique_ptr<ArticulatedSystem> robot_;
  Ground ground_; HeightMap hm_;
  RayCollisionList rays_;
  bool haveGround_ = false;
  double groundZ_ = 0, dt_ = 0.005;
  Vec<3> g_{0, 0, -9.81};
};

}  // namespace raisim
