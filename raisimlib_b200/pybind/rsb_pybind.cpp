// pybind11 module over the C-ABI (SURVEY 8f row N4): the batched device state as DLPack tensors, zero-copy.
// Replaces the numpy path of upstream raisimGymTorch/env/raisim_gym.cpp ([RECALL]; not in the reference snapshot): a PyTorch trainer
// on the same GPU takes `torch.from_dlpack(batch.gc())` and reads / writes the rows the step kernel works on -- no host round trip.
// Only include/rsb.h is used: the module links librsb.so, it contains no CUDA code of its own.
#include <pybind11/pybind11.h>
#include <pybind11/stl.h>

#include <cstdint>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/rsb.h"

namespace py = pybind11;

// ---- DLPack (dlpack.h v0.8 ABI, restated: the header is not vendored here) -------------------------------------------------------
extern "C" {
typedef enum { kDLCPU = 1, kDLCUDA = 2 } DLDeviceType;
typedef struct { int32_t device_type; int32_t device_id; } DLDevice;
typedef struct { uint8_t code; uint8_t bits; uint16_t lanes; } DLDataType;      // code 0 int, 1 uint, 2 float
typedef struct { void* data; DLDevice device; int32_t ndim; DLDataType dtype; int64_t* shape; int64_t* strides; uint64_t byte_offset; } DLTensor;
typedef struct DLManagedTensor { DLTensor dl_tensor; void* manager_ctx; void (*deleter)(struct DLManagedTensor*); } DLManagedTensor;
}

namespace {

void check(int rc, const char* what) {
  if (rc < 0) throw std::runtime_error(std::string(what) + ": " + rsb_last_error());
}

struct ModelHandle {
  rsb_model* m = nullptr;
  explicit ModelHandle(const std::string& urdf) { check(rsb_model_create_from_urdf(urdf.c_str(), &m), "Model"); }
  ~ModelHandle() { if (m) rsb_model_destroy(m); }
};

struct Holder {               // keeps the batch alive as long as a tensor made from it
  std::shared_ptr<void> keep;
  int64_t shape[2], strides[2];
};
void dl_deleter(DLManagedTensor* t) { delete static_cast<Holder*>(t->manager_ctx); delete t; }
void capsule_destructor(PyObject* cap) {
  if (PyCapsule_IsValid(cap, "dltensor")) {     // never consumed: free it ourselves (a consumer renames the capsule to "used_dltensor")
    auto* t = static_cast<DLManagedTensor*>(PyCapsule_GetPointer(cap, "dltensor"));
    if (t && t->deleter) t->deleter(t);
  }
}

class Batch : public std::enable_shared_from_this<Batch> {
 public:
  Batch(std::shared_ptr<ModelHandle> model, int num_envs, int device) : model_(std::move(model)), device_(device) {
    check(rsb_batch_create(model_->m, num_envs, device, &b_), "Batch");
    check(rsb_batch_device_ptrs(b_, &view_), "device_ptrs");
  }
  ~Batch() { if (b_) rsb_batch_destroy(b_); }
  rsb_batch* raw() const { return b_; }

  py::capsule tensor(float* base, int64_t rows, int64_t cols, int64_t row_stride) {
    auto* h = new Holder;
    h->keep = shared_from_this();
    h->shape[0] = rows; h->shape[1] = cols; h->strides[0] = row_stride; h->strides[1] = 1;
    auto* t = new DLManagedTensor;
    t->dl_tensor.data = base;
    t->dl_tensor.device = DLDevice{kDLCUDA, device_};
    t->dl_tensor.ndim = 2;
    t->dl_tensor.dtype = DLDataType{2, 32, 1};
    t->dl_tensor.shape = h->shape; t->dl_tensor.strides = h->strides; t->dl_tensor.byte_offset = 0;
    t->manager_ctx = h; t->deleter = dl_deleter;
    return py::capsule(t, "dltensor", capsule_destructor);
  }
  // zero-copy views of the padded rows the kernel reads and writes: [num_envs, nq | nv], row stride gc_stride | gv_stride
  py::capsule gc() { return tensor(view_.gc, view_.num_envs, view_.nq, view_.gc_stride); }
  py::capsule gv() { return tensor(view_.gv, view_.num_envs, view_.nv, view_.gv_stride); }
  py::capsule tau_ff() { return tensor(view_.tau_ff, view_.num_envs, view_.nv, view_.gv_stride); }
  py::capsule pd_target() { return tensor(view_.ptarget, view_.num_envs, view_.nq, view_.gc_stride); }
  py::capsule pd_velocity_target() { return tensor(view_.vtarget, view_.num_envs, view_.nv, view_.gv_stride); }

  void set_ground(float z) { check(rsb_batch_set_ground(b_, z), "set_ground"); }
  void set_stream(uintptr_t s) { check(rsb_batch_set_stream(b_, reinterpret_cast<void*>(s)), "set_stream"); }
  void set_pd_gains(const std::vector<float>& kp, const std::vector<float>& kd) {
    if ((int)kp.size() != view_.nv || (int)kd.size() != view_.nv) throw std::runtime_error("set_pd_gains: need nv gains");
    check(rsb_batch_set_pd_gains(b_, kp.data(), kd.data()), "set_pd_gains");
  }
  void integrate(int substeps) { check(rsb_batch_integrate(b_, substeps), "integrate"); }
  void update_kinematics() { check(rsb_batch_update_kinematics(b_), "update_kinematics"); }
  void sync() { check(rsb_batch_sync(b_), "sync"); }
  // one control step with everything on the device: obs = DLPack-importable tensor address ([num_envs, ob_dim] float32, contiguous)
  void control_step(uintptr_t ptarget_dev, int substeps, uintptr_t obs_dev) {
    check(rsb_batch_control_step(b_, reinterpret_cast<const float*>(ptarget_dev), nullptr, RSB_DEVICE, substeps, reinterpret_cast<float*>(obs_dev), RSB_DEVICE), "control_step");
  }
  void set_heightmap(int xs, int ys, float x_size, float y_size, float cx, float cy, const std::vector<float>& h) {
    if ((long long)h.size() != (long long)xs * ys) throw std::runtime_error("set_heightmap: need x_samples * y_samples heights");
    check(rsb_batch_set_heightmap(b_, xs, ys, x_size, y_size, cx, cy, h.data()), "set_heightmap");
  }
  // terrain sensing into device memory: out = address of a float32 [env_count, out_stride] tensor (out_stride 0: num_frames * num_points)
  void height_scan(const std::vector<int32_t>& frames, const std::vector<float>& points_xy, uintptr_t out_dev, int out_stride, int env_begin, int env_count) {
    if (points_xy.size() % 2) throw std::runtime_error("height_scan: points_xy holds (x, y) pairs");
    const int np = (int)(points_xy.size() / 2);
    if (env_count < 0) env_count = view_.num_envs - env_begin;
    check(rsb_batch_height_scan(b_, frames.data(), (int)frames.size(), points_xy.data(), np, reinterpret_cast<float*>(out_dev),
                                out_stride > 0 ? out_stride : (int)frames.size() * np, env_begin, env_count, RSB_DEVICE), "height_scan");
  }
  // rays fixed in frames (origins / dirs: flat host lists of num_rays * 3); out = address of [env_count, num_frames, num_rays] 32-byte records
  void ray_test(const std::vector<int32_t>& frames, const std::vector<float>& origins, const std::vector<float>& dirs, float length, uintptr_t out_dev,
                int env_begin, int env_count) {
    if (frames.empty() || origins.size() % 3 || dirs.size() != origins.size()) throw std::runtime_error("ray_test: need frames and num_rays * 3 origins and directions");
    if (env_count < 0) env_count = view_.num_envs - env_begin;
    check(rsb_batch_ray_test(b_, frames.data(), (int)frames.size(), origins.data(), dirs.data(), (int)(origins.size() / 3), length,
                             reinterpret_cast<rsb_ray_hit*>(out_dev), env_begin, env_count, RSB_DEVICE), "ray_test");
  }
  // world-frame rays from device memory: origins / dirs = addresses of float32 [env_count, num_rays, 3] tensors
  void ray_test_world(uintptr_t origins_dev, uintptr_t dirs_dev, int num_rays, float length, uintptr_t out_dev, int env_begin, int env_count) {
    if (env_count < 0) env_count = view_.num_envs - env_begin;
    check(rsb_batch_ray_test(b_, nullptr, 0, reinterpret_cast<const float*>(origins_dev), reinterpret_cast<const float*>(dirs_dev), num_rays, length,
                             reinterpret_cast<rsb_ray_hit*>(out_dev), env_begin, env_count, RSB_DEVICE), "ray_test_world");
  }
  int num_envs() const { return view_.num_envs; }
  int nq() const { return view_.nq; }
  int nv() const { return view_.nv; }
  int ob_dim() const { return rsb_batch_ob_dim(b_); }
  long launch_count() const { return (long)rsb_batch_launch_count(b_); }

 private:
  std::shared_ptr<ModelHandle> model_;
  rsb_batch* b_ = nullptr;
  rsb_device_view view_{};
  int device_ = 0;
};

}  // namespace

PYBIND11_MODULE(_rsb_py, m) {
  m.doc() = "raisimlib_b200: batched World::integrate() on the GPU, device state as DLPack tensors (zero-copy)";
  py::class_<ModelHandle, std::shared_ptr<ModelHandle>>(m, "Model").def(py::init<const std::string&>(), py::arg("urdf_path_or_xml"));
  py::class_<Batch, std::shared_ptr<Batch>>(m, "Batch")
      .def(py::init<std::shared_ptr<ModelHandle>, int, int>(), py::arg("model"), py::arg("num_envs"), py::arg("device") = 0)
      .def("gc", &Batch::gc, "generalized coordinates [num_envs, nq] as a DLPack capsule (zero-copy view of the batch rows)")
      .def("gv", &Batch::gv)
      .def("tau_ff", &Batch::tau_ff)
      .def("pd_target", &Batch::pd_target)
      .def("pd_velocity_target", &Batch::pd_velocity_target)
      .def("set_ground", &Batch::set_ground)
      .def("set_stream", &Batch::set_stream)
      .def("set_pd_gains", &Batch::set_pd_gains)
      .def("integrate", &Batch::integrate, py::arg("substeps") = 1)
      .def("update_kinematics", &Batch::update_kinematics)
      .def("control_step", &Batch::control_step)
      .def("sync", &Batch::sync)
      .def("set_heightmap", &Batch::set_heightmap, py::arg("x_samples"), py::arg("y_samples"), py::arg("x_size"), py::arg("y_size"), py::arg("center_x"),
           py::arg("center_y"), py::arg("heights"))
      .def("height_scan", &Batch::height_scan, py::arg("frames"), py::arg("points_xy"), py::arg("out"), py::arg("out_stride") = 0, py::arg("env_begin") = 0,
           py::arg("env_count") = -1, "height scan into a device tensor (address): rsb_batch_height_scan")
      .def("ray_test", &Batch::ray_test, py::arg("frames"), py::arg("origins"), py::arg("dirs"), py::arg("length"), py::arg("out"), py::arg("env_begin") = 0,
           py::arg("env_count") = -1, "frame-attached rays into a device buffer of 32-byte records (address): rsb_batch_ray_test")
      .def("ray_test_world", &Batch::ray_test_world, py::arg("origins"), py::arg("dirs"), py::arg("num_rays"), py::arg("length"), py::arg("out"),
           py::arg("env_begin") = 0, py::arg("env_count") = -1, "world-frame rays from device tensors (addresses): rsb_batch_ray_test")
      .def_property_readonly("num_envs", &Batch::num_envs)
      .def_property_readonly("nq", &Batch::nq)
      .def_property_readonly("nv", &Batch::nv)
      .def_property_readonly("ob_dim", &Batch::ob_dim)
      .def_property_readonly("launch_count", &Batch::launch_count);
}
