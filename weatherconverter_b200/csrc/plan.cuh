// Shared scaffolding of the model-level launch plans (unet.cu, unet_train.cu, legacy.cu, seg.cu, srgan.cu): parameter
// table, bump allocator over the host-provided workspace, op lists, the builder base every plan builder derives from,
// and the binding / workspace-query templates.
//
// Each plan handle has a `Geom` (the shape key of a binding, with ==), `geom` / `ws` / `ws_bytes` (the current binding),
// `arena`, `params`, `reset_plan()` (drops the ops and FLOP counts of the current plan) and a
//   int build(const Net& net, const Net::Geom& g, Net* out, cudaStream_t st, size_t* need)
// that builds the plan for `g` into `out` over out->ws, or, with out == nullptr (a dry build), only measures the workspace
// the plan needs into *need without touching the handle or the device.
#pragma once
#include <functional>
#include <string>
#include <unordered_map>
#include <vector>

#include "conv.cuh"

namespace wc {

class Bump {
 public:
  Bump() = default;
  Bump(void* base, size_t cap) : base_(static_cast<uint8_t*>(base)), cap_(cap) {}
  void* take(size_t bytes) {
    const size_t off = (off_ + 255) & ~static_cast<size_t>(255);
    off_ = off + bytes;
    if (!base_ || off_ > cap_) { overflow_ = true; return nullptr; }
    return base_ + off;
  }
  size_t used() const { return off_; }
  bool overflow() const { return overflow_; }
  static Bump dry() { return Bump(reinterpret_cast<void*>(static_cast<uintptr_t>(4096)), ~static_cast<size_t>(0) >> 1); }

 private:
  uint8_t* base_ = nullptr;
  size_t cap_ = 0, off_ = 0;
  bool overflow_ = false;
};

struct ParamTable {
  std::unordered_map<std::string, const float*> ptr;
  const float* get(const std::string& name, int* err) const {
    auto it = ptr.find(name);
    if (it == ptr.end()) {
      if (!*err) *err = fail("missing parameter '" + name + "'");
      return nullptr;
    }
    return it->second;
  }
};

using OpList = std::vector<std::function<int(cudaStream_t)>>;

inline int run_ops(const OpList& ops, cudaStream_t st) {
  for (auto& op : ops)
    if (int e = op(st)) return e;
  return 0;
}

inline Act make_act(Bump& bump, int B, int H, int W, int C) {
  Act a;
  a.B = B; a.H = H; a.W = W; a.C = C; a.ld = C;
  a.ptr = static_cast<__nv_bfloat16*>(bump.take(a.pixels() * C * sizeof(__nv_bfloat16)));
  return a;
}
inline Act slice_act(const Act& a, int c0, int C) {
  Act v = a;
  v.ptr = a.ptr ? a.ptr + c0 : nullptr;
  v.C = C;
  return v;
}

// Base of the plan builders.  `net` is the handle the plan is built into, nullptr in a dry build: a dry build only takes
// workspace, so it reads no parameter, records no op and allocates nothing on the device.
template <class Net>
struct PlanBuilder {
  Net* net;
  Bump bump;
  DeviceArena* arena;
  cudaStream_t st;
  bool dry;
  int B;
  int err = 0;

  PlanBuilder(Net* out, int B, cudaStream_t st)
      : net(out), bump(out ? Bump(out->ws, out->ws_bytes) : Bump::dry()), arena(out ? out->arena.get() : nullptr), st(st),
        dry(!out), B(B) {}

  const float* P(const std::string& name) { return dry ? nullptr : net->params.get(name, &err); }
  Act act(int H, int W, int C) { return make_act(bump, B, H, W, C); }

  // End of a build: a dry build reports the workspace it took (plus alignment slack), a real one fails if it did not fit.
  int finish(const char* model, size_t* need) {
    if (err) return err;
    if (dry) *need = bump.used() + 4096;
    else if (bump.overflow()) return fail(std::string(model) + " workspace too small: need " + std::to_string(bump.used()) + " bytes");
    return 0;
  }
};

template <class Net>
using BuildFn = int (*)(const Net&, const typename Net::Geom&, Net*, cudaStream_t, size_t*);

// Builds the plan for geometry g over `ws` into `net`, unless `net` is bound to exactly these already (`rebuild`: always).
template <class Net>
int bind(Net* net, const typename Net::Geom& g, void* ws, size_t ws_bytes, cudaStream_t st, BuildFn<Net> build,
         bool rebuild = false) {
  if (!rebuild && net->geom == g && net->ws == ws && net->ws_bytes == ws_bytes) return 0;
  net->reset_plan();
  net->arena = std::make_unique<DeviceArena>();
  net->geom = g; net->ws = ws; net->ws_bytes = ws_bytes;
  if (int e = build(*net, g, net, st, nullptr)) {
    net->geom = {};
    net->reset_plan();
    return e;
  }
  return 0;
}

// Workspace bytes the plan for geometry g needs (0 if it cannot be built), from a dry build.
template <class Net>
size_t plan_workspace_bytes(const Net& net, const typename Net::Geom& g, BuildFn<Net> build) {
  size_t need = 0;
  return build(net, g, nullptr, nullptr, &need) == 0 ? need : 0;
}

}  // namespace wc
