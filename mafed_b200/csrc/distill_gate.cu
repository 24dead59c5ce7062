// The gated backward of the one-pass step (mafed_distill_bwd with skip_if_equals).
//
// The one-pass step writes its gradients during the forward, for an ASSUMED upstream gradient.  When autograd later
// delivers the real one, somebody has to compare the two -- on the device, because the value lives there -- and to
// redo the backward exactly if they differ.  Round 1 launched the whole persistent backward grid (148 CTAs x 544
// threads x 131 KB of shared memory) just to let every CTA read one float and return: 3.5 us of a drained GPU per
// step (tools/probes/cdp_probe.cu: 7.5 vs 4.0 us per iteration).  Here the comparison is a 1-CTA kernel, and only
// when it fails does that kernel start the real backward itself, as a device-side launch into its tail-launch
// stream: the backward then runs after the gate and before anything that follows the gate in the stream, exactly as
// if the host had launched it.  An idle gate costs 0.1-0.2 us next to no launch at all (same probe).
//
// Device-side launches need relocatable device code, which changes register allocation (ABI-conforming calls), so
// this unit is compiled separately (-rdc=true, device-linked with cudadevrt) and instantiates its OWN copies of the
// backward kernels in namespace mafed_gate; every ordinary launch keeps using the whole-program-compiled kernels of
// distill_abi.cu.
#define MAFED_NS mafed_gate
#define MAFED_DEVICE_LAUNCH 1
#include "distill_gate.h"

#include <atomic>
#include <type_traits>

#include "distill_dispatch.cuh"

namespace mafed_gate {
namespace {

struct GateArgs {
  const float* grad_out;   // device scalar or nullptr (= 1)
  float scale;             // host factor on *grad_out
  float assumed;           // the upstream gradient the forward baked in
  float* seen;             // optional: where to leave the upstream gradient that really arrived
  unsigned grid, block, smem;
};

struct NoExtra {};

// Kernel: the tag of the backward kernel to start (distill_dispatch.cuh); Extra: its second parameter, if any
// (the ring geometry of the TMA kernels, the flag of the generic one).
template <typename Kernel, typename Extra>
__global__ void __launch_bounds__(32) k_gate(const GateArgs ga, const PathParams p, const Extra x) {
  pdl_wait();   // the producer of *grad_out has completed
  if (threadIdx.x != 0) return;
  const float g = (ga.grad_out != nullptr ? *ga.grad_out : 1.f) * ga.scale;
  if (ga.seen != nullptr) *ga.seen = g;
  if (g == ga.assumed) return;
  if constexpr (std::is_same<Extra, NoExtra>::value) Kernel::tail_launch(ga.grid, ga.block, ga.smem, p);
  else Kernel::tail_launch(ga.grid, ga.block, ga.smem, p, x);
}

// Launcher policy: instead of the kernel itself, enqueue its gate.
struct GateLaunch {
  cudaStream_t st;
  bool pdl;
  GateArgs ga;
  template <typename Kernel, typename Extra>
  void gate(unsigned grid, unsigned block, size_t smem, const PathParams& p, const Extra& x) const {
    GateArgs a = ga;
    a.grid = grid;
    a.block = block;
    a.smem = (unsigned)smem;
    launch_pdl(k_gate<Kernel, Extra>, 1, 32, 0, st, pdl, a, p, x);
  }
  template <typename Kernel>
  void run(unsigned grid, unsigned block, size_t smem, const PathParams& p) const {
    gate<Kernel, NoExtra>(grid, block, smem, p, NoExtra{});
  }
  template <typename Kernel, typename Extra>
  void run(unsigned grid, unsigned block, size_t smem, const PathParams& p, const Extra& x) const {
    gate<Kernel, Extra>(grid, block, smem, p, x);
  }
};

}  // namespace

// The kernel that follows a gate in its stream must not be a programmatic dependent of it.  A dependent launch may
// become resident as soon as the gate's single block has exited -- while the backward the gate started from the
// device is still waiting to be scheduled -- and a resident persistent grid (one CTA per SM, most of the shared
// memory each) blocked in griddepcontrol.wait would then hold exactly the resources that backward needs: the
// dependent waits for the gate's grid (children included) to complete, the child waits for an SM.  So the library
// remembers the streams a gate went to and launches its next kernel there fully serialised (the only cost: that
// kernel's launch latency is not hidden behind a 2 us gate; kernels of other libraries are not programmatic launches).
namespace {
constexpr int kGateMarks = 16;
std::atomic<uintptr_t> g_gate_marks[kGateMarks];
inline uintptr_t stream_key(void* stream) { return reinterpret_cast<uintptr_t>(stream) + 1; }   // 0 = empty slot
}  // namespace

void note_gate_launch(void* stream) {
  const uintptr_t key = stream_key(stream);
  for (auto& m : g_gate_marks)
    if (m.load(std::memory_order_relaxed) == key) return;
  for (auto& m : g_gate_marks) {
    uintptr_t empty = 0;
    if (m.compare_exchange_strong(empty, key)) return;
  }
  g_gate_marks[key % kGateMarks].store(key);     // table full: overwrite (the displaced stream loses only its mark)
}

bool consume_gate_mark(void* stream) {
  const uintptr_t key = stream_key(stream);
  for (auto& m : g_gate_marks) {
    uintptr_t expect = key;
    if (m.load(std::memory_order_relaxed) == key && m.compare_exchange_strong(expect, 0)) return true;
  }
  return false;
}

int gated_backward(const mafed_shape_t* shape, const void* const* student_ptrs, const void* const* teacher_ptrs,
                   void* const* grad_ptrs, const int64_t* attn_mask, const float* bwd_scale, const float* grad_out,
                   float grad_out_scale, float assumed, float* grad_out_seen, void* stream) {
  PathParams p;
  int rc = fill_params(shape, student_ptrs, teacher_ptrs, grad_ptrs, attn_mask, p);
  if (rc) return rc;
  p.bwd_scale = bwd_scale;
  p.grad_out = grad_out;       // the started kernel reads the upstream gradient itself
  p.gout_scale = grad_out_scale;
  const bool pdl = !consume_gate_mark(stream);   // (a gate right behind a gate)
  GateLaunch go{(cudaStream_t)stream, pdl, GateArgs{grad_out, grad_out_scale, assumed, grad_out_seen, 0, 0, 0}};
  rc = dispatch<kPassBwd>(*shape, p, go);
  note_gate_launch(stream);
  return rc;
}

}  // namespace mafed_gate
