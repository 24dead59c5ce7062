#!/usr/bin/env python
"""Benchmark of the MAFED distillation hot path (fused forward + backward) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload C4|C2|C3|C1] [--impl ours|reference]
                    [--dump-outputs DIR]

Metric (BASELINE.json): distill fwd+bwd tokens*layers/sec, and the fraction of HBM peak.
A "step" is one pass of the hot path (forward over all selected layers, loss algebra, backward) over one
synthetic batch of hidden states, through the call a user makes: ``FeatureDistillation.distill`` then
``loss.backward()``.  Default workload: the VLPythia-1B shape the metric is quoted on (C4: 16 layers -> 15
distilled, D=2048, T=256+32, bf16) at 64 samples per GPU, i.e. weak scaling to C4's global batch 512 on 8 GPUs.
Prints ONE JSON line on rank 0.  Besides the contract's keys the line carries:

  roofline          the fused kernel against the measured HBM peak (CUDA events around every launch)
  two_pass          north_star's two-kernel form (5*D*e bytes per token*layer)
  other_workloads   C2 / C3 / C1 and cosine / fp32-input variants through the same API (N=1)
  c5                BASELINE configs[4]: per-GPU batch 8..128 x text 32 / 256 x all-ones / ragged masks, through
                    the API and at kernel level, at this N
  sharded_parity    (N>1) one small ragged step sharded over the ranks against the same step on the concatenated
                    batch on one GPU and against the CPU oracle; the run FAILS if it is out of tolerance
  e2e               the same metric with HOST buffers through the C ABI's host step (copies inside the timed region)
  cpu_baseline      the UNMODIFIED reference (oracle/_ref) on the host cores, full per-GPU shard
``--impl reference`` times that unmodified reference alone (rank 0 only).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # a run leaves the tree as it found it (it may be read-only): no __pycache__ there

METRIC = "distill fwd+bwd tokens*layers/sec"
UNIT = "tokens*layers/s"

WORKLOADS = {
    # name: (description, hidden-state tuple length, distilled layers (reference rule L-1), per-GPU B, txt, D, dtype)
    "C4": ("VLPythia-1B (16 layers, d=2048) all-layer MAFED distillation, bf16, 64 samples/GPU (C4 shard; 512 on 8 GPUs)",
           17, 15, 64, 32, 2048, "bf16"),
    "C2": ("VLPythia-base (12 layers, d=768) MAFED distillation, batch 128, bf16", 13, 11, 128, 32, 768, "bf16"),
    "C3": ("VLPythia-410M (24 layers, d=1024) MAFED distillation, batch 256, bf16", 25, 23, 256, 32, 1024, "bf16"),
    "C1": ("VLPythia-base MAFED distillation, batch 8, fp32", 13, 11, 8, 32, 768, "fp32"),
}
N_VIS = 256
RECIPE = dict(modality="balanced", layer_strategy="discounted", loss="mse", gamma=0.5)  # scripts/run_seed42.sh:74-93


def measured_traffic(wl):
    """DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` capture (profiles/)."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f).get(wl, {}).get("fused_kernel_dram_bytes")
    return None


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    """Samples SM clock + throttle reasons during the timed region (pynvml, else nvidia-smi)."""

    def __init__(self, index):
        self.index = index
        self.samples, self.reasons = [], set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._go = threading.Event()
        self._thread = None
        self._nv = self._handle = None
        try:                                    # set up before the timed region: a 10 ms region must still be sampled
            import pynvml as nv
            nv.nvmlInit()
            self._handle = nv.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(self._handle, nv.NVML_CLOCK_SM)
            self._nv = nv
        except Exception:
            self._nv = None

    def _loop_nvml(self):
        nv, h = self._nv, self._handle
        if nv is None:
            raise RuntimeError("no nvml")
        names = {
            getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksThrottleReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake_slowdown",
        }
        self._go.wait()                         # the thread exists before the barrier; it samples from `go()` on
        time.sleep(0.001)                       # let the first launches reach the GPU
        while not self._stop.is_set():
            self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
            try:
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            if self._stop.wait(0.003):
                break

    def _loop_smi(self):
        import subprocess
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        self._go.wait()
        while not self._stop.is_set():
            out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                 capture_output=True, text=True).stdout.strip().split(",")
            if len(out) >= 6:
                self.samples.append(int(float(out[0])))
                self.max_mhz = int(float(out[1]))
                for n, v in zip(names, out[2:]):
                    if v.strip().lower().startswith("active"):
                        self.reasons.add(n)

    def __enter__(self):
        def run():
            try:
                self._loop_nvml()
            except Exception:
                try:
                    self._loop_smi()
                except Exception:
                    pass
        self._thread = threading.Thread(target=run, daemon=True)
        self._thread.start()
        return self

    def go(self):
        """Start sampling: called right after the timed region's first event is recorded."""
        self._go.set()

    def __exit__(self, *exc):
        self._stop.set()
        self._go.set()
        self._thread.join(timeout=5)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": 0}
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ----------------------------------------------------------------------------- workload
def torch_dtype(name):
    return {"bf16": torch.bfloat16, "fp32": torch.float32, "fp16": torch.float16}[name]


def make_device_inputs(wl, rank, device):
    _, n_tuple, n_sel, B, txt, D, dt = WORKLOADS[wl]
    g = torch.Generator(device=device).manual_seed(1234 + rank)
    T = N_VIS + txt
    st, te = [], []
    for _ in range(n_sel):
        s = torch.randn(B, T, D, generator=g, device=device, dtype=torch.float32)
        t = s + 0.1 * torch.randn(B, T, D, generator=g, device=device, dtype=torch.float32)
        st.append(s.to(torch_dtype(dt)))
        te.append(t.to(torch_dtype(dt)))
        del s, t
    # headline runs use an all-ones mask so that byte accounting is unambiguous (SURVEY 8d)
    am = torch.ones(B, txt, dtype=torch.int64, device=device)
    return st, te, am


class Opts:
    tasks = ["a", "b", "c"]
    batch_size = 64
    seed = 42
    pin_mem = False
    accumulate_grad_batches = 1


class Out:
    def __init__(self, hs):
        self.hidden_states = hs


def make_method(n_sel, loss=None):
    from mafed_b200.methods import CLMethod
    return CLMethod["featdistill"](
        memory_size=8, opts=Opts(), model_type="vlpythia",
        distillation_modality_weighing_strategy=RECIPE["modality"],
        distillation_layer_weighing_strategy=RECIPE["layer_strategy"], distillation_coeff=1.0,
        distillation_layer=None, distillation_loss=loss or RECIPE["loss"], gamma=RECIPE["gamma"],
        num_hidden_layers=n_sel)


# ----------------------------------------------------------------------------- CPU baseline (the unmodified reference)
def cpu_reference_steps(wl, steps, warmup, budget_s=150.0):
    """``FeatureDistillation.distill`` + ``backward()`` of the UNMODIFIED reference (oracle/_ref: byte-identical
    copies of mafed/methods/*.py, imported with stubbed third-party modules) on CPU tensors of the full per-GPU
    shard, under ``torch.autocast("cpu", bfloat16)`` for the bf16 workloads (what ``replay`` does on the GPU,
    distillation.py:90), with every host thread torch can use.  If the reference files are not there the oracle
    restatement is timed instead and says so (kind "port")."""
    from oracle import distill_oracle as O
    from oracle import ref_harness as R
    _, n_tuple, n_sel, B, txt, D, dt = WORKLOADS[wl]
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    st, te, am = O.make_inputs(n_sel, B, txt, D, n_vis=N_VIS, dtype=torch_dtype(dt), seed=1234, teacher="close",
                               mask="full")
    kind = "reference" if R.available() else "port"
    if kind == "reference":
        fd = R.make_reference_method(modality=RECIPE["modality"], layer_strategy=RECIPE["layer_strategy"],
                                     loss=RECIPE["loss"], gamma=RECIPE["gamma"], num_hidden_layers=n_sel, n_vis=N_VIS)

        def step():
            return R.reference_forward_backward(fd, st, te, am, autocast_bf16=(dt != "fp32"))["loss"]
    else:
        cfg = O.OracleConfig(modality_strategy=RECIPE["modality"], layer_strategy=RECIPE["layer_strategy"],
                             gamma=RECIPE["gamma"], num_hidden_layers=n_sel, distillation_layer=None,
                             loss=RECIPE["loss"], num_vision_tokens=N_VIS)

        def step():
            return O.forward_backward(st, te, am, cfg)["loss"]
    times, loss = [], None
    t_start = time.perf_counter()
    done_warm = 0
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        loss = step()
        dt_s = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt_s)
        else:
            done_warm += 1
        if time.perf_counter() - t_start + dt_s > budget_s and times:
            break    # bounded: never let the baseline leg run for more than a few minutes
    units = B * (N_VIS + txt) * n_sel
    mean_s = sum(times) / len(times)
    what = ("unmodified reference FeatureDistillation.distill + backward (oracle/_ref, mafed/methods/distillation.py:105-166)"
            if kind == "reference" else "oracle restatement of distillation.py:105-166 (reference files absent)")
    return {"value": units / mean_s, "unit": UNIT, "cores": cores, "kind": kind,
            "sample": f"{wl} per-GPU shard at full size: B={B} of {B} samples, {n_sel} layers, T={N_VIS + txt}, D={D}, {dt}"
                      f"{' under torch.autocast(cpu, bfloat16)' if dt != 'fp32' else ''}; {what}; torch CPU ops + autograd on "
                      f"{cores} threads; mean of {len(times)} steps after {done_warm} warm-up",
            "ms_per_step": 1e3 * mean_s, "best_ms": 1e3 * min(times), "steps_run": len(times), "warmup_run": done_warm,
            "loss": float(loss)}


def eager_gpu_baseline(wl, st, te, am, iters=5, warmup=2):
    """The reference's own op chain (oracle port: ATen kernels + autograd, distillation.py:105-166 under
    autocast) run on the SAME GPU on the same tensors -- what the unmodified reference would spend on this
    path on a B200.  A baseline leg like `cpu_baseline`; the product never calls it."""
    from oracle import distill_oracle as O
    _, n_tuple, n_sel, B, txt, D, dt = WORKLOADS[wl]
    cfg = O.OracleConfig(modality_strategy=RECIPE["modality"], layer_strategy=RECIPE["layer_strategy"],
                         gamma=RECIPE["gamma"], num_hidden_layers=n_sel, distillation_layer=None, loss=RECIPE["loss"],
                         num_vision_tokens=N_VIS)
    leaves = [s.detach().requires_grad_(True) for s in st]

    def step():
        for s in leaves:
            s.grad = None
        with torch.autocast("cuda", dtype=torch.bfloat16):
            total, per_layer, _ = O.distill(leaves, te, am, cfg)
            _ = [float(v) for v in per_layer.values()]      # the reference's per-layer .item() for W&B (:165)
        total.backward()

    for _ in range(warmup):
        step()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(iters):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / iters
    units = B * (N_VIS + txt) * n_sel
    return {"value": units / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms,
            "what": "reference op chain (oracle port, eager PyTorch ATen kernels + autograd, autocast bf16) on this GPU"}


def run_reference_arm(args):
    """`--impl reference`: the unmodified reference's CPU implementation of the path on this box's host cores, same
    config / metric / unit as the main arm.  Rank 0 alone runs and prints it."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = args.workload
    _, n_tuple, n_sel, B, txt, D, dt = WORKLOADS[wl]
    base = cpu_reference_steps(wl, steps=max(1, args.steps), warmup=max(0, args.warmup))
    line = {
        "impl": "reference", "metric": METRIC, "value": base["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": base["steps_run"], "warmup": base["warmup_run"], "ms_per_step": base["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": dt, "data": "synthetic",
        "config": workload_config(wl, args.gpus),
        "cpu_baseline": {k: base[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "loss": base["loss"],
        "note": "per-GPU shard on the host cores (the reference has no multi-GPU path, README.md:47); per-unit "
                "throughput does not depend on --gpus",
    }
    emit(line)


def workload_config(wl, n_gpus):
    desc, n_tuple, n_sel, B, txt, D, dt = WORKLOADS[wl]
    return {"workload": desc, "id": wl, "layers_distilled": n_sel, "hidden_state_tuple": n_tuple, "D": D,
            "T": N_VIS + txt, "n_vis": N_VIS, "per_gpu_batch": B, "global_batch": B * n_gpus,
            "recipe": "mse/balanced/discounted gamma=0.5", "mask": "all-ones",
            "l2": "inputs (student+teacher) far larger than the 126 MB L2; no explicit flush",
            "parallelism": f"batch-sharded dp{n_gpus}, one allreduce of 2L+2 fp64"}


# ----------------------------------------------------------------------------- output
_REAL_STDOUT = None


def claim_stdout():
    """Route everything libraries print to stdout (NCCL's version banner, warnings) to stderr so that
    stdout carries exactly one line: the JSON result."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


DUMP_GRAD_BYTES = 32 << 20      # budget of the sampled gradient rows; every dump stays under 64 MB


def dump_outputs(out_dir, loss, fd, leaves, batch):
    """Write what the caller of the timed path received from its last step, as ``out_dir/<name>.npy``:

      loss             float64 ()           the returned loss
      layer_losses     float32 (L,)         the per-layer values the step logs (W&B payload)
      lang_masks       float32 (B, T)       the masks the step leaves in ``batch``
      image_masks      float32 (B, T)
      grad_rows        float32 (L, R, D)    rows ``grad_row_index`` of every distilled layer's gradient, flattened to
                                            (B*T, D): a fixed sample (seed 0) of R rows, R set by DUMP_GRAD_BYTES
      grad_row_index   float64 (R,)
      grad_row_sums    float64 (L, B, T)    the sum over D of every gradient row, so that no element goes unchecked

    The inputs depend only on the arguments, so two builds run with the same arguments can be compared file by file."""
    import numpy as np
    L = len(fd.last_layers)
    grads = [leaves[l].grad for l in fd.last_layers]
    B, T, D = grads[0].shape
    rows = min(B * T, max(1, DUMP_GRAD_BYTES // (L * D * 4)))
    index = torch.randperm(B * T, generator=torch.Generator().manual_seed(0))[:rows].sort().values
    idx_dev = index.to(grads[0].device)
    arrays = {
        "loss": np.asarray(float(loss.detach()), dtype=np.float64),
        "layer_losses": fd.last_layer_losses[:L].float().cpu().numpy(),
        "lang_masks": batch["lang_masks"].float().cpu().numpy(),
        "image_masks": batch["image_masks"].float().cpu().numpy(),
        "grad_rows": torch.stack([g.reshape(B * T, D)[idx_dev].float() for g in grads]).cpu().numpy(),
        "grad_row_index": index.double().numpy(),
        "grad_row_sums": torch.stack([g.double().sum(-1) for g in grads]).cpu().numpy(),
    }
    total = sum(a.nbytes for a in arrays.values())
    assert total <= 64 << 20, f"--dump-outputs would write {total} bytes"
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ----------------------------------------------------------------------------- helpers of the main arm
class Ctx:
    """Process-wide facts of one bench run."""

    def __init__(self, args):
        import torch.distributed as dist
        self.args = args
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local_rank)
        self.device = torch.device("cuda", self.local_rank)
        self.dist = dist
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.device)
        self.peak, self.peak_src = peaks()

    def sync_all(self, align=False):
        """Barrier + device synchronize.  ``align``: the ranks additionally leave together -- NCCL's barrier lets them go
        ~160 us apart (measured: `start_skew.barrier_exit_spread_us` before this was added), which a K-step timed
        region of a coupled step pays once, i.e. 8 us per step at K = 20; so they agree on a moment of the system-wide
        monotonic clock 300 us after the last one arrived and spin until then."""
        torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
            torch.cuda.synchronize()
            if align:
                t = torch.tensor([time.perf_counter()], dtype=torch.float64, device=self.device)
                self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
                go_at = float(t) + 300e-6
                torch.cuda.synchronize()
                while time.perf_counter() < go_at:
                    pass

    def max_over_ranks(self, values):
        t = torch.tensor(list(values), dtype=torch.float64, device=self.device)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return t.tolist()


class ApiLoop:
    """The user's call, step after step: ``fd.distill(output, batch)`` then ``loss.backward()``.  Across batch shards
    the token counts of a batch leave for the peers when the batch is "drawn" (``fd.prefetch_counts``, what ``replay``
    does as soon as it has a memory batch, a whole student forward ahead of ``distill``).  There is no forward here,
    so the loop draws two batches ahead: once step i is launched it sends the counts of batch i+2; the 1-CTA prefetch
    (ordered behind the work already on the stream, because it reads the mask) then runs beside step i+1 and never
    sits between two steps.  Three mask tensors rotate so that a prefetched batch is a different object from the ones
    in use."""

    def __init__(self, ctx, fd, leaves, masks):
        self.ctx, self.fd, self.leaves = ctx, fd, leaves
        self.prefetch = ctx.world > 1
        self.masks = list(masks) + ([masks[0].clone()] if self.prefetch else [])
        self.out = Out(tuple(leaves))
        self.i = 0

    def prime(self):
        if self.prefetch and self.fd.process_group is not False:
            n = len(self.masks)
            for m in (self.masks[self.i % n], self.masks[(self.i + 1) % n]):
                tk = self.fd._tickets.get(id(m))
                if tk is None or tk[0] is not m or tk[1] != m._version:      # (still in flight from the last loop)
                    self.fd.prefetch_counts({"attention_mask": m})

    def step(self):
        fd, i = self.fd, self.i
        self.i += 1
        for s in self.leaves:
            s.grad = None
        n = len(self.masks)
        self.batch = {"attention_mask": self.masks[i % n]}
        loss = fd.distill(self.out, self.batch)
        loss.backward()
        if self.prefetch and fd.process_group is not False:
            fd.prefetch_counts({"attention_mask": self.masks[(i + 2) % n]})
        return loss

    def timed(self, steps, warmup, sampler=None, snapshot=None):
        """(GPU ms for `steps` steps, host us per step to enqueue one, last loss).  ``snapshot(k)``: called with 0
        where the timed region opens and 1 where it closes (stream-ordered diagnostics; must not synchronise)."""
        self.prime()
        for _ in range(warmup):
            self.step()
        ec, e0, e1 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        cm = sampler if sampler is not None else _Null()
        with cm:        # (the sampler's thread is created before the barrier, so that the ranks leave it together)
            self.ctx.sync_all(align=True)
            t_barrier = time.perf_counter()
            # The K timed steps run between two events on the device.  The opening event is queued behind ONE more
            # untimed step issued after the barrier, so the region starts with the GPU busy and the host a step ahead
            # -- the state every step of a training run is in -- instead of with an idle GPU waiting ~0.15-0.5 ms for
            # the first launch to arrive (at N > 1: for the slowest rank's first launch; 2-5 % of a 20-step region).
            # `cold_ms_per_step` is the same loop timed from the barrier, that step and its launch latency included.
            ec.record()
            self.step()
            self.first_step_enqueued_us = (time.perf_counter() - t_barrier) * 1e6
            t0 = time.perf_counter()
            e0.record()
            if snapshot is not None:
                snapshot(0)
            cm.go()
            for k in range(steps):
                loss = self.step()
            e1.record()
            if snapshot is not None:
                snapshot(1)
            self.t0_monotonic = t_barrier
            host_us = (time.perf_counter() - t0) / steps * 1e6   # CPU time to enqueue one step (no sync inside)
            self.ctx.sync_all()
        self.cold_ms_per_step = ec.elapsed_time(e1) / (steps + 1)
        return e0.elapsed_time(e1), host_us, loss


class _Null:
    def __enter__(self):
        return self

    def go(self):
        pass

    def __exit__(self, *exc):
        return False


def make_masks(B, txt, device, ragged=False):
    am = torch.ones(B, txt, dtype=torch.int64, device=device)
    if ragged:
        for b in range(B):
            am[b, : txt - (1 + (7 * b) % txt)] = 0       # left-padded, valid length 1 + (7 b mod txt) (SURVEY 8d)
    return [am, am.clone()]


def synth(n_sel, B, T, D, dtype, device, seed):
    g = torch.Generator(device=device).manual_seed(seed)
    st, te = [], []
    for _ in range(n_sel):
        s = torch.randn(B, T, D, generator=g, device=device, dtype=torch.float32)
        t = s + 0.1 * torch.randn(B, T, D, generator=g, device=device, dtype=torch.float32)
        st.append(s.to(dtype))
        te.append(t.to(dtype))
        del s, t
    return st, te


def live_rows(masks, n_vis):
    """Rows the kernels really stream: visual rows + valid text rows (padded rows are neither read nor, beyond the
    zero fill, computed)."""
    am = masks[0]
    return int(am.shape[0]) * n_vis + int(am.sum())


# ----------------------------------------------------------------------------- sharded parity (N > 1)
def sharded_parity(ctx):
    """SURVEY 8(e): the N-GPU result (loss and the concatenation of the per-rank gradients) must equal the
    single-device result on the full concatenated batch.  One small step with per-rank ragged masks (every rank holds
    a different number of valid text tokens, which is exactly what separates global from per-rank normalisation),
    fp32 and bf16; the concatenated batch is recomputed on this GPU with the exchange off and, on rank 0, by the CPU
    oracle.  Raises if a tolerance is exceeded (fp32 1e-5, bf16 2e-3)."""
    from oracle import distill_oracle as O
    dist, world, rank, device = ctx.dist, ctx.world, ctx.rank, ctx.device
    L, B, txt, D = 3, 3, 8, 256
    result = {"shape": {"layers": L, "per_rank_batch": B, "T": N_VIS + txt, "D": D}, "tolerance": {"fp32": 1e-5, "bf16": 2e-3}}
    worst_ok = True
    for name, dtype, tol in (("fp32", torch.float32, 1e-5), ("bf16", torch.bfloat16, 2e-3)):
        g = torch.Generator(device="cpu").manual_seed(4321)
        s_all = [torch.randn(world * B, N_VIS + txt, D, generator=g).to(dtype) for _ in range(L)]
        t_all = [(s.float() + 0.3 * torch.randn(world * B, N_VIS + txt, D, generator=g)).to(dtype) for s in s_all]
        am_all = torch.zeros(world * B, txt, dtype=torch.int64)
        for b in range(world * B):
            am_all[b, txt - (1 + (5 * b) % txt):] = 1
        lo, hi = rank * B, (rank + 1) * B

        def run(students, teachers, am, group):
            fd = make_method(L)
            fd.process_group = group
            fd.grad_multiplier = 1.0        # compare hidden-state gradients of the GLOBAL loss (no DDP averaging here)
            leaves = [s.to(device).requires_grad_(True) for s in students]
            tc = [t.to(device) for t in teachers]
            fd.past_model = lambda **kw: Out(tuple(tc))
            loss = fd.distill(Out(tuple(leaves)), {"attention_mask": am.to(device)})
            loss.backward()
            return loss.detach(), [x.grad for x in leaves]

        loss_s, grads_s = run([s[lo:hi] for s in s_all], [t[lo:hi] for t in t_all], am_all[lo:hi], None)
        loss_f, grads_f = run(s_all, t_all, am_all, False)
        torch.cuda.synchronize()
        # gather the per-rank gradients in rank order
        gathered = []
        for gl in grads_s:
            parts = [torch.empty_like(gl) for _ in range(world)]
            dist.all_gather(parts, gl.contiguous())
            gathered.append(torch.cat(parts, 0))
        bits = loss_s.view(torch.int32).reshape(1)
        every = [torch.zeros_like(bits) for _ in range(world)]
        dist.all_gather(every, bits)
        bitwise = all(int(e) == int(every[0]) for e in every)
        loss_rel = abs(float(loss_s) - float(loss_f)) / abs(float(loss_f))
        num = sum(float((a.double() - b.double()).pow(2).sum()) for a, b in zip(gathered, grads_f))
        den = sum(float(b.double().pow(2).sum()) for b in grads_f)
        grad_rel = (num / den) ** 0.5
        entry = {"loss_rel": loss_rel, "grad_rel": grad_rel, "bitwise_equal_across_ranks": bitwise,
                 "loss_sharded": float(loss_s), "loss_single_device": float(loss_f)}
        if rank == 0:
            cfg = O.OracleConfig(modality_strategy=RECIPE["modality"], layer_strategy=RECIPE["layer_strategy"],
                                 gamma=RECIPE["gamma"], num_hidden_layers=L, distillation_layer=None, loss=RECIPE["loss"],
                                 num_vision_tokens=N_VIS)
            ref = O.forward_backward(s_all, t_all, am_all, cfg)
            entry["oracle_loss_rel"] = abs(float(loss_s) - float(ref["loss"])) / abs(float(ref["loss"]))
            n2 = sum(float((a.cpu().double() - r.double()).pow(2).sum()) for a, r in zip(gathered, ref["grads"]))
            d2 = sum(float(r.double().pow(2).sum()) for r in ref["grads"][:L])
            entry["oracle_grad_rel"] = (n2 / d2) ** 0.5
        ok = loss_rel <= tol and grad_rel <= tol and bitwise and entry.get("oracle_loss_rel", 0.0) <= tol \
            and entry.get("oracle_grad_rel", 0.0) <= tol
        entry["within_tolerance"] = bool(ok)
        worst_ok = worst_ok and ok
        result[name] = entry
    result["loss_rel"] = max(result["fp32"]["loss_rel"], result["bf16"]["loss_rel"])
    result["grad_rel"] = max(result["fp32"]["grad_rel"], result["bf16"]["grad_rel"])
    result["bitwise_equal_across_ranks"] = result["fp32"]["bitwise_equal_across_ranks"] and result["bf16"]["bitwise_equal_across_ranks"]
    flag = torch.tensor([0 if worst_ok else 1], device=device)
    dist.all_reduce(flag)
    result["within_tolerance"] = int(flag) == 0
    if int(flag) != 0:
        if rank == 0:
            sys.stderr.write("sharded_parity FAILED: " + json.dumps(result) + "\n")
        raise SystemExit("bench.py: the batch-sharded step does not match the single-device step (sharded_parity)")
    return result


# ----------------------------------------------------------------------------- C5 sweep and other workloads
def measure_point(ctx, n_sel, B, txt, D, dt, ragged, steps, warmup, loss="mse", kernel_level=True, graphed=True, seed=77):
    """One shape through the public API (and at kernel level): tokens*layers/s over ALL ranks, per-GPU GB/s on the
    3*D*e basis counting only the rows that are really streamed."""
    from mafed_b200.distill_op import distill_backward, distill_fused
    device, world = ctx.device, ctx.world
    T = N_VIS + txt
    dtype = torch_dtype(dt)
    esize = torch.finfo(dtype).bits // 8
    st, te = synth(n_sel, B, T, D, dtype, device, seed + ctx.rank)
    masks = make_masks(B, txt, device, ragged)
    fd = make_method(n_sel, loss=loss)
    fd.past_model = lambda **kw: Out(tuple(te))
    leaves = [s.detach().requires_grad_(True) for s in st]
    loop = ApiLoop(ctx, fd, leaves, masks)
    api_ms, host_us, _ = loop.timed(steps, warmup)
    rec = {"per_gpu_batch": B, "txt": txt, "T": T, "mask": "ragged" if ragged else "all-ones"}
    kern_ms = None
    if kernel_level:
        layers = list(range(n_sel))
        coeffs, modality_kind, lang_weights = fd._tables(layers)
        plan = fd._plan(layers, coeffs, fd.distillation_coeff, modality_kind, lang_weights)
        grads = [torch.empty_like(s) for s in st]
        gout = torch.ones((), dtype=torch.float32, device=device)
        tickets = [None, None]

        def kstep(i):
            if world > 1:
                tickets[(i + 1) % 2] = fd.prefetch_counts({"attention_mask": masks[(i + 1) % 2]})
            out, scale, ln = distill_fused(st, te, grads, masks[i % 2], plan, group=None, ticket=tickets[i % 2])
            distill_backward(ln, grads, scale, gout, skip_if_equals=plan.assumed_grad_out * plan.grad_multiplier,
                             grad_out_scale=plan.grad_multiplier)
        if world > 1:
            tickets[0] = fd.prefetch_counts({"attention_mask": masks[0]})
        for i in range(warmup):
            kstep(i)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ctx.sync_all()
        kstep(warmup)                           # (the region opens behind one untimed step, like ApiLoop.timed)
        e0.record()
        for i in range(warmup + 1, warmup + 1 + steps):
            kstep(i)
        e1.record()
        ctx.sync_all()
        kern_ms = e0.elapsed_time(e1)
    graph_ms, graph_host_us = None, None
    if graphed:
        # the same API calls captured once into a CUDA graph and replayed (mafed_b200.graphed): what the step costs a
        # trainer that graphs its training step -- the host no longer walks Python and the autograd engine per step
        from mafed_b200.graphed import GraphedDistillStep
        gfd = make_method(n_sel, loss=loss)
        gstep = GraphedDistillStep(gfd, st, te, masks[0])
        for _ in range(warmup):
            gstep.replay()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ctx.sync_all()
        gstep.replay()                          # (the region opens behind one untimed step, like ApiLoop.timed)
        t0 = time.perf_counter()
        e0.record()
        for _ in range(steps):
            gstep.replay()
        e1.record()
        graph_host_us = (time.perf_counter() - t0) / steps * 1e6
        ctx.sync_all()
        graph_ms = e0.elapsed_time(e1)
        del gstep, gfd
    api_ms, kern_ms_m, graph_ms_m = ctx.max_over_ranks([api_ms, kern_ms if kern_ms is not None else 0.0,
                                                        graph_ms if graph_ms is not None else 0.0])
    ms = api_ms / steps
    units = B * T * n_sel * world
    live = live_rows(masks, N_VIS) * n_sel            # rows streamed on THIS rank (2 reads + 1 write each)
    padded = B * T * n_sel - live                     # padded text rows: never read, only their zero gradient is written
    step_bytes = D * esize * (3 * live + padded)      # SURVEY 8(d): "only the zero-fill write counts"
    gbs = step_bytes / (ms * 1e-3) / 1e9
    rec.update({"value": units / (ms * 1e-3), "ms_per_step": ms, "host_us_per_step": host_us,
                "step_gbs_per_gpu": gbs, "frac": gbs / ctx.peak, "algorithmic_bytes_per_step_per_gpu": step_bytes})
    if kernel_level:
        kms = kern_ms_m / steps
        rec.update({"kernel_level_ms_per_step": kms, "kernel_level_value": units / (kms * 1e-3),
                    "api_over_kernel": ms / kms})
    if graphed:
        gms = graph_ms_m / steps
        rec.update({"graphed_ms_per_step": gms, "graphed_value": units / (gms * 1e-3),
                    "graphed_host_us_per_step": graph_host_us,
                    "graphed_frac": step_bytes / (gms * 1e-3) / 1e9 / ctx.peak})
        if kernel_level:
            rec["graphed_over_kernel"] = gms / (kern_ms_m / steps)
    del st, te, leaves, fd, loop
    return rec


def c5_sweep(ctx, steps=40, warmup=8):
    """BASELINE.json configs[4] / SURVEY 8(d) row C5: VLPythia-1B distillation, 15 layers, bf16, per-GPU batch 8 ..
    1024 / N (global batch up to 1024) x text 32 / 64 / 128 / 256 (visual:text 8:1 .. 1:1) x all-ones / ragged masks
    (ragged at text 32 and 256; the points of 256 samples per GPU and more: all-ones only, fewer steps, no graphed
    leg)."""
    points, skipped = [], []
    for B in (8, 16, 32, 64, 128, 256, 512, 1024):
        if B * ctx.world > 1024:                      # configs[4]: global batch up to 1024
            continue
        for txt in (32, 64, 128, 256):
            resident = 3 * 15 * B * (N_VIS + txt) * 2048 * 2          # student + teacher + gradients, bytes
            if resident > 60e9:
                skipped.append({"per_gpu_batch": B, "txt": txt, "resident_gb": resident / 1e9,
                                "why": "left out to keep the default run's memory bounded (fits the 180 GB part)"})
                continue
            big = B >= 256
            for ragged in ((False,) if big or txt in (64, 128) else (False, True)):
                try:
                    points.append(measure_point(ctx, 15, B, txt, 2048, "bf16", ragged, 12 if big else steps,
                                                4 if big else warmup, graphed=not big))
                except torch.cuda.OutOfMemoryError as exc:      # (a smaller part, or memory held by a neighbour)
                    skipped.append({"per_gpu_batch": B, "txt": txt, "why": "out of memory: " + str(exc)[:80]})
                    torch.cuda.empty_cache()
    small = [p for p in points if p["per_gpu_batch"] == 8 and p["txt"] == 32 and p["mask"] == "all-ones"][0]
    return {"what": "VLPythia-1B (D=2048, 15 distilled layers, bf16): per-GPU batch x text length x mask through "
                    "fd.distill() + loss.backward() (`value`, `ms_per_step`; max over ranks), the same calls captured "
                    "into a CUDA graph and replayed (`graphed_*`), and the kernel-level loop (C-ABI calls from Python, "
                    "no autograd) beside them; GB/s per GPU on the 3*D*e basis over streamed rows",
            "n_gpus": ctx.world, "steps": steps, "warmup": warmup, "points": points, "skipped": skipped,
            "global_batch_range": [8 * ctx.world, max(p["per_gpu_batch"] for p in points) * ctx.world],
            "smallest_point_api_over_kernel": small["api_over_kernel"],
            "smallest_point_graphed_over_kernel": small.get("graphed_over_kernel")}


def other_workloads(ctx, skip, steps=100, warmup=20):
    """The other BASELINE.json configurations that fit one GPU, through the public API (one-pass step), plus the
    cosine loss and fp32 hidden states at the base / 1B shapes.  Informational; the headline stays `value`."""
    out = {}
    rows = [("C2", WORKLOADS["C2"], "mse"), ("C3", WORKLOADS["C3"], "mse"), ("C1", WORKLOADS["C1"], "mse"),
            ("C2_cosine", WORKLOADS["C2"], "cosine"), ("C4_cosine", WORKLOADS["C4"], "cosine"),
            ("C2_fp32", WORKLOADS["C2"][:6] + ("fp32",), "mse"), ("C4_fp32", WORKLOADS["C4"][:6] + ("fp32",), "mse")]
    for name, (desc, n_tuple, n_sel, B, txt, D, dt), loss in rows:
        if name == skip:
            continue
        rec = measure_point(ctx, n_sel, B, txt, D, dt, False, steps, warmup, loss=loss, kernel_level=True,
                            graphed=name in ("C1", "C2"))
        esize = 4 if dt == "fp32" else 2
        rec.update({"workload": desc + (f" [{loss}]" if loss != "mse" else "") + (" [fp32 hidden states]" if name.endswith("fp32") else ""),
                    "unit": UNIT, "bytes_per_unit": 3 * D * esize,
                    "note": "L2-assisted: student+teacher+gradient = 234 MB vs 126 MB L2" if name == "C1" else ""})
        out[name] = rec
    return out


# ----------------------------------------------------------------------------- end to end with host buffers
def run_e2e(ctx, fd, st, te, am, units_per_step):
    """Same metric through the C ABI's host-buffer step (``mafed_host_step_run``) at every N: pinned host
    student / teacher / mask -> device, the one-pass step per layer, gradients and losses -> pinned host, pipelined
    over three streams inside the library; across batch shards the same call carries the communicator (counts sent
    ahead once per step, sums exchanged per layer)."""
    from mafed_b200.host_step import CHostStep
    args, device, world = ctx.args, ctx.device, ctx.world
    hs = CHostStep(fd, st, te, am, device)
    for _ in range(2):
        hs.step()
    ctx.sync_all()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for _ in range(args.e2e_steps):
        loss = hs.step()
    e1.record()
    torch.cuda.synchronize()
    wall_ms = (time.perf_counter() - t0) * 1e3
    (ms,) = ctx.max_over_ranks([max(e0.elapsed_time(e1), wall_ms)])
    ms /= args.e2e_steps
    rec = {"value": units_per_step / (ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": hs.h2d_bytes,
           "d2h_bytes_per_step": hs.d2h_bytes, "ms_per_step": ms, "steps": args.e2e_steps,
           "loss": float(loss), "note": hs.note,
           "h2d_gbs_per_rank_in_step": hs.h2d_bytes / (ms * 1e-3) / 1e9, "d2h_gbs_per_rank_in_step": hs.d2h_bytes / (ms * 1e-3) / 1e9}
    # what the host path of this box gives every rank when all ranks copy at once (the bound of the leg above)
    try:
        n = 1 << 30
        hbuf = torch.empty(n, dtype=torch.uint8, pin_memory=True)
        hbuf2 = torch.empty(n, dtype=torch.uint8, pin_memory=True)
        dbuf = torch.empty(n, dtype=torch.uint8, device=device)
        dbuf2 = torch.empty(n, dtype=torch.uint8, device=device)
        s2 = torch.cuda.Stream(device)
        probe = {}
        for label in ("h2d", "d2h", "both"):
            ctx.sync_all()
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            for _ in range(3):
                if label in ("h2d", "both"):
                    dbuf.copy_(hbuf, non_blocking=True)
                if label in ("d2h", "both"):
                    with torch.cuda.stream(s2):
                        hbuf2.copy_(dbuf2, non_blocking=True)
            torch.cuda.current_stream(device).wait_stream(s2)
            a1.record()
            torch.cuda.synchronize()
            (pms,) = ctx.max_over_ranks([a0.elapsed_time(a1)])
            probe[label + "_gbs_per_rank"] = 3 * n / (pms * 1e-3) / 1e9
        probe["note"] = "1 GiB pinned copies, all ranks at once, slowest rank; 'both' = each direction while the other runs"
        rec["pcie_probe"] = probe
        h2d, d2h = probe["both_gbs_per_rank"], probe["both_gbs_per_rank"]
        rec["pcie_bound_ms"] = max(hs.h2d_bytes / (h2d * 1e9), hs.d2h_bytes / (d2h * 1e9)) * 1e3
    except Exception as exc:   # the probe is informational
        rec["pcie_probe"] = {"error": repr(exc)}
    hs.close()
    return rec


# ----------------------------------------------------------------------------- main arm
def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="C4", choices=list(WORKLOADS))
    ap.add_argument("--variant", default="default", choices=["default", "ldg", "tma"])
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-other-workloads", action="store_true")
    ap.add_argument("--no-c5", action="store_true")
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (rank 0; see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.gpus > 1 and "WORLD_SIZE" not in os.environ:
        # plain `python bench.py --gpus N`: relaunch as one process per GPU (what the driver does itself)
        os.dup2(_REAL_STDOUT.fileno(), 1)
        os.execvp(sys.executable, [sys.executable, "-m", "torch.distributed.run", "--nnodes=1",
                                   f"--nproc-per-node={args.gpus}", "--master-addr", "127.0.0.1", "--master-port",
                                   str(29000 + os.getpid() % 2000), os.path.abspath(__file__), *sys.argv[1:]])
    if args.impl == "reference":
        return run_reference_arm(args)
    if args.warmup < 3:
        args.warmup = 3
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the distillation path has no CPU fallback")
    ctx = Ctx(args)
    world, rank, device, dist = ctx.world, ctx.rank, ctx.device, ctx.dist

    from mafed_b200 import build, cabi, node
    if rank == 0:
        build.build()
        build.build_torch_ext()
    if world > 1:
        dist.barrier()
    cabi.load()
    node.load()
    variant = {"default": 0, "ldg": 1, "tma": 2}[args.variant]
    with cabi.tuning(variant=variant) if variant else _Null():
        line = run_main(ctx)
    if rank == 0:
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_main(ctx):
    from mafed_b200.distill_op import distill_backward, distill_forward, distill_fused
    args, world, rank, device, dist = ctx.args, ctx.world, ctx.rank, ctx.device, ctx.dist
    peak, peak_src = ctx.peak, ctx.peak_src
    parity = sharded_parity(ctx) if world > 1 else None     # before anything is timed; fails the run if wrong

    wl = args.workload
    desc, n_tuple, n_sel, B, txt, D, dt = WORKLOADS[wl]
    T = N_VIS + txt
    esize = torch.finfo(torch_dtype(dt)).bits // 8
    st, te, am = make_device_inputs(wl, rank, device)
    masks = [am, am.clone()]
    fd = make_method(n_sel)
    fd.populate_batch_masks = True
    fd.past_model = lambda **kw: Out(tuple(te))
    leaves = [s.detach().requires_grad_(True) for s in st]
    units_per_step = B * T * n_sel * world
    loop = ApiLoop(ctx, fd, leaves, masks)

    # ---- (1) kernel-level steps with per-stage events (for the roofline of each kernel)
    layers = list(range(n_sel))
    coeffs, modality_kind, lang_weights = fd._tables(layers)
    plan = fd._plan(layers, coeffs, fd.distillation_coeff, modality_kind, lang_weights)
    grads = [torch.empty_like(s) for s in st]
    gout = torch.ones((), dtype=torch.float32, device=device)
    fixed = plan.assumed_grad_out * plan.grad_multiplier
    tickets = [None, None]
    counter = [0]

    def two_pass_step(ev=None):
        if ev:
            ev[0].record()
        out, scale, ln = distill_forward(st, te, am, plan, group=None)      # fwd kernel (losses in its last CTA)
        if ev:
            ev[1].record()
        distill_backward(ln, grads, scale, gout, grad_out_scale=plan.grad_multiplier)   # bwd kernel
        if ev:
            ev[2].record()
        return out

    def one_pass_step(ev=None):
        i = counter[0]
        counter[0] += 1
        if world > 1:
            tickets[(i + 1) % 2] = fd.prefetch_counts({"attention_mask": masks[(i + 1) % 2]})
        if ev:
            ev[0].record()
        out, scale, ln = distill_fused(st, te, grads, masks[i % 2], plan, group=None, ticket=tickets[i % 2])  # the whole step
        if ev:
            ev[1].record()
        distill_backward(ln, grads, scale, gout, skip_if_equals=fixed, grad_out_scale=plan.grad_multiplier)   # the gate
        if ev:
            ev[2].record()
        return out

    peer = None
    if world > 1:
        from mafed_b200.comm import get_peer_comm
        peer = get_peer_comm(None)
        tickets[0] = fd.prefetch_counts({"attention_mask": masks[0]})

    step_stats = {}

    def stage_loop(step_fn):
        for _ in range(args.warmup):
            step_fn()
        evs = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(args.steps)]
        ctx.sync_all()
        for i in range(args.steps):
            step_fn(evs[i])
        ctx.sync_all()
        a = statistics.mean(e[0].elapsed_time(e[1]) for e in evs)
        b = statistics.mean(e[1].elapsed_time(e[2]) for e in evs)
        per_step = [e[0].elapsed_time(e[2]) for e in evs]
        step_stats[step_fn.__name__] = {"median_ms": statistics.median(per_step), "best_ms": min(per_step)}
        return a, b, evs[0][0].elapsed_time(evs[-1][2])

    fwd_ms, bwd_ms, two_raw_ms = stage_loop(two_pass_step)
    fused_ms, gate_ms, one_raw_ms = stage_loop(one_pass_step)

    # what the backward's check of the upstream gradient costs a step: back-to-back kernel-level steps (no events
    # inside the loop) with no check at all, with the 1-CTA gate, and with round 1's form (the whole persistent
    # backward grid launched to read one float and return)
    def plain_loop(mode):
        from mafed_b200 import cabi
        def one(i):
            out, scale, ln = distill_fused(st, te, grads, masks[i % 2], plan, group=False)
            if mode:
                distill_backward(ln, grads, scale, gout, skip_if_equals=fixed, grad_out_scale=plan.grad_multiplier)
        with cabi.tuning(TUNE_NO_GATE=1) if mode == "full_grid" else _Null():
            for i in range(args.warmup):
                one(i)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            one(1)                              # (the region opens behind one untimed step, like ApiLoop.timed)
            e0.record()
            for i in range(args.steps):
                one(i)
            e1.record()
            torch.cuda.synchronize()
        return e0.elapsed_time(e1) / args.steps
    # (interleaved rounds, differences taken inside a round: under a power cap the step time drifts by a few percent
    #  over a second, which is more than what is being measured here)
    ab_rounds = []
    for _ in range(3):
        ab_rounds.append([plain_loop(None), plain_loop("gate"), plain_loop("full_grid"),
                          loop.timed(args.steps, args.warmup)[0] / args.steps])
    base_ms = statistics.median(r[0] for r in ab_rounds)
    gate_loop_ms = statistics.median(r[1] for r in ab_rounds)
    full_loop_ms = statistics.median(r[2] for r in ab_rounds)
    gate_us = statistics.median(r[1] - r[0] for r in ab_rounds) * 1e3
    full_grid_us = statistics.median(r[2] - r[0] for r in ab_rounds) * 1e3
    api_minus_kernel_us = statistics.median(r[3] - r[1] for r in ab_rounds) * 1e3

    # ---- (2) the public API: the headline `value`
    fd.single_pass = False
    two_api_ms, _, _ = loop.timed(args.steps, args.warmup)
    fd.single_pass = True

    def uncoupled_loop():
        # the same API step with the exchange switched off (per-rank loss), all ranks at once: what every GPU does on
        # its own.  The coupled step cannot be faster than the slowest of these.
        fd.process_group = False
        own_ms, _, _ = loop.timed(args.steps, args.warmup)
        fd.process_group = None
        own = torch.tensor([own_ms / args.steps], dtype=torch.float64, device=device)
        every = [torch.zeros_like(own) for _ in range(world)]
        dist.all_gather(every, own)
        return [float(x) for x in every]

    # (the uncoupled loop runs before AND after the coupled one: step times drift by ~1 % as the GPUs warm up)
    uncoupled_before = uncoupled_loop() if world > 1 else None
    # SM cycles the in-kernel exchanges take on rank 0: two stream-ordered snapshots of the communicator's counters
    # (mafed_comm_trace_async), taken where the timed region opens and closes -- exactly the K timed steps
    trace_buf = torch.zeros((2, 4), dtype=torch.int64).pin_memory() if peer is not None else None
    snapshot = (lambda k: peer.trace_into(trace_buf[k])) if peer is not None else None
    sampler = ClockSampler(ctx.local_rank)
    api_ms, host_us, loss = loop.timed(args.steps, args.warmup, sampler, snapshot)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, loss, fd, leaves, loop.batch)
    trace0, trace1 = (trace_buf[0].tolist(), trace_buf[1].tolist()) if peer is not None else (None, None)
    cold_ms = loop.cold_ms_per_step
    start_skew = None
    if world > 1:
        # how far apart the ranks left the barrier (CLOCK_MONOTONIC is system-wide) and how long each took to enqueue
        # the step behind which the timed region opens (what `timed_region.cold_ms_per_step` still pays, once)
        mine = torch.tensor([loop.t0_monotonic, loop.first_step_enqueued_us], dtype=torch.float64, device=device)
        every = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(every, mine)
        t0s = [float(x[0]) for x in every]
        start_skew = {"barrier_exit_spread_us": (max(t0s) - min(t0s)) * 1e6,
                      "first_step_enqueued_us_per_rank": [float(x[1]) for x in every]}
    uncoupled = None
    if world > 1:
        uncoupled_after = uncoupled_loop()
        uncoupled = [0.5 * (a + b) for a, b in zip(uncoupled_before, uncoupled_after)]
    # the same two API calls captured once into a CUDA graph and replayed (fd.capture): the host side of a step that
    # is part of a graphed training step
    gstep = make_method(n_sel).capture(st, te, masks[0])
    for _ in range(args.warmup):
        gstep.replay()
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ctx.sync_all()
    gstep.replay()                              # (the region opens behind one untimed step, like ApiLoop.timed)
    t_host = time.perf_counter()
    g0.record()
    for _ in range(args.steps):
        gstep.replay()
    g1.record()
    graph_host_us = (time.perf_counter() - t_host) / args.steps * 1e6
    ctx.sync_all()
    graph_ms = g0.elapsed_time(g1)
    graph_loss = float(gstep.loss)
    del gstep
    api_ms, two_api_ms, one_raw_ms, two_raw_ms, fwd_ms, bwd_ms, fused_ms, gate_ms, graph_ms, cold_ms = ctx.max_over_ranks(
        [api_ms, two_api_ms, one_raw_ms, two_raw_ms, fwd_ms, bwd_ms, fused_ms, gate_ms, graph_ms, cold_ms])
    ms_per_step = api_ms / args.steps
    value = units_per_step / (ms_per_step * 1e-3)

    row_bytes = D * esize
    per_gpu_units = B * T * n_sel
    gbs = lambda nbytes, ms: nbytes / (ms * 1e-3) / 1e9
    fused_bytes = 3 * row_bytes * per_gpu_units
    bwd_bytes = 3 * row_bytes * per_gpu_units
    fwd_bytes = 2 * row_bytes * per_gpu_units
    two_ms = two_api_ms / args.steps
    launches_per_step = 2 if world == 1 else (3 if peer is not None else 8)

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": dt,
        "data": "synthetic", "config": workload_config(wl, world),
        "arithmetic": f"{dt} hidden states widened exactly to fp32; fp32 accumulation, fp64 final reduction; "
                      f"gradients rounded once to {dt}",
        "mode": "one-pass (loss sums + gradients from a single read of student and teacher; 3*D*e bytes per "
                "token*layer; upstream gradient checked on the device by a 1-CTA gate in backward)",
        "api": "FeatureDistillation.distill(output, batch) + loss.backward(): one call into the compiled autograd node "
               "(csrc/torch_node.cpp) per direction",
        "roofline": {"bound": "hbm", "kernel": "k_bwd_tma<kFused> (whole step: masks, scale table, sums, gradients, losses): "
                                                "2 reads + 1 write",
                     "achieved": gbs(fused_bytes, fused_ms), "peak": peak, "unit": "GB/s",
                     "frac": gbs(fused_bytes, fused_ms) / peak, "traffic": measured_traffic(wl), "peak_source": peak_src,
                     "bytes_per_launch": fused_bytes, "bytes_per_unit": 3 * row_bytes, "ms_per_launch": fused_ms,
                     "gate_launch_ms": max(0.0, gate_us * 1e-3), "fixup_launch_ms": max(0.0, gate_us * 1e-3),
                     "gate": {"what": "per-step cost of checking the upstream gradient in backward, from back-to-back "
                                      "kernel-level steps on this rank: fused kernel alone / + 1-CTA gate (the product) "
                                      "/ + the full persistent grid that returns at once (round 1); three interleaved "
                                      "rounds, median of the in-round differences",
                              "fused_only_ms_per_step": base_ms, "with_gate_ms_per_step": gate_loop_ms,
                              "with_full_grid_fixup_ms_per_step": full_loop_ms,
                              "gate_us": gate_us, "full_grid_us": full_grid_us,
                              "rounds_ms": [r[:3] for r in ab_rounds],
                              "gate_event_pair_ms": gate_ms}},
        "roofline_step": {"achieved": gbs(fused_bytes, ms_per_step), "peak": peak, "unit": "GB/s",
                          "frac": gbs(fused_bytes, ms_per_step) / peak,
                          "frac_of_nominal_8000": gbs(fused_bytes, ms_per_step) / 8000.0, "bytes_per_unit": 3 * row_bytes},
        "kernel_value": units_per_step / (one_raw_ms / args.steps * 1e-3),
        "timed_region": {"what": "barrier + synchronize, one more untimed step, event, the K timed steps, event, barrier + "
                                 "synchronize: the region opens on the device behind that step, with the GPU busy and the "
                                 "host a step ahead as in every step of a training run; `cold_ms_per_step` is the same loop "
                                 "timed from the barrier over K + 1 steps, the idle GPU's wait for the first launch included",
                         "cold_ms_per_step": cold_ms, "cold_value": units_per_step / (cold_ms * 1e-3)},
        "host_us_per_step": host_us,
        "graphed": {"what": "fd.capture(...): distill() + backward() captured once into a CUDA graph, replayed per step",
                    "ms_per_step": graph_ms / args.steps, "value": units_per_step / (graph_ms / args.steps * 1e-3),
                    "host_us_per_step": graph_host_us, "loss": graph_loss},
        "kernel_level_step_ms": {"one_pass": step_stats.get("one_pass_step"), "two_pass": step_stats.get("two_pass_step")},
        "two_pass": {
            "note": "north_star's two-kernel form (fused forward, then fused backward): 5*D*e bytes per token*layer",
            "value": units_per_step / (two_ms * 1e-3), "ms_per_step": two_ms,
            "kernel_value": units_per_step / (two_raw_ms / args.steps * 1e-3),
            "roofline_fwd": {"kernel": "k_fwd_tma (losses + scale table in its last CTA): 2 reads", "achieved": gbs(fwd_bytes, fwd_ms), "unit": "GB/s",
                             "frac": gbs(fwd_bytes, fwd_ms) / peak, "bytes_per_launch": fwd_bytes, "ms_per_launch": fwd_ms},
            "roofline_bwd": {"kernel": "k_bwd_* <kBackward>: 2 reads + 1 write", "achieved": gbs(bwd_bytes, bwd_ms),
                             "unit": "GB/s", "frac": gbs(bwd_bytes, bwd_ms) / peak, "bytes_per_launch": bwd_bytes,
                             "ms_per_launch": bwd_ms},
            "roofline_step": {"achieved": gbs(fwd_bytes + bwd_bytes, two_ms), "unit": "GB/s",
                              "frac": gbs(fwd_bytes + bwd_bytes, two_ms) / peak,
                              "frac_of_nominal_8000": gbs(fwd_bytes + bwd_bytes, two_ms) / 8000.0,
                              "bytes_per_unit": 5 * row_bytes},
        },
        # per step: the fused kernel (modality masks, scale table, loss sums + gradients, and the loss algebra in its
        # last CTA) and the 1-CTA backward gate; batch-sharded over peer memory: those two plus the 1-CTA count
        # prefetch of the next batch; NCCL sequence: masks, counts, scale, fused, reduce, finalize, gate + 2 allreduces
        "gpu_launches": args.steps * launches_per_step,
        "exchange": "none" if world == 1 else (
            "nvlink peer-memory mailboxes: token counts sent ahead of the step by a 1-CTA launch when the batch is drawn "
            "(the fused kernel reads them from its own mailbox), sums exchanged by the fused kernel's last CTA"
            if peer is not None else "nccl allreduce"),
        "loss": float(loss.detach()),
    }
    if parity is not None:
        line["sharded_parity"] = parity
    if trace0 is not None:
        # SM cycles the in-kernel exchanges took on rank 0 (mafed_comm_trace), per step, in us at the sampled SM clock
        mhz = float(sampler.summary().get("sm_mhz") or 1900.0)
        calls = max(1, trace1[3] - trace0[3])
        line["exchange_trace_us"] = {
            "counts_exchange_in_fused_kernel": (trace1[0] - trace0[0]) / calls / mhz,
            "sums_publish_in_tail": (trace1[1] - trace0[1]) / calls / mhz,
            "sums_wait_for_peers_in_tail": (trace1[2] - trace0[2]) / calls / mhz,
            "steps_traced": calls, "includes_warmup": False}
    if uncoupled is not None:
        line["uncoupled_ms_per_rank"] = uncoupled
        line["uncoupled_ms_per_rank_before_after"] = [uncoupled_before, uncoupled_after]
        line["coupling_cost_us"] = (ms_per_step - max(uncoupled)) * 1e3
        line["uncoupled_note"] = ("API step with the exchange off, all ranks running at once; the coupled step waits for "
                                  "the slowest GPU every step: ms_per_step vs max(uncoupled) is the cost of the exchange "
                                  "itself, max(uncoupled) vs the 1-GPU run is GPU-to-GPU variation")
    line["clocks"] = sampler.summary()
    if start_skew is not None:
        line["start_skew"] = start_skew
    # the API loop against the kernel-level loop (fused + gate), same interleaved rounds
    line["api_minus_kernel_loop_us"] = api_minus_kernel_us if world == 1 else None

    if not args.no_c5:
        try:
            line["c5"] = c5_sweep(ctx)
        except Exception as exc:
            line["c5"] = {"error": repr(exc)}
    if world == 1 and not args.no_other_workloads:
        try:
            line["other_workloads"] = other_workloads(ctx, wl)
        except Exception as exc:
            line["other_workloads"] = {"error": repr(exc)}
    # ---- (3) end to end with HOST buffers (pinned): H2D inputs, step, D2H gradients + loss
    if not args.no_e2e:
        try:
            line["e2e"] = run_e2e(ctx, fd, st, te, am, units_per_step)
        except Exception as exc:  # keep the headline line even if the host path cannot allocate
            line["e2e"] = {"error": repr(exc)}
    if world == 1 and not args.no_cpu_baseline:
        try:
            line["eager_torch_gpu"] = eager_gpu_baseline(wl, st, te, am)
        except Exception as exc:
            line["eager_torch_gpu"] = {"error": repr(exc)}
    if rank == 0 and not args.no_cpu_baseline and world == 1:
        try:
            base = cpu_reference_steps(wl, steps=3, warmup=1, budget_s=60.0)
            line["cpu_baseline"] = {k: base[k] for k in ("value", "unit", "cores", "kind", "sample")}
        except Exception as exc:
            line["cpu_baseline"] = {"error": repr(exc)}
    return line


if __name__ == "__main__":
    main()
