"""libmafed_cached_step.so without a GPU: build, exports, SASS, header, argument errors, which steps it takes, no
programmatic dependent launches, and which path ``FeatureDistillation.distill`` picks for a replay step."""
import ctypes
import os
import re
import subprocess
import types

import pytest
import torch

from mafed_b200 import build, cabi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "mafed_cached_step.h")
SOURCE = os.path.join(ROOT, "mafed_b200", "csrc", "cached_step.cu")

EXPECTED_EXPORTS = sorted(["mafed_cached_step_abi_version", "mafed_cached_step_error_string",
                           "mafed_cached_step_supported", "mafed_cached_step", "mafed_cached_step_bwd"])

vp, i32, i64 = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64


def _lib():
    lib = ctypes.CDLL(build.build_cached_step())
    lib.mafed_cached_step_error_string.restype = ctypes.c_char_p
    lib.mafed_cached_step_supported.argtypes = [vp, vp, vp, i64, i32]
    lib.mafed_cached_step.argtypes = [vp, vp, vp, i64, i32, vp, vp, vp, vp, ctypes.c_float, vp, vp, vp, vp, vp, vp, vp]
    lib.mafed_cached_step_bwd.argtypes = [vp, vp, vp, i64, i32, vp, vp, vp, vp, vp, ctypes.c_float, vp, vp, vp]
    return lib


def test_exports_are_exactly_the_header_and_the_sass_uses_bulk_copies():
    path = build.build_cached_step()
    declared = sorted(set(re.findall(r"\b(mafed_cached_step\w*)\s*\(", open(HEADER).read())))
    assert declared == EXPECTED_EXPORTS
    out = subprocess.run(["nm", "-D", "--defined-only", path], capture_output=True, text=True).stdout
    assert sorted(line.split()[-1] for line in out.splitlines() if " T " in line and "mafed_" in line) == EXPECTED_EXPORTS
    sass = subprocess.run(["cuobjdump", "-sass", path], capture_output=True, text=True).stdout
    assert "sm_100a" in sass or "sm_100" in sass
    assert "UBLKCP" in sass and "k_bwd_tma_cached" in sass
    assert _lib().mafed_cached_step_abi_version() == 1


def test_header_is_plain_c99(tmp_path):
    src = tmp_path / "consumer.c"
    src.write_text('#include "mafed_cached_step.h"\nint main(void) { return MAFED_CACHED_MAX_SAMPLES == 2048 ? 0 : 1; }\n')
    res = subprocess.run(["gcc", "-std=c99", "-pedantic", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"),
                          "-c", str(src), "-o", str(tmp_path / "consumer.o")], capture_output=True, text=True)
    assert res.returncode == 0, res.stderr


def test_no_programmatic_dependent_launch_in_the_source():
    """Every launch of the library is a plain stream launch (see the header): none can become resident ahead of a
    backward that a gate of libmafed_distill.so started from the device."""
    text = open(SOURCE).read()
    code = re.sub(r"//[^\n]*", "", text)
    for word in ("Programmatic", "programmatic", "launch_pdl", "HostLaunch", "cudaLaunchKernelEx", "cudaLaunchAttribute"):
        assert word not in code, word


def _ptrs(*vals):
    return (ctypes.c_void_p * len(vals))(*vals)


A, U = 0x7f0000001000, 0x7f0000001008      # 16-byte aligned / 8-byte aligned fake device addresses


def _shape(L=2, B=3, T=12, n_vis=5, D=64, dtype=cabi.F32, loss=cabi.LOSS_MSE, cls=False, t_dtype=None):
    return cabi.make_shape(L, B, T, n_vis, D, dtype, loss, cls, t_dtype)


def test_supported_truth_table():
    lib = _lib()

    def ok(shape, s=A, c=A, M=5, T_c=14):
        L = shape.n_layers
        return lib.mafed_cached_step_supported(ctypes.byref(shape), _ptrs(*[s] * L), _ptrs(*[c] * L), M, T_c)

    for dt in (cabi.F32, cabi.BF16, cabi.F16):
        for loss in (cabi.LOSS_MSE, cabi.LOSS_COSINE):
            assert ok(_shape(dtype=dt, loss=loss)) == 1
    for t in (cabi.BF16, cabi.F16):
        assert ok(_shape(t_dtype=t)) == 1
        assert ok(_shape(D=68, t_dtype=t)) == 0            # a half-precision teacher row is not whole 16-byte chunks
        assert ok(_shape(D=72, t_dtype=t)) == 1
    assert ok(_shape(dtype=cabi.BF16, t_dtype=cabi.F32)) == 0   # no kernel for a student narrower than its teacher
    assert ok(_shape(dtype=cabi.BF16, t_dtype=cabi.F16)) == 0
    assert ok(_shape(cls=True, loss=cabi.LOSS_COSINE)) == 0
    assert ok(_shape(D=63)) == 0 and ok(_shape(dtype=cabi.BF16, D=60)) == 0      # rows of partial chunks
    assert ok(_shape(D=8192)) == 1 and ok(_shape(D=8196)) == 0                    # rows up to 32 KB
    assert ok(_shape(dtype=cabi.BF16, D=16384)) == 1 and ok(_shape(dtype=cabi.BF16, D=16392)) == 0
    assert ok(_shape(), s=U) == 0 and ok(_shape(), c=U) == 0
    assert ok(_shape(), T_c=11) == 0 and ok(_shape(), M=0) == 0
    assert ok(_shape(B=2048)) == 1 and ok(_shape(B=2049)) == 0
    with cabi.tuning(variant=cabi.VARIANT_LDG):
        assert ok(_shape()) == 0
    with cabi.tuning(TUNE_NO_TAIL=1):
        assert ok(_shape()) == 0
    assert lib.mafed_cached_step_supported(None, None, None, 5, 14) == 0


def test_argument_errors_without_a_gpu():
    lib = _lib()
    w = cabi.make_weights(cabi.MODW_EQUAL, 1.0, [1.0, 1.0])
    ws = out = scale = A

    def step(shape, idx, M=5, T_c=14, s=A, c=A, g=A, mask=A):
        L = shape.n_layers
        ix = (ctypes.c_int64 * len(idx))(*idx) if idx is not None else None
        sp = _ptrs(*[s] * L) if s is not None else None
        cp = _ptrs(*[c] * L) if c is not None else None
        gp = _ptrs(*[g] * L)
        a = lib.mafed_cached_step(ctypes.byref(shape), sp, cp, M, T_c, ix, gp, mask, ctypes.byref(w), 1.0, ws, out,
                                  scale, None, None, None, None)
        b = lib.mafed_cached_step_bwd(ctypes.byref(shape), sp, cp, M, T_c, ix, gp, mask, scale, None, 1.0, None, None,
                                      None)
        return a, b

    E = -1     # MAFED_E_ARG: every call below is refused before anything touches a device
    assert step(_shape(), [0, 1, 2], s=None) == (E, E)              # null tables
    assert step(_shape(), [0, 1, 2], c=None) == (E, E)
    assert step(_shape(), None) == (E, E)
    assert step(_shape(), [0, -1, 2]) == (E, E)                     # index < 0
    assert step(_shape(), [0, 5, 2]) == (E, E)                      # index >= M
    assert step(_shape(T=15), [0, 1, 2]) == (E, E)                  # T > T_c
    assert step(_shape(T=4, n_vis=5), [0, 1, 2]) == (E, E)          # T < n_vis
    assert step(_shape(B=2049), list(range(2049)), M=4096) == (E, E)    # more samples than one launch carries
    assert step(_shape(cls=True, loss=cabi.LOSS_COSINE), [0, 1, 2]) == (E, E)
    assert b"memory index" in lib.mafed_cached_step_error_string(-1)


# ---------------------------------------------------------------- which path FeatureDistillation.distill takes
class _Out:
    def __init__(self, hs):
        self.hidden_states = hs


class _Opts:
    tasks = ["a", "b", "c"]; batch_size = 4; seed = 1; pin_mem = False; accumulate_grad_batches = 1


def _fd(monkeypatch, cache_kind="replicated", **kw):
    from mafed_b200 import teacher_cache as TC
    from mafed_b200.methods import CLMethod
    from mafed_b200.methods import distillation as D
    loss = kw.pop("loss", "mse")
    fd = CLMethod["featdistill"](memory_size=8, opts=_Opts(), model_type="vlpythia",
                                 distillation_modality_weighing_strategy="balanced",
                                 distillation_layer_weighing_strategy="discounted", distillation_layer=None,
                                 distillation_loss=loss, gamma=0.5, num_hidden_layers=3, teacher_cache=True, **kw)
    fd.num_vision_tokens = 4
    layers = fd.loss_weights.get_distillation_layers()
    states = [torch.zeros(6, 10, 16) for _ in layers]
    if cache_kind == "replicated":
        cache = TC.TeacherCache(layers, states, 10, 4)
    else:
        cache = object.__new__(TC.ShardedTeacherCache)
        cache.layers, cache.T_c, cache.n_vis = list(layers), 10, 4
    fd._teacher_cache = cache
    calls = []
    L = len(layers)

    def fake_cached(students, cache_states, idx, T_c, attn, plan, mask_out=None, seen=None, return_masks=False):
        calls.append(("cached", list(idx), T_c))
        return torch.tensor(1.0), torch.zeros(3 * L), None

    def fake_launch(plan, batch, students, teachers, teachers_detached=False):
        calls.append(("ordinary", len(teachers)))
        return torch.tensor(2.0), torch.zeros(3 * L)

    def fake_gather(self, idx, T, layers):
        calls.append(("gather", list(idx), T))
        return [torch.zeros(len(idx), T, 16) for _ in layers]

    monkeypatch.setattr(D, "cached_distill_loss", fake_cached)
    monkeypatch.setattr(D, "seen_slot", lambda: torch.zeros(1))
    monkeypatch.setattr(D, "modality_masks", lambda attn, n_vis: (None, None))
    monkeypatch.setattr(fd, "_launch", fake_launch)
    monkeypatch.setattr(TC.TeacherCache, "gather", fake_gather)
    monkeypatch.setattr(TC.ShardedTeacherCache, "gather", fake_gather)
    return fd, calls


def _distill(fd, idx=(1, 5)):
    fd._memory_index = list(idx)
    hs = tuple(torch.zeros(len(idx), 9, 16, requires_grad=True) for _ in range(4))
    batch = {"attention_mask": torch.ones(len(idx), 5, dtype=torch.int64), "labels": torch.zeros(1)}
    total = fd.distill(_Out(hs), batch)
    assert "labels" not in batch and fd._memory_index is None
    return float(total)


def test_replicated_eager_one_pass_step_reads_the_cache(monkeypatch):
    fd, calls = _fd(monkeypatch)
    assert _distill(fd) == 1.0
    assert calls == [("cached", [1, 5], 10)]


def test_refused_launch_falls_back_to_the_gather(monkeypatch):
    from mafed_b200.methods import distillation as D
    fd, calls = _fd(monkeypatch)
    monkeypatch.setattr(D, "cached_distill_loss", lambda *a, **k: calls.append(("cached?",)))
    assert _distill(fd) == 2.0
    assert calls == [("cached?",), ("gather", [1, 5], 9), ("ordinary", 3)]


@pytest.mark.parametrize("case", ["sharded", "two-pass", "cls", "process-group"])
def test_gather_and_step_elsewhere(case, monkeypatch):
    from mafed_b200.methods import distillation as D
    kw = {"two-pass": dict(single_pass=False), "cls": dict(cls_distillation=True, loss="cosine")}.get(case, {})
    fd, calls = _fd(monkeypatch, "sharded" if case == "sharded" else "replicated", **kw)
    if case == "process-group":
        monkeypatch.setattr(D, "resolve_group", lambda group: (True, None))
        monkeypatch.setattr(fd, "_step_plan", lambda layers: types.SimpleNamespace(
            layers=list(layers), single_pass=True, cls=False))
    assert _distill(fd) == 2.0
    assert calls == [("gather", [1, 5], 9), ("ordinary", 3)]


def test_out_of_range_index_is_the_gathers_error(monkeypatch):
    from mafed_b200.methods import distillation as D
    fd, calls = _fd(monkeypatch)
    monkeypatch.setattr(D, "cached_distill_loss", lambda *a, **k: pytest.fail("launched"))
    with pytest.raises(cabi.MafedDistillError, match="out of range"):
        _distill(fd, idx=(1, 6))
    fd._memory_index = [0]
    with pytest.raises(cabi.MafedDistillError, match="does not fit"):
        fd._teacher_cache.step_inputs([0], 11, fd._teacher_cache.layers)
