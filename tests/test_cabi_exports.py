"""The C-ABI library builds for sm_100a, loads, and exports every symbol the header declares (not gpu)."""
import ctypes
import os
import re
import subprocess

from mafed_b200 import build, cabi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    text = open(os.path.join(ROOT, "include", "mafed_distill.h")).read()
    return sorted(set(re.findall(r"\b(mafed_(?:distill|comm|host)_[a-z_]+)\s*\(", text)))


# The whole product ABI (ABI v4).  Round 1 exported 34 symbols, among them overlapping generations of the same
# stage (_reduce / _finalize / _epilogue / _prologue / _fused_comm / _scalar_stage_comm) and two process-global
# knob setters (_set_variant / _set_tuning); they are gone -- knobs travel per call in mafed_shape_t::tuning.
EXPECTED_EXPORTS = sorted([
    "mafed_distill_abi_version", "mafed_distill_error_string", "mafed_distill_ws_bytes", "mafed_distill_sums_len",
    "mafed_distill_out_len", "mafed_distill_step", "mafed_distill_fwd_step", "mafed_distill_bwd",
    "mafed_distill_prefetch_counts", "mafed_distill_fwd", "mafed_distill_fused", "mafed_distill_scalar_stage",
    "mafed_distill_modality_masks", "mafed_distill_token_norm_sums", "mafed_comm_handle_bytes", "mafed_comm_create",
    "mafed_comm_connect", "mafed_comm_status", "mafed_comm_trace", "mafed_comm_trace_async", "mafed_comm_set_timeout", "mafed_comm_destroy",
    "mafed_host_step_device_bytes", "mafed_host_step_create", "mafed_host_step_run", "mafed_host_step_destroy",
    "mafed_host_register", "mafed_host_unregister"])


def test_export_list_is_exactly_the_header():
    """Header, ctypes binding and the dynamic symbol table of the built library agree on one reduced list."""
    build.build()
    assert _declared() == EXPECTED_EXPORTS
    assert sorted(cabi.EXPORTS) == EXPECTED_EXPORTS
    out = subprocess.run(["nm", "-D", "--defined-only", cabi.LIB_PATH], capture_output=True, text=True).stdout
    exported = sorted(line.split()[-1] for line in out.splitlines() if " T mafed_" in line)
    assert exported == EXPECTED_EXPORTS
    for gone in ("mafed_distill_set_variant", "mafed_distill_set_tuning", "mafed_distill_epilogue",
                 "mafed_distill_fused_comm", "mafed_distill_scalar_stage_comm"):
        assert gone not in out


def test_no_process_global_knobs():
    """Experiment knobs are per call: a Tuning rides in the shape of the calls made inside `cabi.tuning(...)`."""
    assert cabi.active_tuning_address() == 0
    with cabi.tuning(variant=cabi.VARIANT_LDG, TUNE_NO_TAIL=1) as t:
        sh = cabi.make_shape(1, 1, 4, 2, 8, cabi.F32, cabi.LOSS_MSE)
        assert sh.tuning.contents.v[cabi.TUNE_VARIANT_ALL] == cabi.VARIANT_LDG and sh.tuning.contents.v[cabi.TUNE_NO_TAIL] == 1
        assert cabi.active_tuning_address() == ctypes.addressof(t)
        with cabi.tuning(TUNE_NO_GATE=1) as inner:
            assert inner.v[cabi.TUNE_NO_TAIL] == 1 and inner.v[cabi.TUNE_NO_GATE] == 1
    assert cabi.active_tuning_address() == 0
    assert not cabi.make_shape(1, 1, 4, 2, 8, cabi.F32, cabi.LOSS_MSE).tuning
    # only the three keys the library reads are accepted; a retired or misspelt one is an error, not a silent no-op
    import pytest
    for bad in ({"TUNE_TMA_WARPS": 8}, {"F32": 1}, {"raw": {9: 8}}):
        with pytest.raises(TypeError, match="unknown tuning key"):
            with cabi.tuning(**bad):
                pass
    assert cabi.active_tuning_address() == 0


def test_torch_extension_builds_and_binds():
    """The compiled autograd node (host C++) builds in-tree, imports on a CPU box and binds the C ABI."""
    from mafed_b200 import node
    build.build_torch_ext()
    ext = node.load()
    assert ext.is_bound()
    plan = ext.Plan(cabi.MODW_TABLE, 1.0, [0.25, 0.75], [0.5, 0.5], cabi.LOSS_MSE, False, 256, 1.0, True, 1.0)
    assert plan.n_layers == 2 and plan.single_pass
    import pytest
    import torch
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ext.distill(plan, [torch.zeros(1, 260, 8)] * 2, [torch.zeros(1, 260, 8)] * 2,
                    torch.ones(1, 4, dtype=torch.int64), None, 0, None, None, 0)


def test_library_exports_every_declared_symbol():
    build.build()
    lib = cabi.load()
    names = _declared()
    assert len(names) >= 10
    for n in names:
        assert hasattr(lib, n), n
    assert sorted(cabi.EXPORTS) == names
    assert lib.mafed_distill_abi_version() == cabi.ABI_VERSION
    assert lib.mafed_distill_sums_len(15) == 32 and lib.mafed_distill_out_len(15) == 46
    assert lib.mafed_distill_ws_bytes(15) >= 148 * 15 * 2 * 4
    assert b"invalid argument" in lib.mafed_distill_error_string(-1)


def test_argument_errors_without_a_gpu():
    lib = cabi.load()
    bad = cabi.make_shape(0, 1, 1, 0, 8, cabi.F32, cabi.LOSS_MSE)
    assert lib.mafed_distill_fwd(ctypes.byref(bad), None, None, None, None, None) == -1
    bad = cabi.make_shape(1, 1, 4, 2, 8, 7, cabi.LOSS_MSE)
    assert lib.mafed_distill_fwd(ctypes.byref(bad), None, None, None, None, None) == -2
    ok = cabi.make_shape(1, 1, 4, 2, 8, cabi.F32, cabi.LOSS_MSE)
    assert lib.mafed_distill_fwd(ctypes.byref(ok), None, None, None, None, None) == -1  # null pointer tables
    # the one-call step: weights and the output vector are mandatory, the two masks come as a pair
    w = cabi.make_weights(cabi.MODW_EQUAL, 1.0, [1.0])
    one = ctypes.c_float(1.0)
    assert lib.mafed_distill_step(ctypes.byref(ok), None, None, None, None, None, one, None, None, None, None, None,
                                  None, None, None, None) == -1
    assert lib.mafed_distill_step(ctypes.byref(ok), None, None, None, None, ctypes.byref(w), one, None, 8, None, None,
                                  8, None, None, None, None) == -1
    assert lib.mafed_distill_bwd(ctypes.byref(ok), None, None, None, None, None, None, one, None, None, None) == -1
    # a NULL shape is an argument error on the gate path too (grad table, scale table and skip_if_equals given)
    scale = (ctypes.c_float * 2)()
    assert lib.mafed_distill_bwd(None, None, None, cabi.ptr_array([8]), None, scale, None, one, ctypes.byref(one), None,
                                 None) == -1
    assert lib.mafed_distill_prefetch_counts(ctypes.byref(ok), None, None, None, None) == -1
    assert lib.mafed_distill_scalar_stage(ctypes.byref(ok), None, cabi.STAGE_LOSSES, None, None, None, None, None, None, 0,
                                          None) == -1
    assert lib.mafed_distill_fwd_step(ctypes.byref(ok), None, None, None, None, None, None, None, None, None, None) == -1
    assert lib.mafed_comm_trace(None, None) == -1
    assert lib.mafed_comm_trace_async(None, None, None) == -1


def test_sass_is_sm100_and_uses_bulk_copies():
    out = subprocess.run(["cuobjdump", "-sass", cabi.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in out or "sm_100" in out
    assert "UBLKCP" in out  # cp.async.bulk (TMA engine) in the staged kernels
    assert re.search(r"LDG\.E(\.NA)?\.128", out) and "STG.E.128" in out and "LDS.128" in out


def test_missing_library_fails_loudly(monkeypatch, tmp_path):
    """No CUDA library -> the product raises; there is no eager / CPU fallback to fall into."""
    import pytest
    monkeypatch.setattr(cabi, "_lib", None)
    monkeypatch.setattr(cabi, "LIB_PATH", str(tmp_path / "libmafed_distill.so"))
    with pytest.raises(cabi.MafedDistillError, match="no CPU / eager fallback"):
        cabi.load()


def test_header_is_plain_c_and_links_from_c(tmp_path):
    """include/mafed_distill.h compiles as C99 (-pedantic) and a C program linked against the library can call
    the ABI -- the non-Python binding route of INTEGRATION.md."""
    build.build()
    src = os.path.join(ROOT, "tests", "c", "cabi_consumer.c")
    exe = str(tmp_path / "cabi_consumer")
    lib_dir = os.path.dirname(cabi.LIB_PATH)
    cmd = ["gcc", "-std=c99", "-pedantic", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), src, "-o", exe,
           "-L", lib_dir, "-lmafed_distill", f"-Wl,-rpath,{lib_dir}"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    run = subprocess.run([exe], capture_output=True, text=True)
    assert run.returncode == 0 and run.stdout.strip() == "OK", run.stdout + run.stderr
