"""A student / teacher dtype pair in mafed_shape_t::dtype (MAFED_DTYPE_PAIR): which pairs the library takes, which it
refuses, and that the refusal comes before any pointer check or device query (not gpu)."""
import ctypes
import os
import re
import subprocess

import pytest
import torch

from mafed_b200 import build, cabi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SUPPORTED = [(cabi.F32, cabi.BF16), (cabi.F32, cabi.F16)]
REFUSED = [(cabi.BF16, cabi.F32), (cabi.F16, cabi.F32), (cabi.BF16, cabi.F16), (cabi.F16, cabi.BF16)]


def _shape(student, teacher, loss=cabi.LOSS_MSE):
    return cabi.make_shape(1, 1, 4, 2, 64, student, loss, teacher_dtype=teacher)


def test_make_shape_encodes_the_pair():
    assert cabi.make_shape(1, 1, 4, 2, 8, cabi.F32, cabi.LOSS_MSE).dtype == cabi.F32
    assert cabi.make_shape(1, 1, 4, 2, 8, cabi.BF16, cabi.LOSS_MSE, teacher_dtype=cabi.BF16).dtype == cabi.BF16
    assert _shape(cabi.F32, cabi.BF16).dtype == cabi.F32 | (cabi.BF16 + 1) << 8
    assert _shape(cabi.F32, cabi.F16).dtype == cabi.dtype_pair(cabi.F32, cabi.F16) == 0x300


def test_header_macro_and_cabi_agree(tmp_path):
    src = tmp_path / "pair.c"
    src.write_text('#include <stdio.h>\n#include "mafed_distill.h"\nint main(void) {\n'
                   '  int s, t;\n'
                   '  for (s = 0; s < 3; ++s) for (t = 0; t < 3; ++t) printf("%d %d %d\\n", s, t, MAFED_DTYPE_PAIR(s, t));\n'
                   '  return 0;\n}\n')
    exe = str(tmp_path / "pair")
    res = subprocess.run(["gcc", "-std=c99", "-pedantic", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"),
                          str(src), "-o", exe], capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    rows = [tuple(int(v) for v in ln.split()) for ln in subprocess.run([exe], capture_output=True, text=True,
                                                                        check=True).stdout.splitlines()]
    assert len(rows) == 9
    for s, t, code in rows:
        assert code == cabi.dtype_pair(s, t)


def _step(lib, sh, s_ptrs=None, t_ptrs=None):
    w = cabi.make_weights(cabi.MODW_EQUAL, 1.0, [1.0])
    out = (ctypes.c_float * 4)()
    return lib.mafed_distill_step(ctypes.byref(sh), s_ptrs, t_ptrs, None, None, ctypes.byref(w), ctypes.c_float(1.0),
                                  None, out, None, None, None, None, None, None, None)


def _bwd(lib, sh, gate=False):
    scale = (ctypes.c_float * 2)()
    one = ctypes.c_float(1.0)
    return lib.mafed_distill_bwd(ctypes.byref(sh), None, None, cabi.ptr_array([16]), None, scale, None, one,
                                 ctypes.byref(one) if gate else None, None, None)


@pytest.mark.parametrize("student,teacher", REFUSED)
@pytest.mark.parametrize("loss", [cabi.LOSS_MSE, cabi.LOSS_COSINE])
def test_unsupported_pairs_are_dtype_errors(student, teacher, loss):
    lib = cabi.load()
    sh = _shape(student, teacher, loss)
    assert lib.mafed_distill_fwd(ctypes.byref(sh), None, None, None, None, None) == -2
    assert _step(lib, sh) == -2
    assert _bwd(lib, sh) == -2
    assert _bwd(lib, sh, gate=True) == -2


def test_malformed_codes_are_dtype_errors():
    lib = cabi.load()
    for code in (cabi.dtype_pair(cabi.F32, 3), 3 << 8 | 3, 1 << 16, -1, 4 << 8):
        sh = cabi.make_shape(1, 1, 4, 2, 64, cabi.F32, cabi.LOSS_MSE)
        sh.dtype = code
        assert lib.mafed_distill_fwd(ctypes.byref(sh), None, None, None, None, None) == -2, hex(code)


@pytest.mark.parametrize("student,teacher", SUPPORTED + [(cabi.F32, cabi.F32), (cabi.BF16, cabi.BF16)])
def test_supported_pairs_pass_the_dtype_check(student, teacher):
    """NULL pointer tables are the next thing checked: -1 proves the pair got past the dtype check."""
    lib = cabi.load()
    sh = _shape(student, teacher)
    sh.dtype = cabi.dtype_pair(student, teacher)   # the explicit form, also for a same-dtype "pair"
    assert lib.mafed_distill_fwd(ctypes.byref(sh), None, None, None, None, None) == -1
    assert _step(lib, sh) == -1
    assert _bwd(lib, sh) == -1


@pytest.mark.parametrize("student,teacher", SUPPORTED)
def test_single_input_and_host_step_refuse_pairs(student, teacher):
    lib = cabi.load()
    sh = _shape(student, teacher)
    assert lib.mafed_distill_token_norm_sums(ctypes.byref(sh), None, None, None, None) == -2
    h = ctypes.c_void_p()
    assert lib.mafed_host_step_create(ctypes.byref(sh), ctypes.byref(h)) == -2
    assert not h.value
    assert lib.mafed_host_step_device_bytes(ctypes.byref(sh)) == 0
    plain = cabi.make_shape(1, 1, 4, 2, 64, student, cabi.LOSS_MSE)
    assert lib.mafed_host_step_device_bytes(ctypes.byref(plain)) > 0
    assert lib.mafed_distill_token_norm_sums(ctypes.byref(plain), None, None, None, None) == -1


def _sass_functions():
    out = subprocess.run(["cuobjdump", "-sass", cabi.LIB_PATH], capture_output=True, text=True, check=True).stdout
    return dict(re.findall(r"Function : (\S+)\n(.*?)(?=\n\s+Function : |\Z)", out, flags=re.S))


def test_pair_kernels_are_compiled_and_the_ring_uses_bulk_copies():
    build.build()
    fns = _sass_functions()
    # k_{fwd,bwd}_tma<float, ..., __nv_bfloat16 | __half>: the ring's bulk copies, the teacher's 8-byte shared loads
    tma = {n: body for n, body in fns.items() if re.search(r"k_(fwd|bwd)_tmaIf.*(13__nv_bfloat16|6__half)EEv", n)}
    # per pair: forward and backward / one-pass step x 2 losses in the main unit, the backward x 2 losses in the gate unit
    assert len(tma) == 2 * (2 + 4 + 2)
    for name, body in tma.items():
        assert "UBLKCP" in body and "LDS.64" in body and "LDS.128" in body, name
    for family in ("k_fwd_ldg", "k_bwd_ldg", "k_fwd_generic", "k_bwd_generic"):
        assert any(re.search(family + r"If.*(13__nv_bfloat16|6__half)EEv", n) for n in fns), family


def test_teacher_dtype_option():
    from gpu_util import Opts
    from mafed_b200.methods import CLMethod

    def make(**kw):
        return CLMethod["featdistill"](memory_size=8, opts=Opts(), model_type="vlpythia",
                                       distillation_layer_weighing_strategy="equal", **kw)

    for bad in (torch.float32, torch.float64, "bf16", torch.int8):
        with pytest.raises(ValueError, match="teacher_dtype"):
            make(teacher_dtype=bad)
    model = torch.nn.Sequential(torch.nn.Linear(4, 4), torch.nn.LayerNorm(4))
    fd = make()
    fd._update_model(model)
    assert all(p.dtype == torch.float32 for p in fd.past_model.parameters())
    for dt in (torch.bfloat16, torch.float16):
        fd = make(teacher_dtype=dt)
        fd._update_model(model)
        assert all(p.dtype == dt for p in fd.past_model.parameters())
        assert not fd.past_model.training
    assert all(p.dtype == torch.float32 for p in model.parameters())   # the trained model itself is left alone


@pytest.mark.parametrize("selective", [False, True], ids=["full-tuple", "selective-capture"])
def test_half_precision_snapshot_inside_a_bf16_autocast_region(selective):
    """replay() runs the teacher forward inside its bf16 autocast region.  A snapshot held in fp16 would get bf16 out
    of its linears there and fp16 out of its embedding (and the tiny VL model's concat of the two raises); the teacher
    forward runs under an autocast of the snapshot's own dtype instead, and every teacher state comes out in it --
    also the final layer norm's, which autocast computes in fp32.  (CPU autocast: the same rules as on the GPU.)"""
    from gpu_util import Opts
    from mafed_b200.methods import CLMethod
    from tiny_vl import TinyVL, make_batch
    torch.manual_seed(0)
    model = TinyVL()
    batch = make_batch()
    layers = [0, 1, 2, 3]
    for dt in (torch.float16, torch.bfloat16):
        fd = CLMethod["featdistill"](memory_size=8, opts=Opts(), model_type="vlpythia",
                                     distillation_layer_weighing_strategy="equal", num_hidden_layers=3,
                                     teacher_dtype=dt, selective_capture=selective)
        fd._update_model(model)
        with torch.autocast("cpu", dtype=torch.bfloat16):
            got = fd._past_states(dict(batch), layers)
            full = fd._get_past_hidden_states(dict(batch))
        assert [h.dtype for h in got] == [dt] * 4
        assert all(full[l].dtype == dt for l in fd.loss_weights.get_distillation_layers())
        with torch.no_grad(), torch.autocast("cpu", dtype=dt):
            want = model.to(dt)(**{k: v for k, v in batch.items() if k != "labels"}, output_hidden_states=True).hidden_states
        model.float()
        for g, l in zip(got, layers):
            assert torch.equal(g, want[l].to(dt))
