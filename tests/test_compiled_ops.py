"""The ``mafed::`` torch.library ops without a GPU: schemas, and the shapes and dtypes their fake implementations give
(what torch.compile traces with).  Fake CUDA tensors need no device."""
import pytest
import torch
from torch._subclasses.fake_tensor import FakeTensorMode

from mafed_b200 import cabi, node


@pytest.fixture(scope="module", autouse=True)
def _loaded():
    node.load()


def test_the_three_schemas_are_registered():
    ops = torch.ops.mafed
    step = str(ops.step.default._schema)
    assert step.startswith("mafed::step(Tensor[] students, Tensor[] teachers, Tensor? mask, float[] layer_coeffs, "
                           "float[]? lang_weights, int modality_kind, float distill_coeff, int loss_kind, bool cls, "
                           "int n_vis, float assumed_grad_out, float grad_multiplier, bool[] needs, int comm, "
                           "bool want_masks, int tuning)")
    assert step.endswith("-> (Tensor, Tensor, Tensor, Tensor)")
    fwd = str(ops.fwd_step.default._schema)
    assert "float grad_multiplier, bool[] needs, int comm, bool want_masks, int tuning" in fwd
    assert fwd.endswith("-> (Tensor, Tensor, Tensor)")
    bwd = ops.bwd.default._schema
    assert str(bwd).endswith("-> ()")
    mutated = [a.name for a in bwd.arguments if a.alias_info is not None and a.alias_info.is_write]
    assert mutated == ["grads"]
    for op in (ops.step, ops.fwd_step, ops.bwd):
        assert torch._C._dispatch_has_kernel_for_dispatch_key(op.default.name(), "CUDA")
        assert torch._C._dispatch_has_kernel_for_dispatch_key(op.default.name(), "Autograd") or op is ops.bwd


def _inputs(mode, L, B, T, D, s_dtype, t_dtype, cls, n_vis=4):
    with mode:
        st = [torch.empty(B, T, D, dtype=s_dtype, device="cuda") for _ in range(L)]
        te = [torch.empty(B, T, D, dtype=t_dtype, device="cuda") for _ in range(L)]
        mask = None if cls else torch.empty(B, T - n_vis, dtype=torch.int64, device="cuda")
    return st, te, mask


def _plan_args(L, loss_kind, cls, n_vis=4):
    return ([1.0] * L, None if cls else [0.5] * L, cabi.MODW_CLS if cls else cabi.MODW_TABLE, 1.0, loss_kind, cls,
            n_vis)


CASES = [
    (cabi.LOSS_MSE, False, torch.float32, torch.float32),
    (cabi.LOSS_COSINE, False, torch.float32, torch.float32),
    (cabi.LOSS_MSE, False, torch.bfloat16, torch.bfloat16),
    (cabi.LOSS_COSINE, False, torch.bfloat16, torch.bfloat16),
    (cabi.LOSS_MSE, False, torch.float32, torch.bfloat16),
    (cabi.LOSS_COSINE, False, torch.float32, torch.bfloat16),
    (cabi.LOSS_COSINE, True, torch.float32, torch.float32),
    (cabi.LOSS_COSINE, True, torch.bfloat16, torch.bfloat16),
]


@pytest.mark.parametrize("want_masks", [False, True])
@pytest.mark.parametrize("loss_kind,cls,s_dtype,t_dtype", CASES)
def test_step_fake_shapes_and_dtypes(loss_kind, cls, s_dtype, t_dtype, want_masks):
    L, B, T, D = 3, 2, 10, 64
    mode = FakeTensorMode()
    st, te, mask = _inputs(mode, L, B, T, D, s_dtype, t_dtype, cls)
    needs = [True, False, True]
    with mode:
        out, grads, scale, masks = torch.ops.mafed.step(st, te, mask, *_plan_args(L, loss_kind, cls), 1.0, 1.0, needs,
                                                        0, want_masks, 0)
    assert out.shape == (1 + 3 * L,) and out.dtype == torch.float32 and out.device.type == "cuda"
    assert grads.shape == (2, B, T, D) and grads.dtype == s_dtype and grads.device.type == "cuda"
    assert scale.shape == (2 * L,) and scale.dtype == torch.float32
    assert masks.dtype == torch.int64
    assert masks.shape == ((2, B, T) if want_masks and not cls else (0,))


@pytest.mark.parametrize("want_masks", [False, True])
@pytest.mark.parametrize("loss_kind,cls,s_dtype,t_dtype", CASES)
def test_fwd_step_and_bwd_fake_shapes_and_dtypes(loss_kind, cls, s_dtype, t_dtype, want_masks):
    L, B, T, D = 2, 3, 9, 32
    mode = FakeTensorMode()
    st, te, mask = _inputs(mode, L, B, T, D, s_dtype, t_dtype, cls)
    with mode:
        out, scale, masks = torch.ops.mafed.fwd_step(st, te, mask, *_plan_args(L, loss_kind, cls), 1.0, [True, True],
                                                     0, want_masks, 0)
        grads = torch.empty(2, B, T, D, dtype=s_dtype, device="cuda")
        gout = torch.empty((), dtype=torch.float32, device="cuda")
        assert torch.ops.mafed.bwd(st, te, mask, grads, scale, gout, 1.0, None, [True, True], loss_kind, cls, 4,
                                   0) is None
        assert torch.ops.mafed.bwd(st, te, mask, grads, scale, gout, 1.0, 1.0, [True, True], loss_kind, cls, 4,
                                   0) is None
    assert out.shape == (1 + 3 * L,) and out.dtype == torch.float32 and out.device.type == "cuda"
    assert scale.shape == (2 * L,) and scale.dtype == torch.float32
    assert masks.shape == ((2, B, T) if want_masks and not cls else (0,)) and masks.dtype == torch.int64


def test_the_in_place_pass_is_installed_in_front_of_a_callers_pass():
    from torch._inductor import config
    from mafed_b200 import ops
    assert isinstance(config.post_grad_custom_pre_pass, ops._BwdInPlace)
    seen = []

    class Mine(torch._inductor.custom_graph_pass.CustomGraphPass):
        def __call__(self, graph):
            seen.append(graph)

        def uuid(self):
            return "mine"

    saved = config.post_grad_custom_pre_pass
    try:
        config.post_grad_custom_pre_pass = Mine()
        ops.install_graph_pass()
        ops.install_graph_pass()
        p = config.post_grad_custom_pre_pass
        assert isinstance(p, ops._BwdInPlace) and isinstance(p.then, Mine)
        g = torch.fx.Graph()
        g.output(None)
        p(g)
        assert seen == [g]
        assert p.uuid()[2] == "mine"
    finally:
        config.post_grad_custom_pre_pass = saved


def test_the_in_place_pass_warns_on_a_functionalization_layout_it_does_not_handle():
    from mafed_b200 import ops
    g = torch.fx.Graph()
    g.call_function(torch.ops.higher_order.auto_functionalized, (torch.ops.mafed.bwd.default,), {})
    g.output(None)
    with pytest.warns(RuntimeWarning, match="in-place pass"):
        ops._BwdInPlace()(g)


def test_a_compiled_step_sees_the_tuning_address_as_a_plain_int():
    assert cabi._active_tuning_address == 0
    with cabi.tuning(variant=cabi.VARIANT_LDG):
        outer = cabi._active_tuning_address
        assert outer == cabi.active_tuning_address() != 0
        with cabi.tuning(TUNE_NO_TAIL=1):
            assert cabi._active_tuning_address == cabi.active_tuning_address() not in (0, outer)
        assert cabi._active_tuning_address == outer
    assert cabi._active_tuning_address == 0 == cabi.active_tuning_address()
