"""How a step over layers of several dtypes is split into launches (CPU): the dtype groups, their order, the group of
refused pairs, the composition with the MAFED_MAX_LAYERS chunking, the sub-plans and where each launch's losses land in
the caller's ``aux``."""
import pytest
import torch

from mafed_b200 import cabi
from mafed_b200.distill_op import DistillPlan, aux_runs, dtype_groups, sub_steps

F32, BF16, F16 = torch.float32, torch.bfloat16, torch.float16
M = cabi.MAX_LAYERS


@pytest.mark.parametrize("pair", [(F32, F32), (BF16, BF16), (F16, F16), (F32, BF16), (F32, F16),
                                  (BF16, F32), (BF16, F16)])
def test_one_pair_is_no_split(pair):
    assert dtype_groups([pair] * 5) is None
    assert dtype_groups([pair]) is None
    assert sub_steps(5, None) is None


def test_bf16_model_with_the_fp32_final_layer_norm_entry():
    pairs = [(BF16, BF16)] * 15 + [(F32, F32)]
    assert dtype_groups(pairs) == [list(range(15)), [15]]


def test_interleaved_dtypes_keep_layer_order_and_first_appearance():
    pairs = [(BF16, BF16), (F32, F32), (BF16, BF16), (F32, BF16), (F32, F32), (BF16, BF16), (F32, BF16)]
    assert dtype_groups(pairs) == [[0, 2, 5], [1, 4], [3, 6]]


def test_fp32_students_with_one_fp32_teacher_layer():
    pairs = [(F32, BF16)] * 3 + [(F32, F32)] + [(F32, BF16)] * 2
    assert dtype_groups(pairs) == [[0, 1, 2, 4, 5], [3]]


def test_refused_pairs_form_one_group_at_the_end():
    pairs = [(BF16, F32), (BF16, BF16), (BF16, F16), (F16, F32), (BF16, BF16), (F32, F32)]
    assert dtype_groups(pairs) == [[1, 4], [5], [0, 2, 3]]


def test_only_refused_pairs_is_one_upcast_launch():
    assert dtype_groups([(BF16, F32), (F16, F32), (BF16, F16)]) is None


def test_groups_compose_with_the_launch_chunking():
    n = 2 * M + 5
    pairs = [(BF16, BF16)] * n
    pairs[7] = (F32, F32)
    groups = dtype_groups(pairs)
    assert groups == [[i for i in range(n) if i != 7], [7]]
    steps = sub_steps(n, groups)
    assert [len(s) for s in steps] == [M, M, 4, 1]
    assert sorted(i for s in steps for i in s) == list(range(n))
    assert all(s == sorted(s) for s in steps)
    # one dtype, too many layers: today's chunks
    assert sub_steps(n, None) == [list(range(0, M)), list(range(M, 2 * M)), list(range(2 * M, n))]
    assert sub_steps(M, None) is None


def test_aux_runs_rebuild_the_caller_order():
    steps = [[0, 2, 3, 5], [1, 4]]
    runs = aux_runs(steps)
    assert runs == [(0, 0, 1), (1, 0, 1), (0, 1, 3), (1, 1, 2), (0, 3, 4)]
    # the same slicing distill_loss does, on the values each launch would return
    vals = {i: (10.0 * i, 10.0 * i + 1, 10.0 * i + 2) for i in range(6)}
    parts = []
    for idx in steps:
        parts.append(torch.tensor([vals[i][0] for i in idx] + [v for i in idx for v in vals[i][1:]]))
    aux = torch.cat([parts[k][lo:hi] for k, lo, hi in runs] +
                    [parts[k][len(steps[k]) + 2 * lo:len(steps[k]) + 2 * hi] for k, lo, hi in runs])
    want = [vals[i][0] for i in range(6)] + [v for i in range(6) for v in vals[i][1:]]
    assert aux.tolist() == want
    assert aux_runs([list(range(M)), list(range(M, M + 3))]) == [(0, 0, M), (1, 0, 3)]


def test_plan_split_is_built_once_per_dtype_signature():
    plan = DistillPlan(layers=[0, 1, 2, 3], layer_coeffs=[0.1, 0.2, 0.3, 0.4], modality_kind=cabi.MODW_TABLE,
                       lang_weights=[0.5, 0.6, 0.7, 0.8], loss_kind=cabi.LOSS_COSINE, n_vis=8, grad_multiplier=2.0,
                       single_pass=False, assumed_grad_out=0.25)
    mixed = ((BF16, BF16), (BF16, BF16), (F32, F32), (BF16, BF16))
    split = plan.split(mixed)
    assert plan.split(mixed) is split
    steps, runs = split
    assert [idx for idx, _ in steps] == [[0, 1, 3], [2]]
    a, b = steps[0][1], steps[1][1]
    assert a.layers == [0, 1, 3] and a.layer_coeffs == [0.1, 0.2, 0.4] and a.lang_weights == [0.5, 0.6, 0.8]
    assert b.layers == [2] and b.layer_coeffs == [0.3] and b.lang_weights == [0.7]
    for sub in (a, b):
        assert (sub.modality_kind, sub.loss_kind, sub.n_vis, sub.grad_multiplier, sub.single_pass,
                sub.assumed_grad_out, sub.distill_coeff, sub.cls) == (cabi.MODW_TABLE, cabi.LOSS_COSINE, 8, 2.0, False,
                                                                      0.25, 1.0, False)
    assert runs == [(0, 0, 2), (1, 0, 1), (0, 2, 3)]
    assert plan.split(((F32, BF16),) * 4) is None


def test_distill_loss_runs_one_step_per_group_and_lays_aux_out_in_caller_order(monkeypatch):
    """The host side of distill_loss with the launch replaced by a stand-in: which layers and sub-plan each step gets,
    masks and the counts ticket, the total in group order, and aux back in the caller's order."""
    from mafed_b200 import distill_op
    calls = []

    def fake_step(plan, attn_mask, group, teachers, mask_out, students, ticket, seen):
        calls.append((plan, [s.dtype for s in students], [t.dtype for t in teachers], mask_out, ticket, seen))
        m = len(plan.layers)
        aux = torch.tensor([100.0 * l for l in plan.layers] + [v for l in plan.layers for v in (l + 0.1, l + 0.2)])
        return torch.tensor(float(sum(plan.layers))), aux, ("masks" if mask_out is not None else None)

    monkeypatch.setattr(distill_op, "_any_step", fake_step)
    types = [BF16, F32, BF16, BF16, F32]
    st = [torch.zeros(1, dtype=d) for d in types]
    plan = DistillPlan(layers=[2, 3, 4, 5, 6], layer_coeffs=[1.0] * 5)
    total, aux, masks = distill_op.distill_loss(st, [s.clone() for s in st], None, plan, mask_out=True, ticket="tk",
                                                seen="seen", return_masks=True)
    assert [c[0].layers for c in calls] == [[2, 4, 5], [3, 6]]
    assert [c[1] for c in calls] == [[BF16] * 3, [F32] * 2] and [c[2] for c in calls] == [[BF16] * 3, [F32] * 2]
    assert [c[3] for c in calls] == [True, None]
    assert all(c[4] == "tk" and c[5] == "seen" for c in calls)
    assert float(total) == 2 + 4 + 5 + 3 + 6 and masks == ("m", "a")
    want = [100.0 * l for l in plan.layers] + [v for l in plan.layers for v in (l + 0.1, l + 0.2)]
    assert aux.tolist() == pytest.approx(want)
    # the second step reuses the sub-plans; one dtype pair is one call with the caller's plan
    distill_op.distill_loss(st, [s.clone() for s in st], None, plan)
    assert calls[2][0] is calls[0][0] and calls[3][0] is calls[1][0]
    calls.clear()
    distill_op.distill_loss(st[:1] * 3, st[:1] * 3, None, DistillPlan(layers=[0, 1, 2], layer_coeffs=[1.0] * 3))
    assert len(calls) == 1 and calls[0][0].layers == [0, 1, 2]
