"""world_size-2 gloo test (CPU) of the host side of the `adaptive` importances over batch shards: the device pass is
replaced by a stand-in that returns fixed per-rank vectors, and the collectives are counted."""
import os
import sys
from types import SimpleNamespace

import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
L, N_VIS, TXT = 3, 2, 4


def _vec(rank, k):
    """What the stand-in pass returns for batch ``k`` of ``rank``: ``[2L + 2]`` fp64, positive counts last."""
    return torch.arange(1, 2 * L + 3, dtype=torch.float64) * (rank + 1) + 10.0 * k


def _ratio(totals):
    """``compute_adaptive_weights``' arithmetic on given totals."""
    sums = totals[: 2 * L].reshape(L, 2)
    lang, image = (sums[:, 0] / totals[2 * L]).float(), (sums[:, 1] / totals[2 * L + 1]).float()
    return lang / (lang + image)


class _Model(torch.nn.Module):
    """Hidden states that depend on a parameter, so that the pass's `autograd.grad` has something to differentiate."""

    def __init__(self):
        super().__init__()
        self.w = torch.nn.Parameter(torch.ones(()))

    def forward(self, x=None, **_):
        hs = tuple(x * self.w * (i + 1) for i in range(L + 1))
        return SimpleNamespace(loss=sum(h.sum() for h in hs), hidden_states=hs)


def _loader(n):
    return [{"x": torch.ones(2, N_VIS + TXT, 8), "attention_mask": torch.ones(2, TXT, dtype=torch.int64)}
            for _ in range(n)]


def _worker(rank, world, port, ret):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), MAFED_B200_DIST="nccl")
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from mafed_b200 import cabi, distill_op
    from mafed_b200.methods import CLMethod, DistillationWeights
    from mafed_b200.methods.distillation_loss_weights import modality_masks

    calls = {"allreduce": 0, "all_gather_object": 0, "pass": 0}
    real_allreduce, real_gather = distill_op.allreduce_sums, dist.all_gather_object

    def allreduce(sums, group=None):
        calls["allreduce"] += 1
        return real_allreduce(sums, group)

    def gather(*a, **kw):
        calls["all_gather_object"] += 1
        return real_gather(*a, **kw)

    batch_index = [0]

    def fake_pass(tensors, attn_mask, n_vis, group=False):
        assert group is False and len(tensors) == L and n_vis == N_VIS
        calls["pass"] += 1
        v = _vec(rank, batch_index[0])
        batch_index[0] += 1
        return v

    real_token_norm_sums = distill_op.token_norm_sums
    distill_op.allreduce_sums, dist.all_gather_object = allreduce, gather
    distill_op.token_norm_sums, distill_op.modality_masks = fake_pass, modality_masks

    def reset():
        for k in calls:
            calls[k] = 0
        batch_index[0] = 0

    n_batches = [2, 3]                 # uneven shards: still one exchange per rank
    local = sum(_vec(rank, k) for k in range(n_batches[rank]))
    union = sum(_vec(r, k) for r in range(world) for k in range(n_batches[r]))
    model = _Model()
    dw = DistillationWeights("adaptive", "discounted", num_hidden_layers=L, distillation_layer=None,
                             num_vision_tokens=N_VIS)

    # the totals: one exchange per call, summed over the ranks' shards
    reset()
    got = dw.gradient_norm_sums(model, _loader(n_batches[rank]), process_group=None)
    assert calls["allreduce"] == 1 and calls["pass"] == n_batches[rank]
    assert torch.equal(got, union)
    reset()
    imp = dw.compute_adaptive_weights(model, _loader(n_batches[rank]), process_group=None)
    assert calls["allreduce"] == 1
    assert torch.equal(imp, _ratio(union))
    # the default, and process_group=False: this rank's own totals, no collective
    for kw in ({}, {"process_group": False}):
        reset()
        got = dw.compute_adaptive_weights(model, _loader(n_batches[rank]), **kw)
        assert calls["allreduce"] == 0 and torch.equal(got, _ratio(local))

    # the strategy: `global_importances` hands its process group to the pass and checks the result
    class Opts:
        tasks = ["a", "b", "c"]; batch_size = 2; seed = 42; pin_mem = False; accumulate_grad_batches = 1

    def make(**kw):
        fd = CLMethod["featdistill"](memory_size=8, opts=Opts(), model_type="vlpythia",
                                     distillation_modality_weighing_strategy="adaptive",
                                     distillation_layer_weighing_strategy="discounted", distillation_layer=None,
                                     num_hidden_layers=L, **kw)
        fd.loss_weights.num_vision_tokens = N_VIS
        fd.data_hooks = (None, lambda loader: loader)
        return fd

    fd = make()
    assert fd.global_importances is False
    reset()
    fd.update(list(range(16)), model, _loader(n_batches[rank]))
    assert calls["allreduce"] == 0 and calls["all_gather_object"] == 0
    assert torch.equal(fd.loss_weights.lang_coeff, _ratio(local)) and fd.task_id == 1

    fd = make(global_importances=True)
    for task in range(2):
        reset()
        fd.update(list(range(16)), model, _loader(n_batches[rank]))
        assert calls["allreduce"] == 1 and calls["all_gather_object"] == 1
    assert torch.equal(fd.loss_weights.lang_coeff, _ratio(union)) and fd.task_id == 2
    every = [None] * world
    real_gather(every, fd.loss_weights.kernel_tables()[2])
    assert every[0] == every[1]

    # the guard: a rank whose weights differ from rank 0's makes every rank raise, naming it
    if rank == 1:
        fd.loss_weights.lang_coeff = fd.loss_weights.lang_coeff + 1e-3
    try:
        fd.check_importances()
        raise AssertionError("check_importances() accepted differing weights")
    except cabi.MafedDistillError as e:
        assert "rank(s) [1]" in str(e)
    fd.loss_weights.lang_coeff = torch.tensor([0.5, 0.25, 0.125])
    fd.check_importances()
    make(process_group=False, global_importances=True).check_importances()   # no group: nothing to compare

    # token_norm_sums over a shard: without a peer communicator one allreduce of the assembled vector, also when the
    # tensors take one pass per dtype
    distill_op.token_norm_sums = real_token_norm_sums
    passes = []

    def fake_dtype_pass(tensors, attn_mask, n_vis, peer=None):
        assert peer is None
        n = len(tensors)
        passes.append(n)
        return torch.arange(1, 2 * n + 3, dtype=torch.float64) * (rank + 1) + 100.0 * len(passes)

    distill_op._token_norm_sums = fake_dtype_pass
    attn = torch.ones(2, TXT, dtype=torch.int64)
    mixed = [torch.zeros(2, N_VIS + TXT, 8, dtype=d) for d in (torch.bfloat16, torch.float32, torch.bfloat16)]
    reset()
    local_mixed = distill_op.token_norm_sums(mixed, attn, N_VIS)
    assert calls["allreduce"] == 0 and passes == [2, 1]
    passes.clear()
    got = distill_op.token_norm_sums(mixed, attn, N_VIS, group=None)
    assert calls["allreduce"] == 1 and passes == [2, 1]
    want = [None] * world
    real_gather(want, local_mixed)
    assert torch.equal(got, want[0] + want[1])
    # per tensor in the caller's order: bf16 pass rows 0 and 1, fp32 pass row 0, then the counts of the last pass
    assert torch.equal(local_mixed[:2], torch.tensor([1.0, 2.0], dtype=torch.float64) * (rank + 1) + 100.0)
    reset()
    passes.clear()
    got = distill_op.token_norm_sums(mixed[:1], attn, N_VIS, group=None)
    assert calls["allreduce"] == 1 and passes == [1]
    ret[rank] = True
    dist.destroy_process_group()


def test_two_rank_adaptive_importances_exchange_once():
    mgr = mp.Manager()
    ret = mgr.dict()
    port = 29900 + os.getpid() % 300
    mp.spawn(_worker, args=(2, port, ret), nprocs=2, join=True)
    assert ret.get(0) and ret.get(1)
