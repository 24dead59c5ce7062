#!/usr/bin/env python
"""Batch-sharded parity check, one process per GPU (run under torchrun, NCCL):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29511 \
        tools/multirank_check.py

Every rank holds a contiguous slice of the batch; the sharded loss and the concatenation of the
per-rank gradients must equal the single-device CPU oracle on the full batch (SURVEY.md 8e).

``--teacher-dtype {bf16,fp16}``: instead, fp32 student states against a teacher in that dtype (read as it is by the
kernels); every rank's loss and gradient slice must equal the same step run on one GPU over the concatenated batch.

``--mixed-layers``: instead, layers of several dtypes in one step (a bf16 model's states next to its fp32 final-layer-norm
entry, one launch and one exchange per dtype group), with and without token counts sent ahead; compared the same way.

``--adaptive``: instead, the ``adaptive`` importances computed over the ranks' shards of a task loader
(``FeatureDistillation(global_importances=True)``) on the tiny VL model, against one GPU over all the batches, and the
sharded ``replay()`` step that follows; and ``token_norm_sums(..., group=None)`` on a batch shard.

``--teacher-cache-sharded``: instead, ``shard_teacher_cache=True``: each rank's shard against the replicated cache, and
a sharded cached ``replay()`` step whose every rank's batch draws rows from every rank's shard, against the
``teacher_cache=True`` step (bit for bit) and one GPU on the concatenated batch; then a second ``update()`` that
releases and rebuilds the shards.
"""
import argparse
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--teacher-dtype", choices=["bf16", "fp16"], default=None,
                    help="fp32 students against a teacher in this dtype (default: today's same-dtype cases)")
    ap.add_argument("--mixed-layers", action="store_true",
                    help="layers of several dtypes in one step, one launch per dtype group")
    ap.add_argument("--adaptive", action="store_true",
                    help="adaptive importances over the ranks' loader shards, then a sharded replay() step")
    ap.add_argument("--teacher-cache", action="store_true",
                    help="replay() steps with teacher_cache=True, sharded, against one GPU on the concatenated batch")
    ap.add_argument("--teacher-cache-sharded", action="store_true",
                    help="shard_teacher_cache=True against the replicated cache and one GPU on the concatenated batch")
    args = ap.parse_args()
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    if args.teacher_dtype is not None:
        ok = mixed_teacher_check(rank, world, {"bf16": torch.bfloat16, "fp16": torch.float16}[args.teacher_dtype])
        finish(ok)
    if args.mixed_layers:
        finish(mixed_layers_check(rank, world))
    if args.teacher_cache:
        finish(teacher_cache_check(rank, world))
    if args.teacher_cache_sharded:
        finish(teacher_cache_sharded_check(rank, world))
    if args.adaptive:
        ok = shard_norm_sums_check(rank, world)
        finish(adaptive_check(rank, world) and ok)
    from gpu_util import Out, make_method, rel_err
    from golden_util import oracle_cfg
    from oracle import distill_oracle as O

    ok = True
    for dtype, loss, modality, single_pass in [(torch.float32, "mse", "equal", True), (torch.bfloat16, "mse", "balanced", True),
                                               (torch.bfloat16, "cosine", "equal", False), (torch.float32, "mse", "equal", False)]:
        B = 4 * world + 2  # uneven shards: the last rank gets the remainder
        st, te, am = O.make_inputs(4, B, 9, 768, n_vis=256, dtype=dtype, seed=31, mask="ragged")
        meta = dict(modality=modality, layer_strategy="discounted", loss=loss, gamma=0.5, num_hidden_layers=3,
                    layer=None, n_vis=256, coeff=1.0, cls=False, lang_coeff=None)
        ref = O.forward_backward(st, te, am, oracle_cfg(meta), grad_out=0.5 if not single_pass else 1.0)
        lo = rank * 4
        hi = B if rank == world - 1 else lo + 4
        fd = make_method(meta, single_pass=single_pass)
        fd.grad_multiplier = 1.0      # hidden-state gradients of the GLOBAL loss (the DDP convention is checked below)
        leaves = [s[lo:hi].cuda().contiguous().requires_grad_(True) for s in st]
        teach = [t[lo:hi].cuda().contiguous() for t in te]
        fd.past_model = lambda **kw: Out(tuple(teach))
        loss_v = fd.distill(Out(tuple(leaves)), {"attention_mask": am[lo:hi].cuda()})
        (loss_v * (0.5 if not single_pass else 1.0)).backward()
        torch.cuda.synchronize()
        tol = 1e-5 if dtype == torch.float32 else 2e-3
        e_loss = abs(float(loss_v) - float(ref["loss"])) / abs(float(ref["loss"]))
        e_grad = max(rel_err(leaves[l].grad.float().cpu(), ref["grads"][l][lo:hi].float()) for l in range(3))
        good = e_loss < tol and e_grad < tol
        ok &= good
        print(f"rank {rank}/{world} {dtype} {loss} {modality} single_pass={single_pass}: loss err {e_loss:.2e} "
              f"grad err {e_grad:.2e} {'OK' if good else 'FAIL'}", flush=True)
    from mafed_b200.comm import get_peer_comm
    peer = get_peer_comm(None)
    mode = "nccl" if peer is None else "peer-memory"
    if peer is not None:
        ok &= peer.status() == 0
    if peer is not None:
        ok &= graph_replay_check(rank, world)
        ok &= peer.status() == 0
        ok &= prefetch_check(rank, world)
        ok &= peer.status() == 0
        ok &= host_step_check(rank, world)
        ok &= peer.status() == 0
    ok &= ddp_check(rank, world)
    if os.environ.get("MAFED_B200_DIST", "peer") == "peer":
        ok &= peer is not None          # on one NVLink box the mailboxes must map
    print(f"rank {rank}: exchange path = {mode}", flush=True)
    finish(ok)


def finish(ok):
    """Exit 0 when every rank passed."""
    flag = torch.tensor([1 if ok else 0], device="cuda")
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    dist.barrier()
    dist.destroy_process_group()
    sys.exit(0 if int(flag) == 1 else 1)


def mixed_teacher_check(rank, world, teacher_dtype):
    """fp32 student states, half-precision teacher, batch-sharded one-pass and two-pass steps: the loss equals the
    one-GPU step on the concatenated batch to 1e-6 (the sums are added in another order) and every rank's gradient
    slice equals it bit for bit (mse) or to 1e-6 (cosine: the row statistics of another tile geometry)."""
    from gpu_util import Out, make_method, rel_err
    from mafed_b200.comm import get_peer_comm
    from oracle import distill_oracle as O
    # MAFED_B200_DIST=nccl: no communicator, the sharded steps run the NCCL sequence of ctypes calls (_DistillFunction)
    mode = "nccl" if get_peer_comm(None) is None else "peer-memory"
    ok = True
    for loss, single_pass in [("mse", True), ("cosine", True), ("mse", False), ("cosine", False)]:
        B = 4 * world + 2
        st, te, am = O.make_inputs(4, B, 9, 768, n_vis=256, seed=37, mask="ragged", teacher="independent")
        te = [t.to(teacher_dtype) for t in te]
        meta = dict(modality="equal", layer_strategy="discounted", loss=loss, gamma=0.5, num_hidden_layers=3,
                    layer=None, n_vis=256, coeff=1.0, cls=False, lang_coeff=None)
        lo = rank * 4
        hi = B if rank == world - 1 else lo + 4

        def run(a, b, group):
            fd = make_method(meta, single_pass=single_pass)
            fd.grad_multiplier = 1.0
            fd.process_group = group
            leaves = [s[a:b].cuda().contiguous().requires_grad_(True) for s in st]
            teach = [t[a:b].cuda().contiguous() for t in te]
            fd.past_model = lambda **kw: Out(tuple(teach))
            loss_v = fd.distill(Out(tuple(leaves)), {"attention_mask": am[a:b].cuda()})
            (loss_v * 0.5).backward()
            torch.cuda.synchronize()
            return loss_v.detach(), [l.grad for l in leaves]

        loss_s, g_s = run(lo, hi, None)
        loss_f, g_f = run(0, B, False)
        e_loss = abs(float(loss_s) - float(loss_f)) / abs(float(loss_f))
        pairs = [(a, b[lo:hi]) for a, b in zip(g_s, g_f) if b is not None]
        if loss == "mse":
            same = all(torch.equal(a, b) for a, b in pairs)
        else:
            same = max(rel_err(a.cpu(), b.cpu()) for a, b in pairs) < 1e-6
        good = e_loss < 1e-6 and same and len(pairs) == 3
        ok &= good
        print(f"rank {rank}/{world} ({mode}) fp32 student, {teacher_dtype} teacher, {loss} single_pass={single_pass}: "
              f"loss err {e_loss:.2e} gradients {'equal' if same else 'DIFFER'} {'OK' if good else 'FAIL'}", flush=True)
    return ok


def mixed_layers_check(rank, world):
    """Students and teachers {bf16 x 3, fp32}: one launch per dtype group, each with its own exchange, one-pass and
    two-pass, with the token counts exchanged in the kernels or sent ahead (``prefetch_counts``, whose ticket every
    group's launch reads).  The loss equals the one-GPU step on the concatenated batch to 1e-6 and every rank's gradient
    slice equals it bit for bit (mse) or within 1e-6 / 2e-3 for fp32 / bf16 (cosine)."""
    from gpu_util import Out, make_method, rel_err
    from mafed_b200.comm import get_peer_comm
    from oracle import distill_oracle as O
    peer = get_peer_comm(None)
    mode = "nccl" if peer is None else "peer-memory"
    dtypes = [torch.bfloat16] * 3 + [torch.float32]
    ok = True
    for loss, single_pass, ahead in [("mse", True, False), ("cosine", True, False), ("mse", False, False),
                                     ("cosine", False, False), ("mse", True, True), ("mse", False, True)]:
        B = 4 * world + 2
        st, te, am = O.make_inputs(4, B, 9, 768, n_vis=256, seed=43, mask="ragged", teacher="independent")
        meta = dict(modality="balanced", layer_strategy="discounted", loss=loss, gamma=0.5, num_hidden_layers=4,
                    layer=None, n_vis=256, coeff=1.0, cls=False, lang_coeff=None)
        lo = rank * 4
        hi = B if rank == world - 1 else lo + 4

        def run(a, b, group):
            fd = make_method(meta, single_pass=single_pass)
            fd.grad_multiplier = 1.0
            fd.process_group = group
            leaves = [s[a:b].to(d).cuda().contiguous().requires_grad_(True) for s, d in zip(st, dtypes)]
            teach = [t[a:b].to(d).cuda().contiguous() for t, d in zip(te, dtypes)]
            fd.past_model = lambda **kw: Out(tuple(teach))
            batch = {"attention_mask": am[a:b].cuda().contiguous()}
            if ahead and group is None:
                assert fd.prefetch_counts(batch) is not None or peer is None
            loss_v = fd.distill(Out(tuple(leaves)), batch)
            (loss_v * 0.5).backward()
            torch.cuda.synchronize()
            return loss_v.detach(), [l.grad for l in leaves]

        loss_s, g_s = run(lo, hi, None)
        loss_f, g_f = run(0, B, False)
        e_loss = abs(float(loss_s) - float(loss_f)) / abs(float(loss_f))
        pairs = [(a, b[lo:hi]) for a, b in zip(g_s, g_f)]
        if loss == "mse":
            same = all(a.dtype == b.dtype and torch.equal(a, b) for a, b in pairs)
        else:
            same = all(rel_err(a.cpu(), b.cpu()) < (1e-6 if a.dtype == torch.float32 else 2e-3) for a, b in pairs)
        good = e_loss < 1e-6 and same
        ok &= good
        print(f"rank {rank}/{world} ({mode}) bf16 x 3 + fp32 layers, {loss} single_pass={single_pass} "
              f"counts_ahead={ahead}: loss err {e_loss:.2e} gradients {'equal' if same else 'DIFFER'} "
              f"{'OK' if good else 'FAIL'}", flush=True)
    if peer is not None:
        ok &= peer.status() == 0
    return ok


def teacher_cache_check(rank, world):
    """``teacher_cache=True`` on a batch-sharded run: every rank builds the same cache over the whole memory, with no
    exchange, and a sharded cached ``replay()`` step without a replay loss (its loss is the global-batch distillation
    loss) equals one GPU's cached step on the concatenated batch: loss to 1e-5, the ranks' summed parameter gradients to
    1e-4 (fp32 model: the sums run in another order).  The shards are padded to the global batch's text length, so the
    student sees the same tokens as in the one-GPU batch."""
    import copy
    from torch.utils.data import ConcatDataset
    from gpu_util import rel_err
    from mafed_b200.methods import CLMethod
    from mafed_b200.teacher_cache import repad_left
    from tiny_vl import TinyVL
    from vl_memory import VLSamples, collate

    class Opts:
        tasks = ["a", "b"]; batch_size = 4; seed = 1; pin_mem = False; accumulate_grad_batches = 1

    torch.manual_seed(0)
    teacher = TinyVL(fp32_island=True).cuda()
    student = copy.deepcopy(teacher)
    with torch.no_grad():
        for p in student.parameters():
            p.add_(0.02 * torch.randn_like(p))

    def strategy(group):
        fd = CLMethod["featdistill"](memory_size=32, opts=Opts(), model_type="vlpythia",
                                     distillation_modality_weighing_strategy="balanced",
                                     distillation_layer_weighing_strategy="discounted", distillation_layer=None,
                                     num_hidden_layers=3, replay_coeff=0.0, teacher_cache=True, process_group=group,
                                     grad_multiplier=1.0)
        fd.num_vision_tokens, fd.num_workers = 8, 0
        fd.data_hooks = (collate, lambda loader: loader)
        fd.update(dataset=VLSamples(64, seed=3, max_txt=9), model=teacher, dataloader=None)
        return fd

    def step(fd, idx, text_len):
        memory = ConcatDataset(fd.datasets)
        batch = repad_left(collate([memory[i] for i in idx]), text_len)
        batch.pop("labels")
        batch = {k: v.cuda() if torch.is_tensor(v) else v for k, v in batch.items()}
        batch["memory_index"] = list(idx)
        fd.mem_dataloader = [batch]
        model = copy.deepcopy(student)
        loss, n_ex = fd.replay(model)
        loss.backward()
        torch.cuda.synchronize()
        return loss.detach(), n_ex, [p.grad for p in model.parameters()]

    sharded, full = strategy(None), strategy(False)
    same_cache = all(_all_equal(s) for s in sharded._teacher_cache.states)
    B = 4 * world + 2
    idx = [(5 * i) % 32 for i in range(B)]
    memory = ConcatDataset(full.datasets)
    text_len = max(len(memory[i]["input_ids"]) for i in idx)
    lo = rank * 4
    hi = B if rank == world - 1 else lo + 4
    loss_s, n_s, g_s = step(sharded, idx[lo:hi], text_len)
    loss_f, n_f, g_f = step(full, idx, text_len)
    e_loss = abs(float(loss_s) - float(loss_f)) / abs(float(loss_f))
    e_grad = 0.0
    for a, b in zip(g_s, g_f):
        if b is None:
            e_grad = e_grad if a is None else float("inf")
            continue
        dist.all_reduce(a)
        e_grad = max(e_grad, rel_err(a, b))
    good = same_cache and n_s == hi - lo and n_f == B and e_loss < 1e-5 and e_grad < 1e-4
    print(f"rank {rank}/{world} teacher cache: caches equal on every rank {same_cache}, loss err {e_loss:.2e}, "
          f"summed gradient err {e_grad:.2e} {'OK' if good else 'FAIL'}", flush=True)
    return good


def teacher_cache_sharded_check(rank, world):
    """``shard_teacher_cache=True``: every rank's ``local_states`` equal the replicated cache's rows of its samples and
    its ``nbytes`` is its shard; a sharded cached ``replay()`` step in which every rank's batch holds a sample of every
    rank's shard equals the replicated-cache step on the same ranks bit for bit (loss, every parameter gradient, the
    batch masks) and one GPU's step on the concatenated batch within ``teacher_cache_check``'s tolerances; a second
    ``update()`` releases the first task's shards and builds the next ones."""
    import copy
    from torch.utils.data import ConcatDataset
    from gpu_util import rel_err
    from mafed_b200 import teacher_cache as TC
    from mafed_b200.methods import CLMethod
    from tiny_vl import TinyVL
    from vl_memory import VLSamples, collate

    class Opts:
        tasks = ["a", "b", "c"]; batch_size = 4; seed = 1; pin_mem = False; accumulate_grad_batches = 1

    torch.manual_seed(0)
    teacher = TinyVL(fp32_island=True).cuda()
    student = copy.deepcopy(teacher)
    with torch.no_grad():
        for p in student.parameters():
            p.add_(0.02 * torch.randn_like(p))

    def strategy(group, shard):
        fd = CLMethod["featdistill"](memory_size=64, opts=Opts(), model_type="vlpythia",
                                     distillation_modality_weighing_strategy="balanced",
                                     distillation_layer_weighing_strategy="discounted", distillation_layer=None,
                                     num_hidden_layers=3, replay_coeff=0.0, teacher_cache=True,
                                     shard_teacher_cache=shard, process_group=group, grad_multiplier=1.0)
        fd.num_vision_tokens, fd.num_workers = 8, 0
        fd.data_hooks = (collate, lambda loader: loader)
        fd.update(dataset=VLSamples(64, seed=3, max_txt=9), model=teacher, dataloader=None)
        return fd

    def step(fd, idx, text_len):
        memory = ConcatDataset(fd.datasets)
        batch = TC.repad_left(collate([memory[i] for i in idx]), text_len)
        batch.pop("labels")
        batch = {k: v.cuda() if torch.is_tensor(v) else v for k, v in batch.items()}
        batch["memory_index"] = list(idx)
        fd.mem_dataloader = [batch]
        model = copy.deepcopy(student)
        loss, n_ex = fd.replay(model)
        loss.backward()
        torch.cuda.synchronize()
        return loss.detach(), n_ex, [p.grad for p in model.parameters()], batch

    sharded, replicated, full = strategy(None, True), strategy(None, False), strategy(False, False)
    cache, whole = sharded._teacher_cache, replicated._teacher_cache
    ok = isinstance(cache, TC.ShardedTeacherCache)
    mine = [i for i in range(cache.M) if cache.owner[i] == rank]
    ok &= all(torch.equal(a, b[mine]) for a, b in zip(cache.local_states, whole.states))
    sizes = [s.element_size() for s in whole.states]
    ok &= cache.nbytes == TC.shard_layout(max(cache.count), cache.T_c, cache.D, sizes)[1]
    ok &= cache.count[rank] == len(mine)
    # rank r's batch: one sample of build batch (r + j) % world -- held by rank (r + j) % world -- per j, and one more
    n_batches = -(-cache.M // 4)
    per_rank = [[((r + j) % world % n_batches) * 4 + (r + j) % 4 for j in range(world)] + [(3 * r + 1) % cache.M]
                for r in range(world)]
    idx = per_rank[rank]
    every = [i for r in per_rank for i in r]
    memory = ConcatDataset(full.datasets)
    text_len = max(len(memory[i]["input_ids"]) for i in every)
    remote = sum(cache.owner[i] != rank for i in idx)
    loss_s, n_s, g_s, b_s = step(sharded, idx, text_len)
    loss_r, n_r, g_r, b_r = step(replicated, idx, text_len)
    same = torch.equal(loss_s, loss_r) and n_s == n_r == len(idx)
    same &= all((a is None) == (b is None) and (a is None or torch.equal(a, b)) for a, b in zip(g_s, g_r))
    same &= all(torch.equal(b_s[k], b_r[k]) for k in ("lang_masks", "image_masks"))
    loss_f, n_f, g_f, _ = step(full, every, text_len)
    e_loss = abs(float(loss_s) - float(loss_f)) / abs(float(loss_f))
    e_grad = 0.0
    for a, b in zip(g_s, g_f):
        if b is None:
            e_grad = e_grad if a is None else float("inf")
            continue
        a = a.clone()
        dist.all_reduce(a)
        e_grad = max(e_grad, rel_err(a, b))
    close = n_f == len(every) and e_loss < 1e-5 and e_grad < 1e-4
    # the next task: update() releases these shards (collectively) before it builds the new ones
    first = cache
    sharded.update(dataset=VLSamples(64, seed=4, max_txt=9), model=teacher, dataloader=None)
    second = sharded._teacher_cache
    rebuilt = first._handle is None and isinstance(second, TC.ShardedTeacherCache) and second.M == 2 * first.M
    replicated.update(dataset=VLSamples(64, seed=4, max_txt=9), model=teacher, dataloader=None)
    mine2 = [i for i in range(second.M) if second.owner[i] == rank]
    rebuilt &= all(torch.equal(a, b[mine2]) for a, b in zip(second.local_states, replicated._teacher_cache.states))
    second.release()
    good = ok and same and close and rebuilt and remote >= world - 1
    print(f"rank {rank}/{world} sharded teacher cache: {len(mine)} of {cache.M} samples, {cache.nbytes} bytes "
          f"(replicated {whole.nbytes}), shard rows equal {ok}, step of {len(idx)} samples ({remote} from peers) "
          f"bit-identical to the replicated cache {same}, against one GPU: loss err {e_loss:.2e} summed gradient err "
          f"{e_grad:.2e}, released and rebuilt {rebuilt} {'OK' if good else 'FAIL'}", flush=True)
    return good


def _max_rel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return float(((a - b).abs() / b.abs().clamp_min(1e-300)).max())


def _all_equal(t):
    """True when ``t`` holds the same bits on every rank."""
    every = [torch.empty_like(t) for _ in range(dist.get_world_size())]
    dist.all_gather(every, t.contiguous())
    return all(torch.equal(e, every[0]) for e in every)


def shard_norm_sums_check(rank, world):
    """``token_norm_sums(..., group=None)`` on uneven ragged batch shards, one dtype (with a communicator: the exchange
    inside the reduce launch) and bf16 x 3 + fp32 (one pass per dtype, one allreduce of the assembled vector): the same
    bits on every rank, equal to the ranks' own vectors added in rank order to 1e-12, and to one GPU's pass over the
    whole batch to 1e-6 (its per-CTA fp32 partials group the tokens differently)."""
    from mafed_b200.comm import get_peer_comm
    from mafed_b200.distill_op import token_norm_sums
    mode = "nccl" if get_peer_comm(None) is None else "peer-memory"
    g = torch.Generator().manual_seed(71)
    B, n_vis, txt, D = 3 * world + 1, 256, 9, 768
    full = [torch.randn(B, n_vis + txt, D, generator=g) * (0.5 + l) for l in range(4)]
    am = torch.ones(B, txt, dtype=torch.int64)
    for b in range(B):
        am[b, : (2 * b) % txt] = 0
    lo = 3 * rank
    hi = B if rank == world - 1 else lo + 3
    ok = True
    for name, dtypes in (("fp32", [torch.float32] * 4), ("bf16 x 3 + fp32", [torch.bfloat16] * 3 + [torch.float32])):
        shard = [t[lo:hi].to(d).cuda().contiguous() for t, d in zip(full, dtypes)]
        mask = am[lo:hi].cuda().contiguous()
        mine = token_norm_sums(shard, mask, n_vis)
        every = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(every, mine)
        in_order = every[0].clone()
        for e in every[1:]:
            in_order = in_order + e
        glob = token_norm_sums(shard, mask, n_vis, group=None)
        one = token_norm_sums([t.to(d).cuda().contiguous() for t, d in zip(full, dtypes)], am.cuda(), n_vis)
        torch.cuda.synchronize()
        same, e_ranks, e_one = _all_equal(glob), _max_rel(glob, in_order), _max_rel(glob, one)
        good = same and e_ranks < 1e-12 and e_one < 1e-6
        ok &= good
        print(f"rank {rank}/{world} ({mode}) token_norm_sums on a shard, {name}: same on all ranks {same}, "
              f"vs ranks' vectors {e_ranks:.1e}, vs one GPU {e_one:.1e} {'OK' if good else 'FAIL'}", flush=True)
    return ok


def adaptive_check(rank, world):
    """``adaptive`` importances of a batch-sharded run (``FeatureDistillation(global_importances=True)``), the tiny VL
    model, every rank on its shard of a seeded task loader of uneven length (``update()``, then a second task):
    (a) ``lang_coeff`` is bit-identical on every rank; (b) the exchanged fp64 totals, and the importances formed from them
    in fp64, equal one GPU's pass over all the batches to 1e-12 (only the order of the additions over batches differs),
    and ``lang_coeff`` (the fp32 running average over the tasks) equals that GPU's to 1e-6; (c) the sharded ``replay()`` step that follows (no replay
    loss, so the loss is the global one) gives the same loss on every rank, and parameter gradients summed over the
    ranks equal the one-GPU step on the concatenated memory batch within the fp32 tolerance (1e-5).  The model runs in
    fp32 (``fp32_island``): under bf16 autocast the ranks' weight gradients come out of bf16 products, and their sum
    differed from the full-batch product by 2.4e-3 here, with the loss bit-identical."""
    import copy

    from gpu_util import rel_err
    from mafed_b200.comm import get_peer_comm
    from mafed_b200.methods import CLMethod, DistillationWeights
    from tiny_vl import TinyVL, make_batch
    mode = "nccl" if get_peer_comm(None) is None else "peer-memory"
    n_vis, L = 8, 3

    class Opts:
        tasks = ["a", "b", "c"]; batch_size = 4; seed = 1; pin_mem = False; accumulate_grad_batches = 1

    def strategy(group, global_importances):
        fd = CLMethod["featdistill"](memory_size=8, opts=Opts(), model_type="vlpythia",
                                     distillation_modality_weighing_strategy="adaptive",
                                     distillation_layer_weighing_strategy="discounted", distillation_layer=None,
                                     num_hidden_layers=L, gamma=0.5, replay_coeff=0.0, distillation_coeff=2.0,
                                     process_group=group, grad_multiplier=1.0, global_importances=global_importances)
        fd.num_vision_tokens = fd.loss_weights.num_vision_tokens = n_vis
        fd.data_hooks = (None, lambda loader: loader)
        return fd

    def ratio64(t):
        lang, image = t[0:2 * L:2] / t[2 * L], t[1:2 * L:2] / t[2 * L + 1]
        return lang / (lang + image)

    torch.manual_seed(0)
    model = TinyVL(n_vis=n_vis, fp32_island=True).cuda()
    model.gpt_neox.config._attn_implementation = "eager"    # SDPA's memory-efficient backward adds with atomics
    tasks = [[make_batch(bsz=3 + i % 3, seed=100 * t + i, device="cuda") for i in range(2 * world + 1)] for t in (1, 2)]
    fd = strategy(None, True)
    one = DistillationWeights("adaptive", "discounted", num_hidden_layers=L, distillation_layer=None,
                              num_vision_tokens=n_vis)
    ok = True
    for k, batches in enumerate(tasks):
        fd.update(list(range(16)), model, [dict(b) for b in batches[rank::world]])
        glob = fd.loss_weights.gradient_norm_sums(model, [dict(b) for b in batches[rank::world]], process_group=None)
        tot1 = one.gradient_norm_sums(model, [dict(b) for b in batches])
        one.update_weights(model, [dict(b) for b in batches], k)
        torch.cuda.synchronize()
        coeff = fd.loss_weights.lang_coeff
        same = _all_equal(coeff) and _all_equal(glob)
        e_tot, e_imp = _max_rel(glob, tot1), _max_rel(ratio64(glob), ratio64(tot1))
        e_coeff = _max_rel(coeff, one.lang_coeff)
        good = same and e_tot < 1e-12 and e_imp < 1e-12 and e_coeff < 1e-6
        ok &= good
        print(f"rank {rank}/{world} ({mode}) adaptive importances, task {k}: lang_coeff {coeff.tolist()} "
              f"same on all ranks {same}; vs one GPU: totals {e_tot:.1e}, fp64 importances {e_imp:.1e}, "
              f"lang_coeff {e_coeff:.1e} {'OK' if good else 'FAIL'}", flush=True)

    # the sharded replay() step against one GPU on the concatenated memory batch, with these weights
    torch.manual_seed(1)
    with torch.no_grad():
        for p in model.parameters():
            p.add_(0.02 * torch.randn_like(p))                       # the student has moved away from the teacher
    single = copy.deepcopy(model)
    mem = make_batch(bsz=2 * world + 1, seed=300, device="cuda")
    lo = 2 * rank
    hi = mem["input_ids"].shape[0] if rank == world - 1 else lo + 2
    fd.mem_dataloader = [{k: v[lo:hi].contiguous() for k, v in mem.items()}]
    loss, n_ex = fd.replay(model)
    loss.backward()
    grads = [p.grad if p.grad is not None else torch.zeros_like(p) for p in model.parameters()]
    for g in grads:
        dist.all_reduce(g)
    ref = strategy(False, False)
    ref.past_model, ref.task_id = fd.past_model, fd.task_id
    ref.loss_weights.lang_coeff = fd.loss_weights.lang_coeff.clone()
    ref.mem_dataloader = [dict(mem)]
    loss1, _ = ref.replay(single)
    loss1.backward()
    want = [p.grad if p.grad is not None else torch.zeros_like(p) for p in single.parameters()]
    torch.cuda.synchronize()
    same = _all_equal(loss.detach().reshape(1))
    e_loss = abs(float(loss) - float(loss1)) / abs(float(loss1))
    e_grad = max(rel_err(a.cpu(), b.cpu()) for a, b in zip(grads, want) if b.abs().sum() > 0)
    good = same and n_ex == hi - lo and e_loss < 1e-5 and e_grad < 1e-5
    ok &= good
    print(f"rank {rank}/{world} ({mode}) sharded replay() with the global importances: loss same on all ranks {same}, "
          f"vs one GPU: loss {e_loss:.1e} parameter gradients {e_grad:.1e} {'OK' if good else 'FAIL'}", flush=True)
    peer = get_peer_comm(None)
    if peer is not None:
        ok &= peer.status() == 0
    if os.environ.get("MAFED_B200_DIST", "peer") == "peer":
        ok &= peer is not None
    return ok


def graph_replay_check(rank, world):
    """The sharded one-pass step captured into a CUDA graph (both exchanges inside the fused kernel, epochs on the
    device), replayed with new data, then followed by eager steps: every result equals the full-batch oracle."""
    from golden_util import oracle_cfg
    from gpu_util import rel_err
    from mafed_b200 import cabi
    from mafed_b200.distill_op import DistillPlan, distill_backward, distill_fused
    from oracle import distill_oracle as O
    meta = dict(modality="equal", layer_strategy="discounted", loss="mse", gamma=0.5, num_hidden_layers=3,
                layer=None, n_vis=256, coeff=1.0, cls=False, lang_coeff=None)
    cfg = oracle_cfg(meta)
    layers, coeffs, _ = O.layer_plan(cfg)
    plan = DistillPlan(layers=layers, layer_coeffs=[float(c) for c in coeffs], modality_kind=cabi.MODW_EQUAL)
    B = 3 * world
    lo, hi = 3 * rank, 3 * rank + 3

    def data(seed):
        st, te, am = O.make_inputs(4, B, 9, 768, n_vis=256, dtype=torch.bfloat16, seed=seed, mask="ragged")
        return st, te, am, O.forward_backward(st, te, am, cfg)

    st, te, am, ref = data(41)
    s = [x[lo:hi].cuda().contiguous() for x in st[:3]]
    t = [x[lo:hi].cuda().contiguous() for x in te[:3]]
    g = [torch.empty_like(x) for x in s]
    mask = am[lo:hi].cuda().contiguous()
    gout = torch.ones((), device="cuda")

    def step():
        out, scale, ln = distill_fused(s, t, g, mask, plan, group=None)
        distill_backward(ln, g, scale, gout, skip_if_equals=1.0)
        return out

    def good(out, ref):
        torch.cuda.synchronize()
        e_loss = abs(float(out[0]) - float(ref["loss"])) / abs(float(ref["loss"]))
        e_grad = max(rel_err(g[l].float().cpu(), ref["grads"][l][lo:hi].float()) for l in range(3))
        return e_loss < 2e-3 and e_grad < 2e-3

    ok = True
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        for _ in range(2):
            out = step()
    torch.cuda.current_stream().wait_stream(side)
    ok &= good(out, ref)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = step()
    for seed in (42, 43, 44):
        st, te, am, ref = data(seed)
        for dst, src in zip(s + t, [x[lo:hi] for x in st[:3]] + [x[lo:hi] for x in te[:3]]):
            dst.copy_(src)
        mask.copy_(am[lo:hi])
        graph.replay()
        ok &= good(out, ref)
    eager = step()                      # eager steps after replays: the device-side epochs simply go on
    ok &= good(eager, ref)
    # a rank that arrives late (data loader hiccup, checkpoint write): the peers' kernels wait for it inside the
    # spin bound (60 s by default) and the step is still exact
    import time
    torch.cuda.synchronize()
    if rank == world - 1:
        time.sleep(3.0)
    late = step()
    ok &= good(late, ref)
    print(f"rank {rank}: CUDA-graph replay of the sharded step {'OK' if ok else 'FAIL'}", flush=True)
    return ok


def prefetch_check(rank, world):
    """Token counts sent ahead of the step (`fd.prefetch_counts`): one and two batches ahead, uneven ragged shards,
    a late rank -- every step equals the full-batch oracle; a stale ticket (mask edited after the prefetch) is not
    used."""
    import time

    from golden_util import oracle_cfg
    from gpu_util import Out, make_method, rel_err
    from oracle import distill_oracle as O
    meta = dict(modality="equal", layer_strategy="discounted", loss="mse", gamma=0.5, num_hidden_layers=3,
                layer=None, n_vis=256, coeff=1.0, cls=False, lang_coeff=None)
    cfg = oracle_cfg(meta)
    B = 3 * world
    lo, hi = 3 * rank, 3 * rank + 3
    fd = make_method(meta)
    fd.grad_multiplier = 1.0
    batches = []
    for seed in (51, 52, 53, 54, 55):
        st, te, am = O.make_inputs(4, B, 9, 768, n_vis=256, dtype=torch.float32, seed=seed, mask="ragged")
        batches.append((st, te, am, O.forward_backward(st, te, am, cfg), am[lo:hi].cuda().contiguous()))
    ok = True

    def run(i):
        st, te, am, ref, mask = batches[i]
        leaves = [x[lo:hi].cuda().contiguous().requires_grad_(True) for x in st]
        teach = [x[lo:hi].cuda().contiguous() for x in te]
        fd.past_model = lambda **kw: Out(tuple(teach))
        loss = fd.distill(Out(tuple(leaves)), {"attention_mask": mask})
        loss.backward()
        torch.cuda.synchronize()
        e_loss = abs(float(loss) - float(ref["loss"])) / abs(float(ref["loss"]))
        e_grad = max(rel_err(leaves[l].grad.cpu(), ref["grads"][l][lo:hi]) for l in range(3))
        return e_loss < 1e-5 and e_grad < 1e-5

    # one ahead, two ahead, and a step whose ticket is stale
    assert fd.prefetch_counts({"attention_mask": batches[0][4]}) is not None
    fd.prefetch_counts({"attention_mask": batches[1][4]})
    ok &= run(0)
    fd.prefetch_counts({"attention_mask": batches[2][4]})
    ok &= run(1)
    if rank == world - 1:
        time.sleep(2.0)                 # a late rank: its counts were sent long ago, the sums exchange waits for it
    ok &= run(2)
    fd.prefetch_counts({"attention_mask": batches[3][4]})
    batches[3][4].add_(0)               # in-place touch: the ticket no longer matches the tensor's version
    ok &= run(3)                        # -> counts exchanged inside the kernel instead
    ok &= run(4)                        # no prefetch at all
    print(f"rank {rank}: prefetched token counts {'OK' if ok else 'FAIL'}", flush=True)
    return ok


def host_step_check(rank, world):
    """The C ABI's host-buffer step with a communicator (`mafed_host_step_run(..., comm)`) against the oracle."""
    from golden_util import oracle_cfg
    from gpu_util import make_method, rel_err
    from mafed_b200.host_step import CHostStep
    from oracle import distill_oracle as O
    meta = dict(modality="balanced", layer_strategy="discounted", loss="mse", gamma=0.5, num_hidden_layers=3,
                layer=None, n_vis=256, coeff=1.0, cls=False, lang_coeff=None)
    B = 2 * world
    lo, hi = 2 * rank, 2 * rank + 2
    st, te, am = O.make_inputs(4, B, 9, 1024, n_vis=256, dtype=torch.bfloat16, seed=61, mask="ragged")
    ref = O.forward_backward(st, te, am, oracle_cfg(meta))
    fd = make_method(meta)
    hs = CHostStep(fd, [x[lo:hi].contiguous() for x in st[:3]], [x[lo:hi].contiguous() for x in te[:3]],
                   am[lo:hi].contiguous(), torch.device("cuda", torch.cuda.current_device()))
    ok = hs.comm is not None
    for _ in range(2):
        loss = hs.step()
        e_loss = abs(float(loss) - float(ref["loss"])) / abs(float(ref["loss"]))
        e_grad = max(rel_err(hs.h_g[l].float(), ref["grads"][l][lo:hi].float()) for l in range(3))
        ok &= e_loss < 2e-3 and e_grad < 2e-3
    hs.close()
    print(f"rank {rank}: sharded host-buffer step {'OK' if ok else 'FAIL'}", flush=True)
    return ok


def ddp_check(rank, world):
    """ADVICE r1 (high): under DistributedDataParallel the distillation term must weigh what it weighs on one GPU.
    A tiny model whose forward returns a hidden-state tuple, wrapped in DDP, each rank on its shard with the
    strategy's defaults (batch-sharded global loss, gradients multiplied by world_size because DDP averages): the
    averaged parameter gradients equal those of the same model on the full batch on one device."""
    from gpu_util import Out, make_method, rel_err
    from torch.nn.parallel import DistributedDataParallel as DDP

    class Tiny(torch.nn.Module):
        def __init__(self, d_in=24, d=64):
            super().__init__()
            g = torch.Generator().manual_seed(5)
            self.w0 = torch.nn.Parameter(torch.randn(d_in, d, generator=g) * 0.2)
            self.w1 = torch.nn.Parameter(torch.randn(d, d, generator=g) * 0.2)
            self.w2 = torch.nn.Parameter(torch.randn(d, d, generator=g) * 0.2)

        def forward(self, x):
            h0 = x @ self.w0
            h1 = torch.tanh(h0) @ self.w1
            h2 = torch.tanh(h1) @ self.w2
            return h0, h1, h2

    meta = dict(modality="equal", layer_strategy="discounted", loss="mse", gamma=0.5, num_hidden_layers=3,
                layer=None, n_vis=256, coeff=1.0, cls=False, lang_coeff=None)
    B, txt = 3 * world, 6
    lo, hi = 3 * rank, 3 * rank + 3
    g = torch.Generator().manual_seed(9)
    x = torch.randn(B, 256 + txt, 24, generator=g)
    am = torch.zeros(B, txt, dtype=torch.int64)
    for b in range(B):
        am[b, txt - (1 + (5 * b) % txt):] = 1
    student, teacher = Tiny().cuda(), Tiny().cuda()
    with torch.no_grad():
        for p in teacher.parameters():
            p.add_(0.05)
        t_full = [h.detach() for h in teacher(x.cuda())]

    def grads_of(model, xs, teach, mask, group):
        fd = make_method(meta)
        fd.process_group = group
        fd.past_model = lambda **kw: Out(tuple(teach))
        model.zero_grad(set_to_none=True)
        loss = fd.distill(Out(model(xs)), {"attention_mask": mask})
        loss.backward()
        torch.cuda.synchronize()
        return loss.detach()

    ddp = DDP(student, device_ids=[torch.cuda.current_device()])
    loss_d = grads_of(ddp, x[lo:hi].cuda(), [h[lo:hi].contiguous() for h in t_full], am[lo:hi].cuda(), None)
    got = [p.grad.clone() for p in student.parameters()]
    single = Tiny().cuda()                                                   # same seeded weights, never wrapped
    loss_f = grads_of(single, x.cuda(), t_full, am.cuda(), False)            # the full batch on this GPU alone
    want = [p.grad.clone() for p in single.parameters()]
    e_loss = abs(float(loss_d) - float(loss_f)) / abs(float(loss_f))
    e_grad = max(rel_err(a.cpu(), b.cpu()) for a, b in zip(got, want))
    ok = e_loss < 1e-5 and e_grad < 1e-5
    print(f"rank {rank}: DDP parameter gradients vs full batch on one GPU: loss err {e_loss:.2e} grad err {e_grad:.2e} "
          f"{'OK' if ok else 'FAIL'}", flush=True)
    return ok


if __name__ == "__main__":
    main()
