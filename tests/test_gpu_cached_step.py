"""The one-pass step reading the teacher straight from the teacher cache (``libmafed_cached_step.so``) on the GPU: every
result bit-identical to ``mafed_teacher_gather`` followed by the ordinary step on the gathered tensors, the fix-up
backward, the replay step of the tiny VL model, which launches run and the memory the gathered copy took."""
import copy

import pytest
import torch
from torch.nn.attention import SDPBackend, sdpa_kernel

from mafed_b200 import cabi
from mafed_b200 import teacher_cache as TC
from mafed_b200.distill_op import DistillPlan, cached_distill_loss, distill_loss, seen_slot

pytestmark = pytest.mark.gpu

F32, BF16, F16 = torch.float32, torch.bfloat16, torch.float16


def _bitwise(a, b):
    if a is None or b is None:
        return a is None and b is None
    bits = {8: torch.int64, 4: torch.int32, 2: torch.int16}[a.element_size()]
    return a.shape == b.shape and a.dtype == b.dtype and torch.equal(a.contiguous().view(bits), b.contiguous().view(bits))


def _inputs(L, B, T, T_c, M, D, n_vis, s_dtype, t_dtype, ragged, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    students = [torch.randn((B, T, D), generator=g, device="cuda").to(s_dtype) for _ in range(L)]
    cache = [torch.randn((M, T_c, D), generator=g, device="cuda").to(t_dtype) for _ in range(L)]
    txt = T - n_vis
    if ragged:
        lens = torch.randint(0, txt + 1, (B,), generator=g, device="cuda")
        mask = (torch.arange(txt, device="cuda")[None, :] >= (txt - lens)[:, None]).to(torch.int64)
    else:
        mask = torch.ones((B, txt), dtype=torch.int64, device="cuda")
    return students, cache, mask


def _plan(L, loss, n_vis, table, seed):
    g = torch.Generator().manual_seed(seed)
    coeffs = (torch.rand(L, generator=g) + 0.1).tolist()
    lang = (torch.rand(L, generator=g)).tolist() if table else None
    return DistillPlan(layers=list(range(L)), layer_coeffs=coeffs, distill_coeff=1.5,
                       modality_kind=cabi.MODW_TABLE if table else cabi.MODW_EQUAL, lang_weights=lang,
                       loss_kind=cabi.LOSS_COSINE if loss == "cosine" else cabi.LOSS_MSE, n_vis=n_vis)


def _run(students, plan, mask, upstream, cache=None, idx=None, T_c=None, teachers=None):
    leaves = [s.clone().requires_grad_(True) for s in students]
    seen = seen_slot()
    if cache is not None:
        res = cached_distill_loss(leaves, cache, idx, T_c, mask, plan, mask_out=True, seen=seen, return_masks=True)
        assert res is not None, "the cached step refused a shape it should take"
    else:
        res = distill_loss(leaves, teachers, mask, plan, mask_out=True, seen=seen, return_masks=True)
    total, aux, masks = res
    (total * upstream).backward()
    torch.cuda.synchronize()
    return dict(total=total.detach().clone(), aux=aux.clone(), masks=masks, grads=[l.grad for l in leaves],
                seen=float(seen[0]))


def _same(a, b):
    assert _bitwise(a["total"], b["total"]), (float(a["total"]), float(b["total"]))
    assert _bitwise(a["aux"], b["aux"])
    assert _bitwise(a["masks"][0], b["masks"][0]) and _bitwise(a["masks"][1], b["masks"][1])
    for ga, gb in zip(a["grads"], b["grads"]):
        assert _bitwise(ga, gb)
    assert a["seen"] == b["seen"]


# (L, B, T, T_c, M, D, n_vis, student, teacher, loss, ragged, table): tiles straddle the visual / text boundary and the
# samples (n_vis and T not multiples of the tile rows), T == T_c and T < T_c, B = 1, the unrolled cosine rows
# (96 / 128 / 192 chunks), more than 64 layers, rows of 32 KB
CASES = [
    (3, 6, 13, 13, 9, 64, 5, F32, F32, "mse", True, True),
    (3, 6, 13, 17, 9, 64, 5, F32, F32, "cosine", True, False),
    (2, 5, 37, 41, 11, 768, 29, BF16, BF16, "cosine", True, True),       # 96 chunks
    (2, 5, 37, 37, 11, 1024, 29, BF16, BF16, "cosine", False, False),    # 128 chunks
    (2, 3, 21, 30, 7, 1536, 13, F16, F16, "cosine", True, True),        # 192 chunks
    (2, 4, 19, 25, 7, 768, 11, F32, F32, "cosine", True, False),        # 192 chunks in fp32
    (4, 7, 23, 31, 10, 256, 17, BF16, BF16, "mse", True, True),
    (4, 7, 23, 23, 10, 256, 17, F16, F16, "mse", False, False),
    (3, 5, 19, 24, 8, 512, 9, F32, BF16, "mse", True, True),
    (3, 5, 19, 24, 8, 512, 9, F32, F16, "cosine", True, False),
    (2, 5, 19, 19, 8, 1024, 9, F32, BF16, "cosine", False, True),
    (1, 1, 12, 20, 3, 128, 4, BF16, BF16, "mse", True, False),           # B = 1
    (70, 3, 11, 14, 5, 64, 6, BF16, BF16, "mse", True, True),          # two launches of <= 64 layers
    (2, 3, 9, 12, 4, 8192, 5, F32, F32, "mse", True, False),            # 32 KB rows
    (2, 3, 9, 9, 4, 16384, 5, BF16, BF16, "cosine", True, True),        # 32 KB rows
]


@pytest.mark.parametrize("case", range(len(CASES)))
def test_cached_step_is_bit_identical_to_gather_then_step(case):
    L, B, T, T_c, M, D, n_vis, sd, td, loss, ragged, table = CASES[case]
    students, cache, mask = _inputs(L, B, T, T_c, M, D, n_vis, sd, td, ragged, seed=100 + case)
    idx = [(5 * b + 3) % M for b in range(B)]
    if B > 2:
        idx[1] = idx[0]                     # a sample drawn twice
    plan = _plan(L, loss, n_vis, table, seed=case)
    gathered = TC.gather(cache, idx, T, n_vis)
    for upstream in (1.0, 0.375):           # the assumed upstream gradient, then one the fix-up has to correct
        a = _run(students, plan, mask, upstream, cache=cache, idx=idx, T_c=T_c)
        b = _run(students, plan, mask, upstream, teachers=gathered)
        _same(a, b)
        assert a["seen"] == upstream


def test_cached_and_ordinary_steps_interleave_on_one_stream():
    L, B, T, T_c, M, D, n_vis = 3, 6, 40, 48, 12, 512, 31
    students, cache, mask = _inputs(L, B, T, T_c, M, D, n_vis, BF16, BF16, True, seed=7)
    plan = _plan(L, "mse", n_vis, True, seed=3)
    runs = []
    for k in range(4):                       # no synchronisation between the steps and their backwards
        idx = [(k + 3 * b) % M for b in range(B)]
        leaves = [s.clone().requires_grad_(True) for s in students]
        if k % 2 == 0:
            total, aux = cached_distill_loss(leaves, cache, idx, T_c, mask, plan)
        else:
            total, aux = distill_loss(leaves, TC.gather(cache, idx, T, n_vis), mask, plan)
        (total * (0.5 if k == 2 else 1.0)).backward()
        runs.append((idx, total, aux, [l.grad for l in leaves], 0.5 if k == 2 else 1.0))
    torch.cuda.synchronize()
    for idx, total, aux, grads, up in runs:
        want = _run(students, plan, mask, up, teachers=TC.gather(cache, idx, T, n_vis))
        assert _bitwise(total.detach(), want["total"]) and _bitwise(aux, want["aux"])
        for g, w in zip(grads, want["grads"]):
            assert _bitwise(g, w)


def test_qualifying_step_does_not_gather_and_saves_the_gathered_bytes():
    L, B, T, T_c, M, D, n_vis = 8, 32, 288, 300, 64, 1024, 256
    students, cache, mask = _inputs(L, B, T, T_c, M, D, n_vis, BF16, BF16, True, seed=11)
    plan = _plan(L, "mse", n_vis, True, seed=5)
    idx = list(range(0, 2 * B, 2))
    leaves = [s.clone().requires_grad_(True) for s in students]

    def cached():
        total, _ = cached_distill_loss(leaves, cache, idx, T_c, mask, plan)
        total.backward()

    def gathered():
        total, _ = distill_loss(leaves, TC.gather(cache, idx, T, n_vis), mask, plan)
        total.backward()

    peaks = {}
    for name, fn in (("cached", cached), ("gathered", gathered)):
        for l in leaves:
            l.grad = None
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        fn()
        torch.cuda.synchronize()
        peaks[name] = torch.cuda.max_memory_allocated() - base
    copy_bytes = L * B * T * D * 2
    assert peaks["gathered"] - peaks["cached"] >= 0.95 * copy_bytes, (peaks, copy_bytes)

    for fn, want in ((cached, False), (gathered, True)):
        with _launches() as seen:
            fn()
        assert seen["gather"] == (1 if want else 0) and seen["cached"] == (0 if want else 1)


def test_steps_the_cached_library_does_not_take_return_none():
    L, B, T, T_c, M, D, n_vis = 2, 3, 12, 14, 5, 64, 5
    students, cache, mask = _inputs(L, B, T, T_c, M, D, n_vis, F32, F32, True, seed=1)
    leaves = [s.clone().requires_grad_(True) for s in students]
    idx = [0, 1, 2]
    assert cached_distill_loss(leaves, cache, idx, T_c, mask, _plan(L, "mse", n_vis, False, 0)) is not None
    two_pass = _plan(L, "mse", n_vis, False, 0)
    two_pass.single_pass = False
    assert cached_distill_loss(leaves, cache, idx, T_c, mask, two_pass) is None
    with cabi.tuning(variant=cabi.VARIANT_LDG):
        assert cached_distill_loss(leaves, cache, idx, T_c, mask, _plan(L, "mse", n_vis, False, 0)) is None
    odd = [torch.randn((M, T_c, 63), device="cuda") for _ in range(L)]            # rows of 252 bytes: LDG / generic
    assert cached_distill_loss([torch.randn((B, T, 63), device="cuda", requires_grad=True) for _ in range(L)], odd,
                               idx, T_c, mask, _plan(L, "mse", n_vis, False, 0)) is None
    half = [c.to(BF16) for c in cache]                                           # a bf16 student, fp32 teacher
    assert cached_distill_loss([l.detach().to(BF16).requires_grad_(True) for l in leaves], cache, idx, T_c, mask,
                               _plan(L, "mse", n_vis, False, 0)) is None
    assert cached_distill_loss(leaves, half, idx, T_c, mask, _plan(L, "mse", n_vis, False, 0)) is not None
    with torch.no_grad():
        assert cached_distill_loss(leaves, cache, idx, T_c, mask, _plan(L, "mse", n_vis, False, 0)) is None


# ---------------------------------------------------------------- the replay step of the tiny VL model
class _launches:
    """Counts the launches of the gather kernel (``teacher_cache.gather_raw``, its only caller) and of the cached step
    (``distill_cached`` of the extension) inside the block.  (Counted at the call, not with torch.profiler: many CUPTI
    sessions in one process make later profiles of the suite lose kernels.)"""

    def __enter__(self):
        from mafed_b200 import node
        self.ext, self.counts = node.load_cached(), {"gather": 0, "cached": 0}
        self.raw, self.step = TC.gather_raw, self.ext.distill_cached

        def raw(*a, **k):
            self.counts["gather"] += 1
            return self.raw(*a, **k)

        def step(*a, **k):
            self.counts["cached"] += 1
            return self.step(*a, **k)

        TC.gather_raw, self.ext.distill_cached = raw, step
        return self.counts

    def __exit__(self, *exc):
        TC.gather_raw, self.ext.distill_cached = self.raw, self.step
        return False


def _replay(fd, student, batch):
    model = copy.deepcopy(student)
    fd.mem_dataloader = [batch]
    with sdpa_kernel([SDPBackend.MATH]), _launches() as seen:
        loss, _ = fd.replay(model)
        loss.backward()
        torch.cuda.synchronize()
    return dict(loss=loss.detach().clone(), grads={n: p.grad for n, p in model.named_parameters()}, batch=batch,
                gathered=seen["gather"] > 0, fused=seen["cached"] > 0)


@pytest.mark.parametrize("kw,fused", [
    (dict(), True),
    (dict(loss="cosine"), True),
    (dict(teacher_dtype=torch.bfloat16, num_hidden_layers=4), True),
    (dict(single_pass=False), False),
    (dict(loss="cosine", cls_distillation=True), False),
])
def test_replay_takes_the_cached_step_where_it_qualifies(kw, fused, monkeypatch):
    from test_gpu_teacher_cache import Opts, _models, _strategy, _wandb
    from vl_memory import VLSamples
    logged = _wandb(monkeypatch)
    student, teacher = _models()
    kw = dict(kw)
    cfg = dict(modality="balanced", strategy="discounted", **kw)
    fd = _strategy(True, **cfg)
    fd.update(dataset=VLSamples(40, seed=1, max_txt=9), model=teacher, dataloader=None)
    cache = fd._teacher_cache
    ref = _strategy(False, **cfg)
    ref.task_id, ref.past_model, ref.loss_weights = fd.task_id, fd.past_model, fd.loss_weights
    idx = None

    def gathered(batch, layers):
        batch.pop("labels", None)
        return TC.reference_gather(cache.states, idx, batch["attention_mask"].shape[1] + 8, 8)

    ref._past_states = gathered
    for drawn in fd.mem_dataloader:
        idx = drawn["memory_index"]
        logged.clear()
        a = _replay(fd, student, {k: (v.clone() if torch.is_tensor(v) else v) for k, v in drawn.items()})
        fd.flush_logs()
        la = list(logged)
        logged.clear()
        b = _replay(ref, student, {k: (v.clone() if torch.is_tensor(v) else v) for k, v in drawn.items()
                                   if k != "memory_index"})
        ref.flush_logs()
        assert a["fused"] == fused and a["gathered"] == (not fused)
        assert torch.equal(a["loss"], b["loss"])
        for n, g in b["grads"].items():
            assert _bitwise(a["grads"][n], g), n
        for k in ("lang_masks", "image_masks"):
            if k in b["batch"]:
                assert torch.equal(a["batch"][k], b["batch"][k]), k
        assert la == list(logged)
    assert Opts.batch_size == 4
