"""`adaptive` importances over batch shards on the GPU: without a group the pass is today's, bit for bit; on >= 2 GPUs
``tools/multirank_check.py --adaptive`` over the peer communicator and over NCCL."""
import ctypes
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _abi_sums(tensors, mask, n_vis):
    """The token-norm pass as the C ABI calls it without any exchange: the pass, then REDUCE|COUNTS."""
    from mafed_b200 import cabi
    lib = cabi.load()
    B, T, D = tensors[0].shape
    shape = cabi.make_shape(len(tensors), B, T, n_vis, D, {torch.float32: cabi.F32, torch.bfloat16: cabi.BF16}[
        tensors[0].dtype], cabi.LOSS_MSE)
    ws = torch.empty(lib.mafed_distill_ws_bytes(len(tensors)), dtype=torch.uint8, device="cuda")
    sums = torch.empty(2 * len(tensors) + 2, dtype=torch.float64, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    cabi.check(lib.mafed_distill_token_norm_sums(ctypes.byref(shape), cabi.ptr_array([t.data_ptr() for t in tensors]),
                                                 mask.data_ptr(), ws.data_ptr(), stream), "token_norm_sums")
    cabi.check(lib.mafed_distill_scalar_stage(ctypes.byref(shape), None, cabi.STAGE_REDUCE | cabi.STAGE_COUNTS,
                                              mask.data_ptr(), ws.data_ptr(), sums.data_ptr(), None, None, None, 0,
                                              stream), "reduce")
    return sums


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_token_norm_sums_without_group_is_the_plain_pass(dtype):
    from mafed_b200.distill_op import token_norm_sums
    g = torch.Generator(device="cuda").manual_seed(9)
    B, txt = 5, 11
    grads = [(torch.randn(B, 256 + txt, 1024, generator=g, device="cuda") * (1 + l)).to(dtype) for l in range(3)]
    am = torch.ones(B, txt, dtype=torch.int64, device="cuda")
    for b in range(B):
        am[b, : (2 * b) % txt] = 0
    want = _abi_sums(grads, am, 256)
    assert torch.equal(token_norm_sums(grads, am, 256), want)
    assert torch.equal(token_norm_sums(grads, am, 256, group=False), want)
    # several dtypes: one pass per dtype, the rows in the caller's order, the counts of the last pass
    mixed = grads[:2] + [grads[2].float() if dtype != torch.float32 else grads[2].bfloat16()]
    got = token_norm_sums(mixed, am, 256, group=False)
    assert torch.equal(got, token_norm_sums(mixed, am, 256))
    assert torch.equal(got[:4], _abi_sums(mixed[:2], am, 256)[:4])
    assert torch.equal(got[4:], _abi_sums(mixed[2:], am, 256))


def test_compute_adaptive_weights_without_group_is_unchanged():
    from mafed_b200.distill_op import token_norm_sums
    from mafed_b200.methods import DistillationWeights
    from tiny_vl import TinyVL, make_batch
    torch.manual_seed(0)
    model = TinyVL().cuda()
    model.gpt_neox.config._attn_implementation = "eager"    # SDPA's memory-efficient backward adds with atomics
    batches = [make_batch(bsz=3 + i, seed=20 + i, device="cuda") for i in range(3)]
    dw = DistillationWeights("adaptive", "discounted", num_hidden_layers=3, distillation_layer=None, num_vision_tokens=8)
    default = dw.compute_adaptive_weights(model, [dict(b) for b in batches])
    off = dw.compute_adaptive_weights(model, [dict(b) for b in batches], process_group=False)
    # the pass as it read before the option: one token_norm_sums per batch, then the ratio
    running = None
    for batch in batches:
        with torch.autocast("cuda", dtype=torch.bfloat16):
            out = model(**batch, compute_loss=True, output_hidden_states=True, allow_input_gradients=True)
        grads = torch.autograd.grad(out.loss, [out.hidden_states[l] for l in range(3)])
        now = token_norm_sums(grads, batch["attention_mask"], 8)
        running = now if running is None else running + now
    sums = running[:6].reshape(3, 2)
    lang, image = (sums[:, 0] / running[6]).float(), (sums[:, 1] / running[7]).float()
    want = lang / (lang + image)
    assert torch.equal(default, want) and torch.equal(off, want)
    assert torch.equal(dw.gradient_norm_sums(model, [dict(b) for b in batches], process_group=False), running)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
@pytest.mark.parametrize("path", ["peer", "nccl"])
def test_adaptive_importances_sharded_equal_one_gpu(path):
    n = min(torch.cuda.device_count(), 8)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}",
           "--master-addr", "127.0.0.1", "--master-port", "29527", os.path.join(ROOT, "tools", "multirank_check.py"),
           "--adaptive"]
    env = dict(os.environ, MAFED_B200_DIST=path)
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
