"""BASELINE.json's full sizes (C2, C3, C4 per-GPU shard, a C5 sweep point with text:vision 1:1): size-independent properties plus a plain
PyTorch fp32 restatement of the same op evaluated on the GPU layer by layer."""
import pytest
import torch

from gpu_util import Out, make_method, reference_forward_backward, rel_err
from mafed_b200 import cabi

pytestmark = pytest.mark.gpu

CONFIGS = {
    # name: (tuple_len, num_hidden_layers (ref rule L-1), B, txt, D)
    "C2-base-b128": (13, 11, 128, 32, 768),
    "C4-1b-shard-b64": (17, 15, 64, 32, 2048),
    "C3-410m-b256": (25, 23, 256, 32, 1024),
    # C5: 256 visual + 256 text tokens; 96 x 256 mask entries > 16 Ki -> counts from a prologue launch
    "C5-1b-b96-txt256": (17, 15, 96, 256, 2048),
}


def _inputs(cfg, dtype=torch.bfloat16, seed=1234, ragged=True):
    n_tuple, nh, B, txt, D = cfg
    g = torch.Generator(device="cuda").manual_seed(seed)
    st, te = [], []
    for i in range(n_tuple):
        if i >= nh:  # un-selected tail of the tuple: keep it tiny, the path must not touch it
            st.append(torch.zeros(1, device="cuda", dtype=dtype)); te.append(st[-1]); continue
        s = torch.randn(B, 256 + txt, D, generator=g, device="cuda", dtype=torch.float32)
        t = s + 0.1 * torch.randn(B, 256 + txt, D, generator=g, device="cuda", dtype=torch.float32)
        st.append(s.to(dtype)); te.append(t.to(dtype))
    am = torch.ones(B, txt, dtype=torch.int64, device="cuda")
    if ragged:
        for b in range(B):
            am[b, : txt - (1 + (7 * b) % txt)] = 0
    return st, te, am


def _run(meta, st, te, am, grad_out=1.0, variant=cabi.VARIANT_DEFAULT):
    with cabi.tuning(variant=variant):
        fd = make_method(meta)
        leaves = [s.detach().requires_grad_(True) for s in st]
        fd.past_model = lambda **kw: Out(tuple(te))
        loss = fd.distill(Out(tuple(leaves)), {"attention_mask": am})
        (loss * grad_out).backward()
        torch.cuda.synchronize()
        return loss.detach(), [l.grad for l in leaves], fd


def _torch_reference(meta, st, te, am, nh, gamma=0.5):
    """SURVEY 3.3 formulae with plain torch fp32 ops on the GPU (balanced / discounted / mse)."""
    B, txt = am.shape
    w_text = torch.cat([torch.zeros(B, 256, device="cuda"), am.float()], 1)
    w_vis = torch.cat([torch.ones(B, 256, device="cuda"), torch.zeros(B, txt, device="cuda")], 1)
    coeffs = torch.tensor([gamma ** d for d in range(nh, 0, -1)], dtype=torch.float64)
    coeffs = (coeffs / coeffs.sum()).tolist()
    total, grads = 0.0, []
    for l in range(nh):
        d = st[l].float() - te[l].float()
        D = d.shape[-1]
        tok = d.pow(2).sum(-1).double() / D
        lt = (tok * w_text).sum() / w_text.sum()
        lv = (tok * w_vis).sum() / w_vis.sum()
        total = total + coeffs[l] * (0.5 * lt + 0.5 * lv)
        row = coeffs[l] * 0.5 * (w_text / w_text.sum() + w_vis / w_vis.sum()) * 2.0 / D
        grads.append((d * row.float().unsqueeze(-1)))
    return float(total), grads


META = dict(modality="balanced", layer_strategy="discounted", loss="mse", gamma=0.5, layer=None, n_vis=256)


@pytest.mark.parametrize("name", list(CONFIGS))
@pytest.mark.parametrize("variant", [cabi.VARIANT_LDG, cabi.VARIANT_TMA], ids=["ldg", "tma"])
def test_fullsize_against_torch_fp32(name, variant):
    cfg = CONFIGS[name]
    nh = cfg[1]
    st, te, am = _inputs(cfg)
    loss, grads, _ = _run(dict(META, num_hidden_layers=nh), st, te, am, variant=variant)
    want, ref_grads = _torch_reference(META, st, te, am, nh)
    assert float(loss) == pytest.approx(want, rel=2e-3)       # bf16-input tolerance of the north_star
    assert float(loss) == pytest.approx(want, rel=1e-5)       # ... and in fact fp32-tight: inputs are exact in fp32
    for l in range(nh):
        assert rel_err(grads[l].float(), ref_grads[l]) < 2e-3
        # padded text rows are exactly zero
        pad = torch.cat([torch.zeros_like(am[:, :1]).expand(-1, 256), am], 1) == 0
        pad[:, :256] = False
        assert float(grads[l][pad].abs().max()) == 0.0
    assert all(g is None for g in grads[nh:])


def test_fullsize_properties_c4_shard():
    cfg = CONFIGS["C4-1b-shard-b64"]
    nh = cfg[1]
    meta = dict(META, num_hidden_layers=nh)
    st, te, am = _inputs(cfg)
    loss1, g1, _ = _run(meta, st, te, am)
    loss2, g2, _ = _run(meta, st, te, am)
    # bit-reproducible: no atomics anywhere in the reduction
    assert torch.equal(loss1, loss2) and all(torch.equal(a, b) for a, b in zip(g1[:nh], g2[:nh]))
    # linear in the upstream gradient (a power of two scales bf16 exactly)
    _, gh, _ = _run(meta, st, te, am, grad_out=0.5)
    assert all(torch.equal(a * 0.5, b) for a, b in zip(g1[:nh], gh[:nh]))
    # teacher == student: zero loss and zero gradient
    loss0, g0, _ = _run(meta, st, st, am)
    assert float(loss0) == 0.0 and all(float(g.abs().max()) == 0.0 for g in g0[:nh])
    # both kernel families agree
    la, ga, _ = _run(meta, st, te, am, variant=cabi.VARIANT_LDG)
    lb, gb, _ = _run(meta, st, te, am, variant=cabi.VARIANT_TMA)
    assert float(la) == pytest.approx(float(lb), rel=1e-6)
    assert all(rel_err(a.float(), b.float()) < 1e-3 for a, b in zip(ga[:nh], gb[:nh]))
    # loss is additive over layers: sum of logged layer losses x coefficients == total
    _, _, fd = _run(meta, st, te, am)
    coeffs = [float(fd.loss_weights.get_layer_loss_weight(l)) for l in range(nh)]
    per_layer = fd.last_layer_losses[:nh].double().cpu()
    assert float((per_layer * torch.tensor(coeffs, dtype=torch.float64)).sum()) == pytest.approx(float(loss1), rel=1e-6)


def test_offsets_beyond_2_gib_single_layer():
    """C5's largest per-layer tensor (B=1024, T=512, D=2048, bf16 = 2.1 GiB): byte offsets need 64 bits."""
    B, T, D = 1024, 512, 2048
    free, _ = torch.cuda.mem_get_info()
    if free < 12 * 2**30:
        pytest.skip("needs 12 GiB of free device memory")
    g = torch.Generator(device="cuda").manual_seed(3)
    s = torch.empty(B, T, D, device="cuda", dtype=torch.bfloat16)
    t = torch.empty_like(s)
    for i in range(0, B, 128):                                   # fill in slabs to bound temporaries
        x = torch.randn(128, T, D, generator=g, device="cuda")
        s[i:i + 128] = x.to(torch.bfloat16)
        t[i:i + 128] = (x + 0.1 * torch.randn(128, T, D, generator=g, device="cuda")).to(torch.bfloat16)
    del x
    am = torch.ones(B, T - 256, dtype=torch.int64, device="cuda")
    am[::3, :100] = 0
    meta = dict(modality="equal", layer_strategy="single", loss="mse", gamma=0.5, layer=0, n_vis=256, num_hidden_layers=1)
    for variant in (cabi.VARIANT_TMA, cabi.VARIANT_LDG):
        loss, grads, _ = _run(meta, [s], [t], am, variant=variant)
        # reference in slabs (fp64 accumulation of fp32 row sums)
        w = torch.cat([torch.ones(B, 256, device="cuda"), am.float()], 1)
        tot = torch.zeros((), dtype=torch.float64, device="cuda")
        for i in range(0, B, 128):
            d = s[i:i + 128].float() - t[i:i + 128].float()
            tot += (d.pow(2).sum(-1).double() * w[i:i + 128]).sum()
        want = float(tot / (D * w.sum().double()))               # "equal" weighting == mean over valid tokens
        assert float(loss) == pytest.approx(want, rel=1e-5)
        gscale = 2.0 / (D * float(w.sum()))
        for i in (0, 384, 896):                                  # spot-check slabs at the start, middle and end
            d = (s[i:i + 128].float() - t[i:i + 128].float()) * (gscale * w[i:i + 128]).unsqueeze(-1)
            assert rel_err(grads[0][i:i + 128].float(), d) < 2e-3
        assert float(grads[0][0, 256:356].abs().max()) == 0.0    # padded rows of sample 0
        del grads


@pytest.mark.parametrize("name", list(CONFIGS))
@pytest.mark.parametrize("loss_kind", ["mse", "cosine"])
def test_fullsize_against_the_reference_on_this_gpu(name, loss_kind):
    """BASELINE.json's shapes at full size against the reference's computation run on this GPU on the same tensors,
    under ``torch.autocast("cuda", bfloat16)`` as ``replay()`` runs it (``distillation.py:90``): loss, the per-layer
    values it logs, every gradient.  The unmodified reference where its files are present, otherwise its op-for-op
    restatement (``gpu_util.reference_forward_backward``)."""
    import gc

    cfg = CONFIGS[name]
    nh = cfg[1]
    free, _ = torch.cuda.mem_get_info()
    # inputs + the reference's fp32 temporaries kept for its backward (~6 fp32 copies of a layer, all layers alive)
    need = nh * cfg[2] * (256 + cfg[3]) * cfg[4] * (2 * 2 + 2 + 6 * 4)
    if free < 1.3 * need:
        pytest.skip(f"needs {1.3 * need / 2**30:.0f} GiB of free device memory")
    st, te, am = _inputs(cfg)
    meta = dict(META, num_hidden_layers=nh, loss=loss_kind)
    ref = reference_forward_backward(meta, st, te, am, autocast_bf16=True)
    ref_loss, ref_logged, ref_grads = float(ref["loss"]), dict(ref["logged"]), ref["grads"]
    del ref
    gc.collect()
    torch.cuda.empty_cache()
    loss, grads, mine = _run(meta, st, te, am)
    print(f"{name} {loss_kind}: loss {float(loss):.9g} reference {ref_loss:.9g} rel {abs(float(loss) - ref_loss) / abs(ref_loss):.2e}; "
          f"grad rel {max(rel_err(grads[l].float(), ref_grads[l].float()) for l in range(nh)):.2e}")
    assert float(loss) == pytest.approx(ref_loss, rel=2e-3)      # the north_star's bf16 tolerance ...
    # ... and in fact fp32-tight (exact widening, fp32 sums).  Measured on a B200: mse loss equal to 1e-7 with
    # bit-identical gradients at all four shapes; cosine 1-6e-6 (the reference forms 1 - cos ~ 0.005 in fp32) and 7e-5
    tight = 2e-5 if loss_kind == "mse" else 5e-5
    assert float(loss) == pytest.approx(ref_loss, rel=tight)
    got = mine.layer_loss_dict()
    assert sorted(got) == sorted(ref_logged)
    for k, v in ref_logged.items():
        assert got[k] == pytest.approx(v, rel=tight)
    for l in range(nh):
        assert grads[l].dtype == ref_grads[l].dtype == torch.bfloat16
        assert rel_err(grads[l].float(), ref_grads[l].float()) < 2e-3
        ref_grads[l] = None
    assert all(g is None for g in grads[nh:]) and all(g is None for g in ref_grads[nh:])
