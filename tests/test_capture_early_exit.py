"""HiddenStateCapture(stop_after_last=True) on HF GPTNeoXModel and the tiny VL model (CPU): the captured entries are
the full forward's own, nothing after the highest captured entry runs, and only the capture's own stop is swallowed."""
import pytest
import torch

from mafed_b200.capture import HiddenStateCapture

L = 4


def _neox():
    from transformers import GPTNeoXConfig, GPTNeoXModel
    cfg = GPTNeoXConfig(hidden_size=32, num_hidden_layers=L, num_attention_heads=4, intermediate_size=64,
                        vocab_size=128, max_position_embeddings=64, hidden_dropout=0.0, attention_dropout=0.0)
    torch.manual_seed(0)
    return GPTNeoXModel(cfg).eval()


def _tiny_vl():
    from tiny_vl import TinyVL, make_batch
    torch.manual_seed(0)
    return TinyVL(layers=L).eval(), make_batch()


def _count_completed(modules):
    """Forward (post) hooks: a module is listed once its forward has returned."""
    ran, handles = [], []
    for name, m in modules.items():
        handles.append(m.register_forward_hook(lambda mod, args, out, name=name: ran.append(name)))
    return ran, handles


def _decoder_modules(decoder, head=None):
    mods = {f"layer{i}": layer for i, layer in enumerate(decoder.layers)}
    mods["final_layer_norm"] = decoder.final_layer_norm
    if head is not None:
        mods["head"] = head
    return mods


def _expected_ran(stop):
    """What completes when the forward stops at entry ``stop``: layers 0..stop-1, and for entry L the final norm (never
    the LM head)."""
    return [f"layer{i}" for i in range(min(stop, L))] + (["final_layer_norm"] if stop == L else [])


@pytest.mark.parametrize("layers", [[0], [2], [L - 1], [L], [0, 2, L - 1], [1, L]],
                         ids=["first", "middle", "last-layer-input", "final-norm", "several", "with-final-norm"])
def test_gpt_neox_stops_after_the_highest_entry(layers):
    model = _neox()
    embeds = torch.randn(2, 10, 32)
    with torch.no_grad():
        full = model(inputs_embeds=embeds, output_hidden_states=True).hidden_states
    ran, counting = _count_completed(_decoder_modules(model))
    after = []
    with torch.no_grad(), HiddenStateCapture(model, layers, stop_after_last=True) as cap:
        model(inputs_embeds=embeds)
        after.append("returned")                    # not reached: the forward was stopped
    assert not after
    assert ran == _expected_ran(max(layers))
    assert sorted(cap.states) == sorted(layers)
    for i in layers:
        assert torch.equal(cap.hidden_states[i], full[i]), i
    # the capture's hooks are gone: a second forward runs to the end and records nothing
    cap.states.clear()
    ran.clear()
    with torch.no_grad():
        model(inputs_embeds=embeds)
    assert not cap.states and ran == [f"layer{i}" for i in range(L)] + ["final_layer_norm"]
    for h in counting:
        h.remove()


@pytest.mark.parametrize("stop", [0, 2, L - 1, L])
def test_tiny_vl_stops_before_the_lm_head(stop):
    model, batch = _tiny_vl()
    batch.pop("labels")
    with torch.no_grad():
        full = model(**batch, output_hidden_states=True).hidden_states
    ran, counting = _count_completed(_decoder_modules(model.gpt_neox, head=model.embed_out))
    with torch.no_grad(), HiddenStateCapture(model, [0, stop], stop_after_last=True) as cap:
        model(**batch)
    assert ran == _expected_ran(stop)       # the LM head never runs
    for i in {0, stop}:
        assert torch.equal(cap.hidden_states[i], full[i]), i
    ran.clear()
    with torch.no_grad():
        model(**batch)
    assert ran[-2:] == ["final_layer_norm", "head"]
    for h in counting:
        h.remove()


def test_stopped_student_states_stay_in_the_autograd_graph():
    model, batch = _tiny_vl()
    batch.pop("labels")
    full = model(**batch, output_hidden_states=True).hidden_states
    full[2].pow(2).mean().backward()
    want = {n: p.grad.clone() for n, p in model.named_parameters() if p.grad is not None}
    model.zero_grad(set_to_none=True)
    with HiddenStateCapture(model, [1, 2], stop_after_last=True) as cap:
        model(**batch)
    h = cap.hidden_states[2]
    assert h.requires_grad and h.grad_fn is not None
    h.pow(2).mean().backward()
    got = {n: p.grad for n, p in model.named_parameters() if p.grad is not None}
    assert got.keys() == want.keys() and all(torch.equal(got[n], want[n]) for n in want)
    assert model.gpt_neox.layers[2].attention.query_key_value.weight.grad is None     # layer 2 comes after state 2


def test_other_exceptions_propagate_and_hooks_are_removed():
    model = _neox()
    boom = RuntimeError("raised inside the forward")

    def fail(module, args):
        raise boom

    handle = model.layers[1].register_forward_pre_hook(fail)
    with pytest.raises(RuntimeError) as info:
        with torch.no_grad(), HiddenStateCapture(model, [0, 3], stop_after_last=True) as cap:
            model(inputs_embeds=torch.randn(1, 6, 32))
    assert info.value is boom
    assert sorted(cap.states) == [0] and not cap._handles
    handle.remove()
    # an exception raised in the body of the block propagates too
    with pytest.raises(KeyError):
        with HiddenStateCapture(model, [2], stop_after_last=True):
            raise KeyError("not a stop")
    # a stop belongs to the capture that raised it: an inner capture does not swallow the outer one's
    with torch.no_grad(), HiddenStateCapture(model, [1], stop_after_last=True) as outer:
        with HiddenStateCapture(model, [3], stop_after_last=True) as inner:
            model(inputs_embeds=torch.randn(1, 6, 32))
        raise AssertionError("the outer capture's stop was swallowed by the inner one")
    assert sorted(outer.states) == [1] and not inner.states


def test_without_the_flag_the_forward_runs_to_the_end():
    model = _neox()
    ran, counting = _count_completed(_decoder_modules(model))
    with torch.no_grad(), HiddenStateCapture(model, [1]) as cap:
        out = model(inputs_embeds=torch.randn(1, 6, 32))
    assert out is not None and ran[-1] == "final_layer_norm" and sorted(cap.states) == [1]
    for h in counting:
        h.remove()
