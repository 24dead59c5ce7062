"""Load the committed golden vectors (made by tests/golden/make_golden.py from the reference)."""
import json
import os

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))


def digest(arrays):
    """sha256 of the arrays' bytes, in order: how a golden file pins the inputs it does not store."""
    import hashlib
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def case_inputs(i, m):
    """Inputs of golden case ``i``: regenerated from their seed (make_golden.py), as float32 arrays."""
    from oracle.distill_oracle import make_inputs
    dtype = torch.bfloat16 if m["dtype"] == "bf16" else torch.float32
    st, te, am = make_inputs(m["n_tuple"], m["bsz"], m["txt"], m["dim"], n_vis=m["n_vis"], dtype=dtype, seed=1000 + i,
                             teacher=m["teacher"], mask="ragged")
    return [s.float().numpy() for s in st], [t.float().numpy() for t in te], am


def load_cases():
    z = np.load(os.path.join(HERE, "golden", "distill_cases.npz"))
    meta = json.loads(str(z["meta"]))
    cases = []
    for i, m in enumerate(meta):
        dtype = torch.bfloat16 if m["dtype"] == "bf16" else torch.float32
        st, te, am = case_inputs(i, m)
        # the reference's outputs below were computed on exactly these inputs
        assert digest(st + te) == str(z[f"c{i}_inputs_sha256"]), f"golden case {i}: regenerated inputs differ"
        assert np.array_equal(am.numpy(), z[f"c{i}_mask"]), f"golden case {i}: regenerated mask differs"
        cases.append(dict(
            meta=m,
            students=[torch.from_numpy(a).to(dtype) for a in st],
            teachers=[torch.from_numpy(a).to(dtype) for a in te],
            mask=torch.from_numpy(z[f"c{i}_mask"]),
            loss=float(z[f"c{i}_loss"]),
            grad_layers=[int(x) for x in z[f"c{i}_grad_layers"]],
            grads=[torch.from_numpy(a) for a in z[f"c{i}_grads"]],
            logged_layers=[int(x) for x in z[f"c{i}_logged_layers"]],
            logged=[float(x) for x in z[f"c{i}_logged"]],
        ))
    return cases


def load_plans():
    with open(os.path.join(HERE, "golden", "layer_plans.json")) as f:
        return json.load(f)


def oracle_cfg(m):
    from oracle.distill_oracle import OracleConfig

    return OracleConfig(
        modality_strategy=m["modality"], layer_strategy=m["layer_strategy"], gamma=m["gamma"],
        num_hidden_layers=m["num_hidden_layers"], distillation_layer=m["layer"], distillation_coeff=m["coeff"],
        loss=m["loss"], cls_distillation=m["cls"], num_vision_tokens=m["n_vis"], lang_coeff=m["lang_coeff"])


def case_id(c):
    m = c["meta"]
    return "-".join(str(m[k]) for k in ("modality", "layer_strategy", "loss", "dtype")) + \
        (f"-L{m['layer']}" if m["layer"] is not None else "") + ("-cls" if m["cls"] else "") + \
        (f"-nv{m['n_vis']}" if m["n_vis"] != 8 else "") + (f"-g{m['grad_out']}" if m["grad_out"] != 1.0 else "")
