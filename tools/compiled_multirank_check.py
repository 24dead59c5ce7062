#!/usr/bin/env python
"""Batch-sharded step under torch.compile equals the eager sharded step, bit for bit, on every rank (peer-memory
communicator).  One process per GPU:

    python -m torch.distributed.run --nproc-per-node=2 tools/compiled_multirank_check.py
"""
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    rank = dist.get_rank()
    from mafed_b200 import cabi, node
    from mafed_b200.comm import get_peer_comm
    from mafed_b200.distill_op import DistillPlan, distill_loss
    from oracle import distill_oracle as O
    node.load()
    assert get_peer_comm(None) is not None, "no peer-memory communicator"
    st, te, am = O.make_inputs(3, 4, 9, 1024, n_vis=256, dtype=torch.bfloat16, seed=90 + rank)
    st, te, am = [s.cuda() for s in st], [t.cuda() for t in te], am.cuda()
    for single_pass in (True, False):
        plan = DistillPlan(layers=[0, 1, 2], layer_coeffs=[1.0, 0.5, 0.25], modality_kind=cabi.MODW_TABLE,
                           lang_weights=[0.4, 0.5, 0.6], single_pass=single_pass, grad_multiplier=2.0)

        def f(students):
            return distill_loss(students, te, am, plan)

        results = []
        for fn in (f, torch.compile(f, fullgraph=True)):
            leaves = [s.detach().clone().requires_grad_(True) for s in st]
            total, aux = fn(leaves)
            total.backward()
            torch.cuda.synchronize()
            results.append((total.detach().clone(), aux.clone(), [l.grad for l in leaves]))
        (et, ea, eg), (ct, ca, cg) = results
        assert torch.equal(et, ct) and torch.equal(ea, ca), (rank, single_pass, et, ct)
        for a, b in zip(eg, cg):
            assert torch.equal(a, b), (rank, single_pass)
        torch._dynamo.reset()
    print(f"rank {rank}: compiled sharded step == eager sharded step")
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
