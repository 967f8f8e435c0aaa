"""Multi-process check of partitioned GraphNCF training (run under torchrun; not collected by pytest):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port 29517 tests/mp_peer_train_check.py

Every rank builds the same graph, maps the peers' arenas (CUDA IPC) with a gradient section and runs 3 training steps (sum-MSE,
Adam(fused=True)) through forward_peer + loss.backward(), with an eval forward after each step, for two models:

    dot   dot-product head, no dropout: at every step the gradients are within 1e-5 (max-norm relative, per parameter) of the single-GPU
          gradients at the same parameters (GraphNCF's propagation under autograd), and after the 3 steps the parameters are within 1e-5 of
          a single-GPU run's.  (The MLP head is left out of this comparison: a ReLU input within rounding of 0 switches a unit on in one
          run and off in the other, and Adam turns such differences of near-zero gradient elements into larger ones.)
    mlp   MLP [256, 128] with dropout 0.2 (conv dropout drawn by the owners, MLP dropout by the shard's generator).

For both, the parameters must be bit-identical on all ranks after every step.  With B200REC_PEER_CHECK_SAME_GPU=1 all ranks use cuda:0 and
rendezvous over gloo (the single-GPU test-suite runs it that way); otherwise one GPU per rank over NCCL.  Rank 0 prints one JSON line."""
import copy
import json
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def single_dot(model, g, uid, iid):
    """single-GPU training forward of a dot-product GraphNCF under autograd (GraphNCF.forward's row dot carries no gradient)"""
    from deeprecommendation_b200.graph import get_index
    index = get_index(g)
    skip, dinv = index.masked(index.positions(uid, iid))
    comb = model._encode(g, index, skip, dinv, True)
    return (comb[uid] * comb[iid]).sum(1, keepdim=True)


def main():
    from deeprecommendation_b200 import synth
    from deeprecommendation_b200.graph import IdTable, create_graph
    from deeprecommendation_b200.neural_collaborative_filtering.models import GraphNCF
    from deeprecommendation_b200.parallel import partition_graph
    from deeprecommendation_b200.peer import forward_peer, grad_floats
    same = os.environ.get('B200REC_PEER_CHECK_SAME_GPU') == '1'
    local = 0 if same else int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if same:
        dist.init_process_group('gloo')
    else:
        dist.init_process_group('nccl', device_id=dev)
    rank, world = dist.get_rank(), dist.get_world_size()
    n_users, n_items, n, F, d = (3000, 1200, 100_000, 48, 64) if same else (20000, 8000, 1_500_000, 64, 128)
    users, items, ratings = synth.interactions_zipf(n_users, n_items, n, seed=21)
    rng = np.random.default_rng(4)
    fi, fu = rng.standard_normal((n_items, F)).astype(np.float32), rng.standard_normal((n_users, F)).astype(np.float32)
    g = create_graph(torch.from_numpy(users).to(dev), torch.from_numpy(items).to(dev), torch.from_numpy(ratings).to(dev),
                     torch.from_numpy(fi).to(dev), torch.from_numpy(fu).to(dev),
                     IdTable(torch.arange(n_users, device=dev)), IdTable(torch.arange(n_items, device=dev)))
    pg = None
    info, ok = {}, True
    for name, mlp, dropout in (('dot', None, 0.0), ('mlp', [256, 128], 0.2)):
        kw = dict(item_dim=F, user_dim=F, num_gnn_layers=2, hetero=True, node_emb=d, mlp_dense_layers=mlp or [8], dropout_rate=dropout,
                  use_dot_product=mlp is None)
        m = GraphNCF(**kw).to(dev).train()
        m.load_state_dict(synth.to_torch(synth.graph_ncf_weights(seed=5, **kw)))
        ref, probe = copy.deepcopy(m), copy.deepcopy(m)
        opt, ref_opt = (torch.optim.Adam(x.parameters(), lr=1e-3, fused=True) for x in (m, ref))
        if pg is None:
            pg = partition_graph(g, scheme='peer', d_max=d, batch_max=1024, grad_floats=grad_floats(m))
        errs, gerr, same_bits = [], [], True
        for step in range(3):
            pick = torch.from_numpy(rng.permutation(n)[:1000]).to(dev)
            uid, iid = g.user2item_edge_index[0][pick].contiguous(), g.user2item_edge_index[1][pick].contiguous()
            y = torch.from_numpy(np.random.default_rng(step).standard_normal((1000, 1)).astype(np.float32)).to(dev)
            opt.zero_grad(set_to_none=True)
            ((forward_peer(m, pg, uid, iid) - y) ** 2).sum().backward()
            if mlp is None:
                probe.load_state_dict(m.state_dict())          # the single-GPU gradient at the same parameters
                ((single_dot(probe, g, uid, iid) - y) ** 2).sum().backward()
                pp = dict(probe.named_parameters())
                gerr.append(max(float((p.grad - pp[k].grad).abs().max() / pp[k].grad.abs().max()) for k, p in m.named_parameters()))
                probe.zero_grad(set_to_none=True)
                ref_opt.zero_grad(set_to_none=True)
                ((single_dot(ref, g, uid, iid) - y) ** 2).sum().backward()
                ref_opt.step()
            opt.step()
            m.eval()
            with torch.no_grad():
                forward_peer(m, pg, uid, iid)              # an inference call between training steps, on the same epoch counters
            m.train()
            torch.cuda.synchronize()
            pg.check()
            flat = torch.cat([p.detach().view(-1) for p in m.parameters()]).cpu()
            all_flat = [None] * world
            dist.all_gather_object(all_flat, flat)
            same_bits = same_bits and all(torch.equal(f, all_flat[0]) for f in all_flat)
        if mlp is None:
            rp = dict(ref.named_parameters())
            errs.append(max(float((p.detach() - rp[k].detach()).abs().max() / rp[k].detach().abs().max()) for k, p in m.named_parameters()))
        info[name] = {'bit_identical': same_bits, 'grad_err': gerr, 'param_err': errs}
        ok = ok and same_bits and all(e < 1e-5 for e in gerr) and all(e < 1e-5 for e in errs)
    oks = [None] * world
    dist.all_gather_object(oks, (ok, info))
    if rank == 0:
        print(json.dumps({'world': world, 'same_gpu': same, 'ok': all(o[0] for o in oks), 'per_rank': [o[1] for o in oks]}),
              flush=True)
    dist.destroy_process_group()
    if not ok:
        sys.exit(1)


if __name__ == '__main__':
    main()
