"""Per-rank build of a user-partitioned graph that does NOT fit (or is not wanted) on one GPU — BASELINE configs[4]:
10^7 users x 10^6 items x 10^9 edges on the 8 GPUs of a box (SURVEY.md §8e).

`peer.shard_from_full` cuts a rank's shard out of the full neighbour index, which every rank builds — fine at 5x10^7 directed edges, not at
2x10^9.  Here a rank only ever sees the interactions of ITS users (`users_r0 .. users_r0 + n_local`):

    create_graph semantics (src/content_providers/graph_providers.py:10-66) over the local interactions, in a LOCAL node space
    (items 0..nI-1, local users nI..), with the two quantities that depend on other ranks' interactions made global by one collective
    each at BUILD time (plumbing, not the data path):
        item rating count / sum  -> item means -> item->user edge attrs  (graph_providers.py:17,41-45)      all-reduce of (nI,) int + fp64
        item in-degree           -> deg^-1/2 of the item rows             (gnn_ncf.py:47-50)                 all-reduce of (nI,) int
    user means / degrees are local (all interactions of a user live on its owner).

The result is a `peer.PeerShard` with the same fields as `shard_from_full` produces; `peer.forward_peer` runs on it unchanged.
tests/test_peer_gpu.py checks that this build and `shard_from_full` give the same shard.
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib as L
from .graph import GraphData, GraphIndex, _i32, _ws
from .ops import _ptr, _stream


def create_graph_local(u_local, items, ratings, n_local_users, nI, item_features, user_features_local, reduce_items=None):
    """`graph.create_graph` over a rank's own interactions (dense ids: user index local to the rank, item index global).
    `reduce_items(t, what)` sums an (nI,) tensor over the ranks in place (`what` in 'cnt' / 'sum' / 'deg' names it; None = single rank)."""
    dev = u_local.device
    lib = L.lib()
    n = int(u_local.numel())
    u_node = (u_local.long() + nI).contiguous()
    i_node = items.long().contiguous()
    r = ratings.contiguous().double()
    cnt_u, cnt_i = _i32(n_local_users, dev, zero=True), _i32(nI, dev, zero=True)
    sum_u = torch.zeros(n_local_users, dtype=torch.float64, device=dev)
    sum_i = torch.zeros(nI, dtype=torch.float64, device=dev)
    attr_u = torch.empty(n, dtype=torch.float32, device=dev)
    attr_i = torch.empty(n, dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        st = _stream()
        L.check(lib.b200rec_group_stats(_ptr(u_node), _ptr(r), n, nI, _ptr(cnt_u), _ptr(sum_u), st), 'group_stats')
        L.check(lib.b200rec_group_stats(_ptr(i_node), _ptr(r), n, 0, _ptr(cnt_i), _ptr(sum_i), st), 'group_stats')
    if reduce_items is not None:               # half-star ratings: the fp64 sums are exact, so the order of the reduction does not matter
        reduce_items(cnt_i, 'cnt')
        reduce_items(sum_i, 'sum')
    with torch.cuda.device(dev):
        st = _stream()
        L.check(lib.b200rec_edge_attrs(_ptr(u_node), _ptr(i_node), _ptr(r), n, nI, _ptr(cnt_u), _ptr(sum_u), _ptr(cnt_i), _ptr(sum_i),
                                       _ptr(attr_u), _ptr(attr_i), None, None, st), 'edge_attrs')
        u2i = torch.empty((2, n), dtype=torch.int64, device=dev)
        i2u = torch.empty((2, n), dtype=torch.int64, device=dev)
        L.check(lib.b200rec_edge_scatter(_ptr(u_node), _ptr(i_node), n, None, None, n, _ptr(u2i), st), 'edge_scatter')
        L.check(lib.b200rec_edge_scatter(_ptr(i_node), _ptr(u_node), n, None, None, n, _ptr(i2u), st), 'edge_scatter')
    return GraphData(item_features=item_features, user_features=user_features_local, user2item_edge_index=u2i, item2user_edge_index=i2u,
                     user2item_edge_attr=attr_u, item2user_edge_attr=attr_i)


def shard_from_local(graph_local, *, rank, world, nI, nU, users_r0, arena, d_max, batch_max, reduce_items=None, edges_total=None, catalogue_width=0,
                     grad_floats=0):
    """PeerShard of a rank from the graph of its own interactions (`create_graph_local`).  The local indexes keep the local graph's reverse
    weights `w_bwd` and its interaction positions, so that training can mask the batch targets of the owned users."""
    from .parallel import _LocalIndex
    from .peer import PeerShard, _rows_per_part
    dev = graph_local.item_features.device
    n_local = int(graph_local.user_features.shape[0])
    idx = GraphIndex(graph_local.user2item_edge_index, graph_local.item2user_edge_index, graph_local.user2item_edge_attr,
                     graph_local.item2user_edge_attr, nI + n_local)
    deg_items = idx.deg[:nI].clone()
    if reduce_items is not None:
        reduce_items(deg_items, 'deg')         # in-degree of an item over ALL ranks' users (gnn_ncf.py:47-48 counts both lists; item rows only receive user->item edges)
    dinv_items = torch.empty(nI, dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        L.check(L.lib().b200rec_dinv(_ptr(deg_items), nI, _ptr(dinv_items), _stream()), 'dinv')
    rp = idx.row_ptr
    k_items = int(rp[nI])
    dinv_users = idx.dinv[nI:].contiguous()
    index_items = _LocalIndex(rp[:nI + 1].contiguous(), (idx.col[:k_items] - nI).contiguous(), idx.w[:k_items].contiguous(), idx.pos[:k_items].contiguous(),
                              dinv_items, idx.chunk_size, w_bwd=idx.w_bwd[:k_items].contiguous())
    index_users = _LocalIndex((rp[nI:] - k_items).contiguous(), idx.col[k_items:].contiguous(), idx.w[k_items:].contiguous(), idx.pos[k_items:].contiguous(),
                              dinv_users, idx.chunk_size, w_bwd=idx.w_bwd[k_items:].contiguous())
    own = int(idx.e1 + idx.e2)
    deg_users, n_positions, symmetric = idx.deg[nI:].contiguous(), idx.e1, idx.symmetric
    del idx
    rpp = _rows_per_part(nI, world)
    i0 = min(rank * rpp, nI)
    return PeerShard(rank=rank, world=world, nI=nI, nU=nU, d_max=d_max, rpp=rpp, users_r0=users_r0, users_rows=n_local, index_users=index_users,
                     index_items=index_items, dinv_users=dinv_users, dinv_items_all=dinv_items,
                     item_features_own=graph_local.item_features[i0: min(i0 + rpp, nI)], user_features_own=graph_local.user_features,
                     arena=arena, batch_max=batch_max, edges_total=own if edges_total is None else edges_total, edges_own=own,
                     catalogue_width=catalogue_width, grad_floats=grad_floats, deg_users=deg_users, deg_items_all=deg_items,
                     n_positions=n_positions, symmetric=symmetric)


def build_shard(u_local, items, ratings, *, nI, nU, users_r0, n_local_users, item_features, user_features_local, group=None, d_max=64,
                batch_max=8192, edges_total=None, catalogue_width=0, grad_floats=0):
    """One process per GPU: the PeerShard of this rank from its own interactions + the arena exchange (collectives at build time only).
    `catalogue_width` > 0 adds the catalogue section of `peer.recommend_peer`, `grad_floats` > 0 the gradient section of training."""
    import torch.distributed as dist
    from .peer import PeerArena, PeerShard, _rows_per_part
    world, rank = dist.get_world_size(group), dist.get_rank(group)

    def reduce_items(t, what):
        dist.all_reduce(t, group=group)

    g = create_graph_local(u_local, items, ratings, n_local_users, nI, item_features, user_features_local, reduce_items if world > 1 else None)
    nbytes = PeerShard.layout(world, _rows_per_part(nI, world), d_max, batch_max, catalogue_width, grad_floats)['total']
    arena = PeerArena.ipc(nbytes, group, device=u_local.device)
    return shard_from_local(g, rank=rank, world=world, nI=nI, nU=nU, users_r0=users_r0, arena=arena, d_max=d_max, batch_max=batch_max,
                            reduce_items=reduce_items if world > 1 else None, edges_total=edges_total, catalogue_width=catalogue_width,
                            grad_floats=grad_floats)
