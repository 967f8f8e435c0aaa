"""Host-side parts of peer.recommend_peer (deeprecommendation_b200/peer.py): the catalogue section of the arena layout, the filtering of a
request to a rank's users, and the `ignore_seen` CSR built from a shard's local user index."""
import pytest
import torch

from deeprecommendation_b200.peer import PeerShard, _align, _rows_per_part, catalogue_width, seen_csr, served_rows

LAYOUTS = [(1, 62423, 128, 8192), (8, 62423, 128, 8192), (3, 11, 64, 512), (8, 1_000_000, 64, 8192)]


@pytest.mark.parametrize('case', LAYOUTS)
@pytest.mark.parametrize('width', [64, 256])
def test_catalogue_section_after_stats1(case, width):
    world, nI, d_max, batch_max = case
    rpp = _rows_per_part(nI, world)
    base = PeerShard.layout(world, rpp, d_max, batch_max)
    off = PeerShard.layout(world, rpp, d_max, batch_max, width)
    assert {k: v for k, v in off.items() if k not in ('cat', 'total')} == {k: v for k, v in base.items() if k != 'total'}
    assert off['cat'] == base['total'] == off['stats1'] + _align(world * rpp * 8)
    assert off['cat'] % 256 == 0
    assert off['total'] == off['cat'] + _align(world * rpp * width * 4)


@pytest.mark.parametrize('case', LAYOUTS)
def test_width_zero_is_the_layout_without_catalogue(case):
    world, nI, d_max, batch_max = case
    rpp = _rows_per_part(nI, world)
    assert PeerShard.layout(world, rpp, d_max, batch_max, 0) == PeerShard.layout(world, rpp, d_max, batch_max)
    assert 'cat' not in PeerShard.layout(world, rpp, d_max, batch_max)


def test_catalogue_section_size_at_config5():
    """10^6 items on 8 ranks, d = 64: 256 MB per rank for the running mean, 1 GB for concat at L = 3"""
    rpp = _rows_per_part(1_000_000, 8)
    for width, mb in ((64, 256), (256, 1024)):
        off = PeerShard.layout(8, rpp, 64, 8192, width)
        assert off['total'] - off['cat'] == 8 * rpp * width * 4 == mb * 1_000_000


def test_catalogue_width_of_models():
    from deeprecommendation_b200.neural_collaborative_filtering.models import GraphNCF
    mk = lambda **kw: GraphNCF(item_dim=8, user_dim=8, num_gnn_layers=kw.pop('L', 2), hetero=True, **kw)
    assert catalogue_width(mk(node_emb=64)) == 64
    assert catalogue_width(mk(node_emb=32, use_dot_product=True)) == 64                  # the dot kernel's operand width
    assert catalogue_width(mk(node_emb=48, concat=True, use_dot_product=True)) == 192     # 3 x 48 = 144 -> 192
    assert catalogue_width(mk(node_emb=48, concat=True)) == 144                          # MLP: no padding
    assert catalogue_width(mk(node_emb=64, L=0)) == 64


def test_served_rows_keep_request_order_and_range():
    nI, r0, rows = 100, 40, 25                                  # this rank: user nodes 140 .. 164
    users = torch.tensor([170, 150, 139, 164, 140, 165, 150, 0, 99, 141])
    nodes, local = served_rows(users, nI, r0, rows)
    assert nodes.tolist() == [150, 164, 140, 150, 141]
    assert local.tolist() == [10, 24, 0, 10, 1]
    nodes, local = served_rows(torch.tensor([1, 2, 3]), nI, r0, rows)
    assert nodes.numel() == 0 and local.numel() == 0
    # the ranks' ranges split any request: each node served exactly once
    req = torch.randperm(300)[:120] + nI
    parts = [(0, 90), (90, 110), (200, 100)]
    got = torch.cat([served_rows(req, nI, a, n)[0] for a, n in parts])
    assert sorted(got.tolist()) == sorted(req.tolist())


def test_seen_csr_on_a_local_index_with_more_items_than_owned_users():
    """3 owned users, item ids up to 999: keys row * num_nodes (= 3) + item would collide across rows; row * nI does not"""
    nI = 1000
    row_ptr = torch.tensor([0, 4, 4, 7], dtype=torch.int32)
    col = torch.tensor([999, 5, 700, 6, 3, 998, 0], dtype=torch.int32)
    ptr, idx = seen_csr(row_ptr, col, torch.arange(3), nI)
    assert ptr.dtype == torch.int32 and idx.dtype == torch.int32
    assert ptr.tolist() == [0, 4, 4, 7]
    assert idx.tolist() == [5, 6, 700, 999, 0, 3, 998]
    ptr, idx = seen_csr(row_ptr, col, torch.tensor([2, 0, 2]), nI)        # a subset in request order, repeats allowed
    assert ptr.tolist() == [0, 3, 7, 10]
    assert idx.tolist() == [0, 3, 998, 5, 6, 700, 999, 0, 3, 998]
    ptr, idx = seen_csr(row_ptr, col, torch.zeros(0, dtype=torch.int64), nI)
    assert ptr.tolist() == [0] and idx.numel() == 0
