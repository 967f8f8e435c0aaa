"""Partitioned GraphNCF training, the host side: the gradient section of the peer arena and the parameter count it is sized by."""
import pytest
import torch

from deeprecommendation_b200.peer import PeerShard, _align, _rows_per_part, _train_params, grad_floats

CASES = [(1, 62423, 128, 8192, 0), (8, 62423, 128, 8192, 128), (3, 11, 64, 512, 64), (8, 1_000_000, 64, 8192, 0)]


@pytest.mark.parametrize('world, nI, d_max, batch_max, cat', CASES)
def test_layout_without_grad_section_is_unchanged(world, nI, d_max, batch_max, cat):
    rpp = _rows_per_part(nI, world)
    before = PeerShard.layout(world, rpp, d_max, batch_max, cat)
    assert PeerShard.layout(world, rpp, d_max, batch_max, cat, 0) == before
    off = PeerShard.layout(world, rpp, d_max, batch_max, cat, 1001)
    assert {k: v for k, v in off.items() if k not in ('grad', 'total')} == {k: v for k, v in before.items() if k != 'total'}
    assert off['grad'] == before['total'] and off['grad'] % 256 == 0
    assert off['total'] == off['grad'] + _align(world * 1004 * 4)       # slots of 1001 floats rounded up to 4


def _model(L_, hetero, mlp=(256, 128), d=64, F=48, Fu=40, **kw):
    from deeprecommendation_b200.neural_collaborative_filtering.models import GraphNCF
    return GraphNCF(item_dim=F, user_dim=Fu, num_gnn_layers=L_, hetero=hetero, node_emb=d, mlp_dense_layers=list(mlp or (8,)),
                    use_dot_product=mlp is None, **kw)


@pytest.mark.parametrize('L_', [0, 1, 3])
@pytest.mark.parametrize('hetero', [True, False])
@pytest.mark.parametrize('mlp', [(256, 128), None])
def test_grad_floats_counts_embedding_and_conv_parameters(L_, hetero, mlp):
    m = _model(L_, hetero, mlp, d=64, F=45, Fu=40)
    names = list(_train_params(m))
    emb = ['item_embeddings.0.weight', 'item_embeddings.0.bias', 'user_embeddings.0.weight', 'user_embeddings.0.bias']
    conv = [] if L_ == 0 else (['gnn_convs.0.user2item_W.0.weight', 'gnn_convs.0.user2item_W.0.bias', 'gnn_convs.0.item2user_W.0.weight',
                                'gnn_convs.0.item2user_W.0.bias'] if hetero else ['gnn_convs.0.W.0.weight', 'gnn_convs.0.W.0.bias'])
    assert sorted(names) == sorted(emb + conv)                     # the MLP is trained by ordinary autograd on every rank; aliased layers once
    pad4 = lambda n: (n + 3) // 4 * 4
    want = pad4(64 * 45) + 64 + pad4(64 * 40) + 64 + (0 if L_ == 0 else (2 if hetero else 1) * (64 * 64 + 64))
    assert grad_floats(m) == want and want % 4 == 0
    assert grad_floats(m) >= sum(p.numel() for n, p in m.named_parameters() if not n.startswith('MLP'))

