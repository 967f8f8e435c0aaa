"""The peer arena layout (deeprecommendation_b200/peer.py): the LightGAT sections (item score tables S0 / S1 and the (m, l) statistics of
the receive slots) come after the LightGCN sections, whose offsets stay where they were."""
import pytest

from deeprecommendation_b200.peer import PeerShard, _align, _rows_per_part

# (world, items, d_max, batch_max) -> offsets of recv0, recv1, T0, T1, rows and the end of the rows section
CASES = {
    (1, 62423, 128, 8192): (4096, 31964672, 63925248, 95885824, 127846400, 136235008),
    (8, 62423, 128, 8192): (4096, 31965184, 63926272, 95887360, 127848448, 136237056),
    (3, 11, 64, 512): (4096, 7168, 10240, 13312, 16384, 278528),
    (8, 1_000_000, 64, 8192): (4096, 256004096, 512004096, 768004096, 1024004096, 1028198400),
}


@pytest.mark.parametrize('case', sorted(CASES))
def test_lightgcn_offsets_unchanged_and_gat_sections_appended(case):
    world, nI, d_max, batch_max = case
    rpp = _rows_per_part(nI, world)
    off = PeerShard.layout(world, rpp, d_max, batch_max)
    *old, rows_end = CASES[case]
    assert [off[k] for k in ('recv0', 'recv1', 'T0', 'T1', 'rows')] == old
    assert off['S0'] == rows_end
    assert off['S1'] == off['S0'] + _align(world * rpp * 4)
    assert off['stats0'] == off['S1'] + _align(world * rpp * 4)
    assert off['stats1'] == off['stats0'] + _align(world * rpp * 8)
    assert off['total'] == off['stats1'] + _align(world * rpp * 8)
    assert all(off[k] % 256 == 0 for k in off)
