"""derived.Derived, the store behind every cached derived tensor (packed weights, composites, catalogue tables, graph indices), on CPU tensors."""
import torch

from deeprecommendation_b200.derived import Derived


class _Calls:
    def __init__(self):
        self.n = 0

    def __call__(self):
        self.n += 1
        return object()


class _Source:                                   # a non-tensor source, e.g. a GraphIndex
    pass


def test_hit_on_the_same_tensor_and_miss_after_an_in_place_op():
    d, build, t = Derived(4), _Calls(), torch.zeros(8)
    v = d.get((t,), build)
    assert d.get((t,), build) is v and build.n == 1
    t.add_(1)                                    # bumps _version
    assert d.get((t,), build) is not v and build.n == 2


def test_a_view_is_another_source():
    d, build, t = Derived(4), _Calls(), torch.zeros(8)
    v = d.get((t,), build)
    view = t.view_as(t)                          # same address, shared version counter, different object
    assert view.data_ptr() == t.data_ptr() and view._version == t._version
    assert d.get((view,), build) is not v and build.n == 2
    assert d.get((t,), build) is v


def test_a_freed_source_whose_address_is_reused_misses():
    d, build = Derived(1), _Calls()
    for _ in range(8):                           # malloc may serve the first block of a size from mmap and the next ones from its heap
        a = torch.zeros(1 << 16)
        p = a.data_ptr()
        v = d.get((a,), build)
        del a
        b = torch.ones(1 << 16)
        if b.data_ptr() == p:
            break
    assert b.data_ptr() == p and b._version == 0  # precondition: the allocator handed the block back
    assert d.get((b,), build) is not v


def test_a_replaced_non_tensor_source_misses():
    d, build, s = Derived(4), _Calls(), _Source()
    v = d.get((s,), build)
    assert d.get((s,), build) is v
    assert d.get((_Source(),), build) is not v and build.n == 2


def test_none_sources():
    d, build, t = Derived(4), _Calls(), torch.zeros(3)
    v = d.get((t, None), build)
    assert d.get((t, None), build) is v and build.n == 1
    assert d.get((None, t), build) is not v and build.n == 2


def test_extra_is_part_of_the_key():
    d, build, t = Derived(4), _Calls(), torch.zeros(3)
    v = d.get((t,), build, 'fp32', 64)
    assert d.get((t,), build, 'fp32', 64) is v
    assert d.get((t,), build, 'bf16', 64) is not v and d.get((t,), build, 'fp32', 32) is not v and build.n == 3


def test_nothing_stored_under_grad_for_a_source_that_requires_grad():
    d, build, w = Derived(4), _Calls(), torch.zeros(3, requires_grad=True)
    v = d.get((w,), build)
    assert v is not None and len(d) == 0
    assert d.get((w,), build) is not v and build.n == 2
    with torch.no_grad():
        v = d.get((w,), build)
    assert len(d) == 1 and d.get((w,), build) is v          # a hit is returned in grad mode too
    assert d.get((torch.zeros(3),), build) is not None and len(d) == 2   # no source requires grad: stored


def test_capacity_and_clear():
    d, build = Derived(3), _Calls()
    ts = [torch.full((2,), float(i)) for i in range(4)]
    for t in ts[:3]:
        d.get((t,), build)
    assert len(d) == 3
    d.get((ts[3],), build)                       # full: emptied before the new entry goes in
    assert len(d) == 1 and d.values() == [d.get((ts[3],), build)]
    d.clear()
    assert len(d) == 0
    d.get((ts[3],), build)
    assert build.n == 5
