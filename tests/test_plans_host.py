"""CPU tests of the plan ownership in weatherconverter_b200/_plans.py, with fake C functions in place of the library: handle
lifetime, workspace binding, the plan pool and the autograd Function's lease."""
import gc

import pytest
import torch

from weatherconverter_b200 import _plans
from weatherconverter_b200._plans import PlanFunction, PlanHandle, PlanPool, c_tensor_args


class FakeLib:
    """create / destroy of a C plan: hands out handle values 1, 2, ... and counts the destroys of each."""

    def __init__(self):
        self.made, self.destroyed = 0, {}

    def create(self, handle_ref, *args):
        self.made += 1
        handle_ref._obj.value = self.made
        return 0

    def destroy(self, handle):
        self.destroyed[handle.value] = self.destroyed.get(handle.value, 0) + 1

    def plan(self):
        return PlanHandle(self.create, self.destroy)


class FakeModel:
    """A differentiable model on a fake plan: y = 2 x, dx = 2 dy."""

    def __init__(self):
        self.fake, self.pool = FakeLib(), PlanPool()

    def _grad_plan(self, B, H, W, device):
        return self.pool.lease(("key",), (B, H, W), self.fake.plan)

    def _grad_forward(self, plan, x):
        return x * 2

    def _grad_backward(self, plan, g, needs_input_grad, x):
        return (g * 2,)


def test_handle_is_destroyed_once():
    fake = FakeLib()
    plan = fake.plan()
    assert plan.handle.value == 1 and not plan.busy
    plan.__del__()                     # an explicit destroy, then the collector's
    del plan
    gc.collect()
    assert fake.destroyed == {1: 1}


def test_failed_create_destroys_nothing(monkeypatch):
    def refuse(*a):
        raise RuntimeError("refused")
    monkeypatch.setattr(_plans, "check", lambda rc: rc and refuse())
    fake = FakeLib()
    with pytest.raises(RuntimeError, match="refused"):
        PlanHandle(lambda ref: 1, fake.destroy)
    gc.collect()
    assert fake.destroyed == {}


def test_pool_replaces_its_plan_on_a_key_change_and_destroys_the_old_one_once():
    fake, pool = FakeLib(), PlanPool()
    assert pool.plan is None
    a = pool.one("k1", fake.plan)
    assert pool.one("k1", fake.plan) is a and pool.plan is a and fake.made == 1
    del a
    b = pool.one("k2", fake.plan)
    assert fake.destroyed == {1: 1} and b.handle.value == 2 and pool.plan is b
    del b
    pool.one("k3", fake.plan)
    assert fake.destroyed == {1: 1, 2: 1}


def test_workspace_keeps_one_binding():
    plan = FakeLib().plan()
    sizes = []

    def nbytes(n):
        def fn():
            sizes.append(n)
            return n
        return fn
    ws = plan.workspace((2, 8, 8), nbytes(64), "cpu")
    assert ws.numel() == 64 and ws.dtype == torch.uint8 and plan.ws is ws
    assert plan.workspace((2, 8, 8), nbytes(999), "cpu") is ws and sizes == [64]
    ws2 = plan.workspace((4, 8, 8), nbytes(128), "cpu")
    assert ws2.numel() == 128 and plan.ws is ws2 and sizes == [64, 128]
    assert plan.workspace((2, 8, 8), nbytes(64), "cpu") is not ws     # only the last binding is kept
    assert sizes == [64, 128, 64]


def test_workspace_of_size_zero_raises(monkeypatch):
    codes = []

    def check(rc):
        codes.append(rc)
        if rc:
            raise RuntimeError("wc_b200: refused")
    monkeypatch.setattr(_plans, "check", check)
    plan = FakeLib().plan()
    ws = plan.workspace("a", lambda: 16, "cpu")
    with pytest.raises(RuntimeError, match="refused"):
        plan.workspace("b", lambda: 0, "cpu")
    assert codes[-1] == 1 and plan.ws is ws          # the refused binding leaves the old one in place


def test_lease_does_not_hand_out_a_busy_plan_and_reuses_a_freed_one():
    fake, pool = FakeLib(), PlanPool()
    a = pool.lease("k", (1, 8, 8), fake.plan)
    b = pool.lease("k", (1, 8, 8), fake.plan)
    assert a is not b and a.busy and b.busy and len(pool[(1, 8, 8)]) == 2
    c = pool.lease("k", (2, 8, 8), fake.plan)          # another shape has its own plans
    assert c is not a and c is not b and len(pool[(2, 8, 8)]) == 1
    a.busy = False
    assert pool.lease("k", (1, 8, 8), fake.plan) is a and a.busy
    assert len(pool[(1, 8, 8)]) == 2 and fake.made == 3


def test_key_change_empties_the_pool():
    fake, pool = FakeLib(), PlanPool()
    a = pool.lease("k1", (1, 8, 8), fake.plan)
    a.busy = False
    pool.lease("k1", (2, 8, 8), fake.plan).busy = False
    b = pool.lease("k2", (1, 8, 8), fake.plan)
    assert b is not a and list(pool) == [(1, 8, 8)] and pool[(1, 8, 8)] == [b]
    del a
    assert fake.destroyed == {1: 1, 2: 1}


def test_lease_is_released_by_the_backward_and_a_second_backward_raises():
    m = FakeModel()
    x = torch.ones(1, 3, 4, 4, requires_grad=True)
    y = PlanFunction.apply(m, x)
    plan = m.pool[(1, 4, 4)][0]
    assert plan.busy
    loss = y.sum()
    loss.backward(retain_graph=True)
    assert torch.equal(x.grad, torch.full_like(x, 2.0)) and not plan.busy
    with pytest.raises(RuntimeError, match="FakeModel autograd: this graph has already been backpropagated"):
        loss.backward()
    # the freed plan serves the next graph
    PlanFunction.apply(m, x).sum().backward()
    assert len(m.pool[(1, 4, 4)]) == 1


def test_lease_is_released_when_the_graph_is_freed_without_a_backward():
    m = FakeModel()
    x = torch.ones(1, 3, 4, 4, requires_grad=True)
    y1, y2 = PlanFunction.apply(m, x), PlanFunction.apply(m, x)
    p1, p2 = m.pool[(1, 4, 4)]
    assert p1.busy and p2.busy
    del y1
    gc.collect()
    assert not p1.busy and p2.busy
    y3 = PlanFunction.apply(m, x)
    assert len(m.pool[(1, 4, 4)]) == 2 and p1.busy
    del y2, y3
    gc.collect()
    assert not p1.busy and not p2.busy and m.fake.destroyed == {}


def test_c_tensor_args_checks_and_orders():
    ts = {"b": torch.zeros(3), "a": torch.zeros(2, 2)}
    names, ptrs, numels = c_tensor_args(ts, torch.device("cpu"), "M", torch.float32)
    assert [names[i] for i in range(2)] == [b"b", b"a"]
    assert [ptrs[i] for i in range(2)] == [t.data_ptr() for t in ts.values()] and list(numels) == [3, 4]
    with pytest.raises(RuntimeError, match="M tensor a must be a contiguous float32 tensor on cpu"):
        c_tensor_args({"a": torch.zeros(2, 2).t()}, torch.device("cpu"), "M", torch.float32)
    with pytest.raises(RuntimeError, match="M tensor a must be a contiguous float32 tensor on cpu"):
        c_tensor_args({"a": torch.zeros(2, dtype=torch.float64)}, torch.device("cpu"), "M", torch.float32)
    with pytest.raises(RuntimeError, match="M tensor a must be a contiguous tensor on cuda:0"):
        c_tensor_args({"a": torch.zeros(2)}, torch.device("cuda:0"), "M")
