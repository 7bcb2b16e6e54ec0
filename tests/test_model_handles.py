"""CPU: ownership of the native model handles in the nn.Module shims, against a fake library that records what is created,
finalized and destroyed (no device memory is touched).  One handle per device, built once per parameter version; a
DataParallel replica borrows its owner's handles and never destroys one; the owner destroys each of its handles once."""
import copy
import gc
import os

import pytest
import torch

import sapcu_b200
from sapcu_b200 import _native as N


class FakeLib:
    def __init__(self):
        self.next, self.created, self.finalized, self.destroyed = 1000, [], [], []

    def sapcu_model_create(self, kind, cfg, n):
        self.next += 1
        self.created.append(self.next)
        return self.next

    def sapcu_model_set_tensor(self, h, name, ptr, numel):
        return 0

    def sapcu_model_finalize(self, h):
        self.finalized.append(h)
        return 0

    def sapcu_model_destroy(self, h):
        self.destroyed.append(h)

    def sapcu_last_error(self):
        return b""


@pytest.fixture
def fake(monkeypatch):
    f = FakeLib()
    monkeypatch.setattr(N, "_lib", f)
    return f


def _fn_model():
    from sapcu_b200.fn import config as fc
    return fc.get_model(fc.load_config(os.path.join(sapcu_b200.CONFIG_DIR, "fn.yaml")))


D0, D1, D2 = torch.device("cuda", 0), torch.device("cuda", 1), torch.device("cuda", 2)


def test_one_handle_per_device_built_once(fake):
    m = _fn_model()
    h0 = m._ensure_handle(D0)
    h1 = m._ensure_handle(D1)
    assert h0 != h1 and fake.created == [h0, h1] and fake.finalized == [h0, h1]
    for _ in range(3):                                   # a module switching between two devices
        assert m._ensure_handle(D0) == h0 and m._ensure_handle(D1) == h1
    assert m._ensure_handle("cuda:1") == h1
    assert len(fake.created) == 2 and fake.destroyed == []
    # parameters changed in place: each device's handle is replaced once, by the owner
    with torch.no_grad():
        m.decoder.fc_out.bias.add_(1.0)
    n0 = m._ensure_handle(D0)
    assert n0 not in (h0, h1) and fake.destroyed == [h0]
    assert m._ensure_handle(D0) == n0 and fake.destroyed == [h0]
    n1 = m._ensure_handle(D1)
    assert fake.destroyed == [h0, h1] and len(fake.created) == 4
    del m
    gc.collect()
    assert sorted(fake.destroyed) == sorted([h0, h1, n0, n1])


def test_data_parallel_replica_borrows_and_destroys_nothing(fake):
    m = _fn_model()
    h0 = m._ensure_handle(D0)
    reps = [m._replicate_for_data_parallel() for _ in range(3)]
    assert reps[0]._ensure_handle(D0) == h0                          # same device: the owner's handle
    h1 = reps[1]._ensure_handle(D1)                                  # another device: built once, in the owner's cache
    assert reps[2]._ensure_handle(D1) == h1 and m._ensure_handle(D1) == h1
    h2 = reps[2]._ensure_handle(D2)
    assert len(fake.created) == 3
    rr = reps[2]._replicate_for_data_parallel()                      # a replica of a replica still borrows from the owner
    assert rr._ensure_handle(D2) == h2 and len(fake.created) == 3
    del reps, rr
    gc.collect()
    assert fake.destroyed == []
    assert m._ensure_handle(D0) == h0                                # the owner's handles are still alive and cached
    del m
    gc.collect()
    assert sorted(fake.destroyed) == sorted([h0, h1, h2])            # each exactly once


def test_copies_start_without_handles(fake):
    m = _fn_model()
    h0 = m._ensure_handle(D0)
    c = copy.deepcopy(m)
    hc = c._ensure_handle(D0)                                        # its own handle, not a second owner of h0
    assert hc != h0 and len(fake.created) == 2
    del c
    gc.collect()
    assert fake.destroyed == [hc]
    del m
    gc.collect()
    assert sorted(fake.destroyed) == sorted([hc, h0])
