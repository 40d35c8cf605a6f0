"""The device scratch of a call is what its takes need: a small verify call holds a small arena, not a fixed reserve sized
for the largest batch."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture
def fresh_engine():
    import blsful_b200
    e = blsful_b200.Engine([0])
    yield e
    e.close()


def test_small_verify_holds_a_small_arena(fresh_engine):
    import torch
    eng, n = fresh_engine, 16
    rnd = np.random.default_rng(7)
    scalars = rnd.integers(1, 256, size=(n, 32), dtype=np.uint8)
    scalars[:, 0] = 0  # below the group order
    data = rnd.integers(0, 256, size=n * 8, dtype=np.uint8)
    off = np.arange(0, n * 8 + 1, 8, dtype=np.uint64)
    pks, sigs = eng.testdata_sign(2, 0, scalars, data, off)
    free0 = torch.cuda.mem_get_info(0)[0]
    status = eng.verify_batch_packed(2, 0, pks, sigs, data, off)
    grown = free0 - torch.cuda.mem_get_info(0)[0]
    assert (status == 0).all()
    assert grown < 256 * 2 ** 20, f"a {n}-item verify_batch_packed took {grown / 2 ** 20:.0f} MiB of device memory"
