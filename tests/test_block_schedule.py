"""The hand-over formats of the fn block schedule and of fd's spike tensor, with the yaml models (stress init, 48 patches).

Every format is within the parity tolerances, so a block that silently fell back to a slower fp32 hand-over would still pass
the parity tests; this test pins the formats.  Tap codes of sapcu_model_tap_format: 0 fp32, 1 fp16 (hi, lo) planes, 2 one
fp16 plane.
"""
import os

import pytest
import torch

import sapcu_b200
import sapcu_b200.synthetic as syn
from sapcu_b200 import _native as N
import sapcu_oracle as orc
import oracle_c

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

# mode -> ({block: (snn1, snn_delta2, snn_gamma)}, fd spikes)
EXPECTED = {
    "tc": ({1: (0, 1, 1), 2: (1, 1, 1), 3: (1, 1, 1)}, 1),
    "fast": ({1: (0, 2, 2), 2: (0, 2, 2), 3: (0, 2, 2)}, 2),
}


@pytest.fixture(scope="module")
def models_and_patches():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    torch.cuda.set_device(0)
    from sapcu_b200.fn import config as fc
    from sapcu_b200.fd import config as dc
    mfn = fc.get_model(fc.load_config(os.path.join(sapcu_b200.CONFIG_DIR, "fn.yaml")))
    mfd = dc.get_model(dc.load_config(os.path.join(sapcu_b200.CONFIG_DIR, "fd.yaml")), None)
    syn.init_weights(mfn, seed=100, stress=True)
    syn.init_weights(mfd, seed=200, stress=True)
    cloud = syn.cloud(2048, seed=0, shape="sphere")
    seeds = syn.seeds(cloud, 4, seed=1)[:48]
    p = torch.from_numpy(orc.gather_center(cloud, seeds, oracle_c.knn(cloud, seeds, 100))).to(DEV)
    return mfn.to(DEV), mfd.to(DEV), p


@pytest.mark.parametrize("mode", ["tc", "fast"])
def test_block_hand_over_formats(models_and_patches, mode):
    mfn, mfd, p = models_and_patches
    mfn.set_mode(mode), mfd.set_mode(mode)
    fmt = lambda m, name: N.lib().sapcu_model_tap_format(m._ensure_handle(), name.encode())
    blocks = {}
    for b in (1, 2, 3):
        mfn(p, _stop_after_block=b)          # the formats reported are those of the last block the forward ran
        blocks[b] = tuple(fmt(mfn, "trans%d.%s" % (b, t)) for t in ("snn1", "snn_delta2", "snn_gamma"))
    mfd(p)
    torch.cuda.synchronize()
    N.check_device("block schedule")
    assert (blocks, fmt(mfd, "spikes")) == EXPECTED[mode]
