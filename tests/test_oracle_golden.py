"""CPU: the oracle (torch restatement + plain-C restatement) against the golden vectors generated from the real
reference by oracle/make_golden.py.  These run without the reference checkout."""
import json
import os

import numpy as np
import torch

import sapcu_b200  # noqa: F401
import sapcu_b200.synthetic as syn
import sapcu_oracle as orc
import oracle_c
from conftest import GOLDEN


def _models():
    from sapcu_b200.fn import config as fc
    from sapcu_b200.fd import config as dc
    mfn = fc.get_model(fc.load_config(os.path.join(sapcu_b200.CONFIG_DIR, "fn.yaml")))
    mfd = dc.get_model(dc.load_config(os.path.join(sapcu_b200.CONFIG_DIR, "fd.yaml")), None)
    return mfn, mfd


def test_state_dict_keys_match_reference():
    """Drop-in boundary: the shim modules expose exactly the reference's state_dict names and shapes."""
    inv = json.load(open(os.path.join(GOLDEN, "state_dict_keys.json")))
    mfn, mfd = _models()
    for tag, m in (("fn", mfn), ("fd", mfd)):
        mine = {k: list(v.shape) for k, v in m.state_dict().items()}
        assert mine == inv[tag]


def test_knn_oracles_match_kdtree(golden):
    cloud = syn.cloud(2048, seed=0, shape="sphere")
    seeds = syn.seeds(cloud, 4, seed=1)[:512]
    g = golden.knn
    assert np.array_equal(orc.knn_seed(cloud, seeds, 100), g["idx_sphere"])
    assert np.array_equal(oracle_c.knn(cloud, seeds, 100), g["idx_sphere"])
    cb = syn.cloud(1500, seed=3, shape="boxes")
    sb = syn.seeds(cb, 0.2, seed=4)
    assert np.array_equal(oracle_c.knn(cb, sb, 48), g["idx_boxes"])


def test_neuron_known_answers(golden):
    g = golden.neuron
    x = torch.from_numpy(g["x"])
    prm = {k[2:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("p_")}
    lifp = {k: v for k, v in prm.items() if k not in ("delta_T", "theta_rh")}
    # torch's CPU exp / sigmoid round differently in the last bits on some CPU types: the reference's outputs are reproduced
    # bit for bit where the soft spike alone (the first LIF step) rounds as on the host that stored them, else to a few ulp
    exact = torch.equal(orc.spike_function(x - prm["threshold_base"]), torch.from_numpy(g["lif"][0]))
    for tag, p in (("lif", lifp), ("eif", prm)):
        got = orc.lif_chain(x, p, 7, all_steps=True)
        if exact:
            assert torch.equal(got, torch.from_numpy(g[tag]))
        else:
            np.testing.assert_allclose(got.numpy(), g[tag], rtol=2e-6, atol=1e-7)
    p4 = np.stack([g["p_membrane_decay"], g["p_threshold_adapt"], g["p_refractory_decay"], g["p_threshold_base"]])
    e2 = np.stack([g["p_delta_T"], g["p_theta_rh"]])
    # plain C uses libm expf instead of torch's vectorised exp: equal to a few ulp, not bitwise
    np.testing.assert_allclose(oracle_c.neuron_chain(g["x"], p4, 7), g["lif"], rtol=2e-6, atol=1e-7)
    np.testing.assert_allclose(oracle_c.neuron_chain(g["x"], p4, 7, e2), g["eif"], rtol=2e-6, atol=1e-7)


def test_gate_is_closed_after_first_step(golden):
    """SURVEY.md fact 4: the soft spike is > 0, so every step after the first ignores its input."""
    g = golden.neuron
    prm = {k[2:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("p_")}
    x = torch.from_numpy(g["x"])
    s, st = orc.eif_step(x, prm, None)
    a, _ = orc.eif_step(torch.randn_like(x) * 50, prm, st)
    b, _ = orc.eif_step(torch.zeros_like(x), prm, st)
    assert torch.equal(a, b) and float(s.min()) > 0


def test_patch_ops(golden):
    g = golden.patch_ops
    cloud = syn.cloud(2048, seed=0, shape="sphere")
    seeds = syn.seeds(cloud, 4, seed=1)[:40]
    idx = golden.knn["idx_sphere"][:40]
    for n, R in zip(g["normals"], g["R"]):
        assert np.array_equal(orc.rotation_to_x(n), R)
        np.testing.assert_allclose(oracle_c.rotation_to_x(n), R, rtol=0, atol=1e-15)
    assert np.array_equal(orc.gather_center(cloud, seeds, idx), g["patch"])
    assert np.array_equal(orc.gather_center(cloud, seeds, idx, g["normals"]), g["rotated"])
    assert np.array_equal(oracle_c.gather_center_rotate(cloud, seeds, idx), g["patch"])
    np.testing.assert_allclose(oracle_c.gather_center_rotate(cloud, seeds, idx, g["normals"]), g["rotated"], rtol=0, atol=1e-8)
    assert np.array_equal(orc.displace(seeds, g["unit_normals"], g["dist"]), g["displaced"])
    assert np.array_equal(oracle_c.displace(seeds, g["unit_normals"], g["dist"]), g["displaced"])


def test_model_forwards_match_reference(golden):
    g = golden.models
    mfn, mfd = _models()
    p = torch.from_numpy(g["patches"])
    with torch.no_grad():
        for tag, stress in (("default", False), ("stress", True)):
            syn.init_weights(mfn, seed=100, stress=stress)
            syn.init_weights(mfd, seed=200, stress=stress)
            taps_fn, taps_fd = {}, {}
            n = orc.fn_forward(mfn.state_dict(), p, taps=taps_fn)
            # torch's CPU convolutions block (and so round) by CPU type and thread count, and its exp by CPU type: the
            # reference's outputs are reproduced bit for bit only on the host that stored them, elsewhere to fp32 rounding
            # (the bounds of test_pipeline_matches_reference); spike taps to 2e-3, since last-bit differences can reorder
            # the exact ties of the fd feature-space graphs under the default init
            np.testing.assert_allclose(n.numpy(), g[tag + "_normals"], rtol=0, atol=2e-6)
            np.testing.assert_allclose(taps_fn["snn_init"][:, ::4].numpy(), g[tag + "_fn_snn_init"], rtol=0, atol=2e-6)
            np.testing.assert_allclose(taps_fn["snn_final"][:, ::16].numpy(), g[tag + "_fn_snn_final"], rtol=0, atol=2e-6)
            pf = torch.from_numpy(g[tag + "_patches_fd"])
            d = orc.fd_forward(mfd.state_dict(), pf, taps=taps_fd)
            np.testing.assert_allclose(d.numpy(), g[tag + "_dist"], rtol=2e-5, atol=1e-7)
            np.testing.assert_allclose(taps_fd["spikes"][:, :, ::16].numpy(), g[tag + "_fd_spikes"], rtol=0, atol=2e-3)
            # exact dead-code elimination: closed-gate schedule == faithful schedule, bit for bit
            assert torch.equal(orc.fd_forward(mfd.state_dict(), pf, schedule="dce"), d)


def test_pipeline_matches_reference(golden):
    g = golden.pipeline
    mfn, mfd = _models()
    syn.init_weights(mfn, seed=100, stress=True)
    syn.init_weights(mfd, seed=200, stress=True)
    cloud = syn.cloud(2048, seed=0, shape="sphere")
    S = 8      # a slice of the 32 golden seeds keeps the CPU suite short; per-seed results are independent
    pts, _, n, d = orc.pipeline(mfn.state_dict(), mfd.state_dict(), cloud, g["seeds"][:S], K=100, batch=400,
                                schedule="dce")
    np.testing.assert_allclose(n, g["normals"][:S], rtol=0, atol=2e-6)
    np.testing.assert_allclose(d, g["dist"][:S], rtol=2e-5, atol=1e-7)
    # a different batch size changes torch's conv blocking: agreement is to fp32 rounding, not bitwise
    np.testing.assert_allclose(pts, g["points"][:S], rtol=0, atol=1e-5)


def test_seed_golden_matches_reference_binary(golden, tmp_path):
    """Fixture integrity for the seed-generator row: re-run the compiled reference (when present) on one case."""
    import subprocess
    import pytest
    from conftest import ROOT
    dense = os.path.join(ROOT, "oracle", "_ref", "dense")
    if not os.path.exists(dense):
        pytest.skip("oracle/_ref/dense not built (make -C oracle ref)")
    cloud = syn.cloud(256, seed=5, shape="sphere")
    np.savetxt(tmp_path / "test.xyz", cloud, fmt="%.17g")
    subprocess.check_call([dense, "0.01", "256"], cwd=tmp_path)
    ref = np.loadtxt(tmp_path / "target.xyz").reshape(-1, 3)
    assert np.array_equal(np.rint(ref * 1e6).astype(np.int32), golden.seeds["sphere256_c010"])


def test_outlier_filter_and_fps_oracles(golden):
    g = golden.post
    assert np.array_equal(orc.outlier_filter(g["out_points"], 1.5), g["out_keep"])
    assert np.array_equal(orc.fps(g["fps_xyz"], 512), g["fps_idx"])
    grid = np.stack(np.meshgrid(np.arange(12), np.arange(12), np.arange(12), indexing="ij"), -1).reshape(-1, 3).astype(np.float64)
    assert np.array_equal(orc.fps(grid, 200), g["fps_grid_idx"])


def test_fps_c_oracle_matches_numpy_oracle_and_reference(golden):
    """oracle_c.fps (the plain-C FPS the GPU tests compare whole pick sequences with) equals the numpy restatement and the
    reference's own picks, ties included."""
    g = golden.post
    assert np.array_equal(oracle_c.fps(g["fps_xyz"], 512), g["fps_idx"])
    grid = np.stack(np.meshgrid(np.arange(12), np.arange(12), np.arange(12), indexing="ij"), -1).reshape(-1, 3).astype(np.float64)
    assert np.array_equal(oracle_c.fps(grid, 200), g["fps_grid_idx"])
    rng = np.random.default_rng(21)
    pts = rng.normal(size=(5000, 3))
    assert np.array_equal(oracle_c.fps(pts, 700), orc.fps(pts, 700))
    # tie-heavy: the grid stored twice (every distance is shared by at least two rows), 1e4 + a unit sphere (fp32 at
    # magnitude), identical points, and more picks than points (the picks after exhaustion are index 0)
    twice = np.concatenate([grid, grid], 0)
    assert np.array_equal(oracle_c.fps(twice, 300), orc.fps(twice, 300))
    far = rng.normal(size=(3000, 3)); far = 1e4 + far / np.linalg.norm(far, axis=1, keepdims=True)
    assert np.array_equal(oracle_c.fps(far, 400), orc.fps(far, 400))
    same = np.full((100, 3), 0.25)
    assert np.array_equal(oracle_c.fps(same, 5), orc.fps(same, 5))
    assert np.array_equal(oracle_c.fps(pts[:40], 45), orc.fps(pts[:40], 45))
    assert (oracle_c.fps(pts[:40], 45)[40:] == 0).all()
    for start in (0, 1234, 4999):
        assert np.array_equal(oracle_c.fps(pts, 200, start=start), orc.fps(pts, 200, start=start))
        assert np.array_equal(oracle_c.fps(twice, 100, start=start % 3456), orc.fps(twice, 100, start=start % 3456))
