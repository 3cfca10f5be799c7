"""Pins for the CPU oracle: reference-generated golden vectors (tests/golden/),
published scheduler constants (SURVEY.md appendix C), the public SDXL UNet
parameter count."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import engine as oeng
from oracle import mixing
from oracle.schedulers import EulerAncestralDiscrete, EulerDiscrete
from oracle.sdxl_unet import SDXL_BASE, count_params

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def test_slerp_matches_reference_golden():
    from make_golden import load_slerp_golden
    for k, (p0, p1, f, ref) in enumerate(load_slerp_golden()):
        out = mixing.interpolate_spherical(p0, p1, f)
        assert out.dtype == ref.dtype
        assert torch.equal(out, ref), f"case {k}"


def test_lerp_matches_reference_golden():
    z = np.load(os.path.join(GOLD, "slerp.npz"))
    out = mixing.interpolate_linear(torch.from_numpy(z["lin_a"]), torch.from_numpy(z["lin_b"]), 0.3)
    assert torch.equal(out, torch.from_numpy(z["lin_out"]))
    assert np.array_equal(mixing.interpolate_linear(z["lin_ia"], z["lin_ib"], 0.6), z["lin_iout"])


def test_euler_known_answers():
    s = EulerDiscrete()
    s.set_timesteps(30)
    assert s.timesteps[:3].tolist() == [958.0, 925.0, 892.0] and s.timesteps[-1] == 1.0
    want = [11.4769, 9.5436, 8.0043, 6.7684, 5.7678, 4.9510, 4.2790, 3.7216, 3.2556, 2.8629, 2.5295, 2.2441,
            1.9980, 1.7841, 1.5968, 1.4316, 1.2846, 1.1530, 1.0342, 0.9261, 0.8270, 0.7353, 0.6499, 0.5693,
            0.4924, 0.4179, 0.3439, 0.2677, 0.1822, 0.0413, 0.0]
    np.testing.assert_allclose(s.sigmas.numpy(), want, atol=6e-5)
    assert abs(float(s.init_noise_sigma) - 11.5203) < 1e-4
    full = EulerDiscrete()
    assert abs(float(full.sigmas.max()) - 14.6146) < 1e-4
    assert abs(float(full.sigmas[full.sigmas > 0].min()) - 0.0292) < 1e-4


def test_euler_ancestral_known_answers():
    s = EulerAncestralDiscrete()
    s.set_timesteps(4)
    assert s.timesteps.tolist() == [999.0, 749.0, 499.0, 249.0]
    np.testing.assert_allclose(s.sigmas.numpy(), [14.6146, 4.0817, 1.6129, 0.6932, 0.0], atol=6e-5)
    assert abs(float(s.init_noise_sigma) - 14.6146) < 1e-4
    ups = [float(s.sigma_up_down(i)[0]) for i in range(4)]
    downs = [float(s.sigma_up_down(i)[1]) for i in range(4)]
    np.testing.assert_allclose(ups, [3.9193, 1.4816, 0.6259, 0.0], atol=1e-4)
    np.testing.assert_allclose(downs, [1.1400, 0.6373, 0.2979, 0.0], atol=1e-4)


def test_unet_param_count_is_sdxl():
    assert count_params(SDXL_BASE) == 2_567_463_684


def _tree():
    with open(os.path.join(GOLD, "tree.json")) as f:
        return json.load(f)


def test_branching_sweep_matches_reference():
    for row in _tree()["branching_sweep"]:
        idx, stems = oeng.time_based_branching(row["n"], row["depth_strength"], 0.05, 0.1, **row["kw"])
        assert [int(v) for v in idx] == row["idx"], row
        assert [int(v) for v in stems] == row["stems"], row


def test_guidance_dampening_and_closest_idx_match_reference():
    t = _tree()
    for d in t["damp"]:
        assert abs(oeng.guidance_mid_dampening(4.0, 0.5, d["f"]) - d["g"]) < 1e-12
    for c in t["closest"]:
        assert list(oeng.closest_idx([0.0, 0.25, 0.5, 0.75, 1.0], c["f"])) == c["idx"]


@pytest.mark.parametrize("case", _tree()["cases"], ids=lambda c: c["name"])
def test_oracle_engine_tree_matches_reference(case):
    from fakes import FakeHolder, fake_similarity
    dh = FakeHolder(turbo=case["turbo"])
    be = oeng.OracleEngine(dh, lpips_net=object())
    be.similarity = fake_similarity
    be.set_num_inference_steps(None if case["n_steps"] in (4, 30) else case["n_steps"])
    if case["branch1"]:
        be.set_branch1_crossfeed(*case["branch1"])
    be.set_branching(**case["branching"])
    assert [int(v) for v in be.list_idx_injection] == case["list_idx_injection"]
    assert [int(v) for v in be.list_nmb_stems] == case["list_nmb_stems"]
    for t, gold in enumerate(case["transitions"]):
        if t == 0:
            be.set_prompt1(case["prompts"][0])
            be.set_prompt2(case["prompts"][1])
            recycle = False
        else:
            be.swap_forward()
            be.set_prompt2(case["prompts"][t + 1])
            recycle = True
        dh.calls.clear()
        imgs = be.run_transition(recycle_img1=recycle, fixed_seeds=case["seeds"][t:t + 2])
        assert be.tree_fracts == gold["tree_fracts"]
        assert [int(v) for v in be.tree_idx_injection] == gold["tree_idx_injection"]
        np.testing.assert_allclose(be.tree_similarities, gold["tree_similarities"], rtol=0, atol=0)
        assert len(imgs) == gold["n_imgs"]
        assert [int(np.asarray(im).astype(np.int64).sum()) for im in imgs] == gold["img_sums"]
        assert len(dh.calls) == len(gold["calls"])
        for a, b in zip(dh.calls, gold["calls"]):
            assert a["idx_start"] == b["idx_start"]
            assert a["guidance"] == b["guidance"]
            assert a["n_mix_none"] == b["n_mix_none"]
            if isinstance(b["coeffs"], list):
                np.testing.assert_allclose(a["coeffs"], b["coeffs"], rtol=0, atol=0)
            else:
                assert a["coeffs"] == b["coeffs"]
            assert a["start_sum"] == b["start_sum"] and a["cond_sum"] == b["cond_sum"]
