"""Generate golden fixtures by IMPORTING THE REFERENCE (needs a checkout of
lunarring/latentblending; the tests only read the committed fixture files).

    python tests/golden/make_golden.py <path to the latentblending checkout>

* slerp.npz      -- latentblending/utils.py interpolate_spherical / interpolate_linear
                    outputs on seeded inputs (fp16 and fp32, several fracts incl. 0/1).
                    The tests rebuild the seeded inputs with slerp_cases(), so only the
                    reference's outputs and a checksum of the inputs are stored.
* tree.json      -- the reference BlendingEngine host logic (run_transition,
                    get_mixing_parameters, insert_into_tree, compute_latents_mix
                    coefficient schedules, set_guidance_mid_dampening,
                    get_time_based_branching, swap_forward) driven with the
                    FakeHolder / fake_similarity of tests/golden/fakes.py.
The reference's third-party imports (diffusers, lpips, lunar_tools) are absent
here; they are stubbed with empty modules -- none of their code is on the host
logic exercised.
"""
import hashlib
import json
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
SLERP_FIXTURE = os.path.join(HERE, "slerp.npz")


def _stub(name, **attrs):
    m = types.ModuleType(name)
    for k, v in attrs.items():
        setattr(m, k, v)
    sys.modules[name] = m
    return m


def import_reference(ref_dir):
    _stub("lpips", LPIPS=object)
    _stub("lunar_tools", MovieSaver=object, fill_up_frames_linear_interpolation=None)
    _stub("diffusers", DiffusionPipeline=object, StableDiffusionControlNetPipeline=object, ControlNetModel=object)
    _stub("diffusers.models")
    _stub("diffusers.models.attention_processor", AttnProcessor2_0=object, LoRAAttnProcessor2_0=object,
          LoRAXFormersAttnProcessor=object, XFormersAttnProcessor=object)
    _stub("diffusers.pipelines")
    _stub("diffusers.pipelines.stable_diffusion_xl")
    _stub("diffusers.pipelines.stable_diffusion_xl.pipeline_stable_diffusion_xl", retrieve_timesteps=None)
    sys.path.insert(0, ref_dir)
    import latentblending.utils as ref_utils
    import latentblending.blending_engine as ref_engine
    return ref_utils, ref_engine


def slerp_cases():
    """The seeded (p0, p1, fract) inputs of slerp.npz and the generator they leave behind (it then draws the
    interpolate_linear inputs)."""
    g = torch.Generator().manual_seed(1234)
    shapes = []
    for n, dt in ((64, torch.float16), (4 * 16 * 16, torch.float16), (4 * 64 * 64, torch.float16),
                  (4 * 128 * 128, torch.float16), (777, torch.float32)):
        for f in (0.0, 0.25, 0.5, 0.3141, 1.0):
            shapes.append((n, dt, f))
    cases = []
    for k, (n, dt, f) in enumerate(shapes):
        p0 = (torch.randn(n, generator=g) * (1 + k % 3)).to(dt)
        p1 = (torch.randn(n, generator=g) * 2).to(dt)
        if k % 7 == 3:
            p1 = (p0.float() * 1.5).to(dt)          # parallel vectors -> exercises the 1e-7 clamp
        cases.append((p0, p1, f))
    return cases, g


def slerp_inputs_sha1(cases):
    h = hashlib.sha1()
    for p0, p1, f in cases:
        h.update(p0.numpy().tobytes())
        h.update(p1.numpy().tobytes())
        h.update(np.float64(f).tobytes())
    return h.hexdigest()


def load_slerp_golden():
    """(p0, p1, fract, reference output) of every slerp case."""
    z = np.load(SLERP_FIXTURE)
    cases, _ = slerp_cases()
    assert len(cases) == int(z["n_cases"])
    assert slerp_inputs_sha1(cases) == str(z["inputs_sha1"]), "seeded slerp inputs drifted from the fixture's"
    return [(p0, p1, f, torch.from_numpy(z[f"out_{k}"])) for k, (p0, p1, f) in enumerate(cases)]


def golden_slerp(ref_utils):
    cases, g = slerp_cases()
    out = {f"out_{k}": ref_utils.interpolate_spherical(p0, p1, f).numpy() for k, (p0, p1, f) in enumerate(cases)}
    out["n_cases"] = np.int64(len(cases))
    out["inputs_sha1"] = np.array(slerp_inputs_sha1(cases))
    # interpolate_linear on tensors and uint8 frames
    a = torch.randn(1, 77, 64, generator=g).half()
    b = torch.randn(1, 77, 64, generator=g).half()
    out["lin_a"], out["lin_b"] = a.numpy(), b.numpy()
    out["lin_out"] = ref_utils.interpolate_linear(a, b, 0.3).numpy()
    ia = (torch.rand(8, 8, 3, generator=g) * 255).byte().numpy()
    ib = (torch.rand(8, 8, 3, generator=g) * 255).byte().numpy()
    out["lin_ia"], out["lin_ib"] = ia, ib
    out["lin_iout"] = ref_utils.interpolate_linear(ia, ib, 0.6)
    np.savez_compressed(SLERP_FIXTURE, **out)
    print("slerp.npz:", len(cases), "cases")


def make_ref_engine(ref_engine, turbo, n_steps=None):
    from fakes import FakeHolder, fake_similarity
    be = object.__new__(ref_engine.BlendingEngine)      # skip __init__: it needs diffusers/lpips/cuda
    be.dh = FakeHolder(turbo=turbo)
    be.device = "cpu"
    be.guidance_scale_mid_damper = 0.5
    be.mid_compression_scaler = 1.2
    be.seed1 = be.seed2 = 0
    be.prompt1 = be.prompt2 = ""
    be.tree_latents = [None, None]
    be.tree_fracts = None
    be.tree_final_imgs = []
    be.negative_prompt = None
    be.dt_unet_step, be.dt_vae = 0.05, 0.1
    be.get_lpips_similarity = fake_similarity           # the LPIPS wrapper needs .cuda(); metric is injected
    be.set_guidance_scale()
    be.set_prompt1("")
    be.set_prompt2("")
    be.set_branch1_crossfeed()
    be.set_parental_crossfeed()
    be.set_num_inference_steps(n_steps)
    return be


def run_case(ref_engine, name, turbo, n_steps, branching, prompts, seeds, branch1=None, transitions=1):
    be = make_ref_engine(ref_engine, turbo, n_steps)
    if branch1:
        be.set_branch1_crossfeed(*branch1)
    be.set_branching(**branching)
    rec = dict(name=name, turbo=turbo, n_steps=be.num_inference_steps, branching=branching,
               prompts=prompts, seeds=seeds, branch1=branch1,
               list_idx_injection=[int(v) for v in be.list_idx_injection],
               list_nmb_stems=[int(v) for v in be.list_nmb_stems], transitions=[])
    for t in range(transitions):
        if t == 0:
            be.set_prompt1(prompts[0])
            be.set_prompt2(prompts[1])
            recycle = False
        else:
            be.swap_forward()
            be.set_prompt2(prompts[t + 1])
            recycle = True
        be.dh.calls.clear()
        imgs = be.run_transition(recycle_img1=recycle, fixed_seeds=seeds[t:t + 2])
        rec["transitions"].append(dict(
            tree_fracts=[float(f) for f in be.tree_fracts],
            tree_idx_injection=[int(v) for v in be.tree_idx_injection],
            tree_similarities=[float(s) for s in be.tree_similarities],
            n_imgs=len(imgs),
            img_sums=[int(np.asarray(im).astype(np.int64).sum()) for im in imgs],
            final_latent_sums=[float(tl[-1].float().sum()) for tl in be.tree_latents],
            calls=[dict(c) for c in be.dh.calls],
        ))
    return rec


def golden_tree(ref_engine):
    cases = [
        run_case(ref_engine, "turbo_n4_b3", True, None, dict(nmb_max_branches=3), ["alpha", "beta"], [420, 421]),
        run_case(ref_engine, "base_n30_b15", False, None, dict(depth_strength=0.5, nmb_max_branches=15),
                 ["photo_of a lake", "alien planet"], [420, 421]),
        run_case(ref_engine, "base_n30_b30_x", False, None, dict(nmb_max_branches=30),
                 ["one", "two"], [1, 2], branch1=(0.8, 0.6, 0.4)),
        run_case(ref_engine, "base_n30_t20", False, None, dict(), ["one", "two"], [5, 6]),
        run_case(ref_engine, "base_n20_b6_under", False, 20, dict(depth_strength=0.4, nmb_max_branches=6),
                 ["x", "y"], [7, 8]),
        run_case(ref_engine, "turbo_n4_b12_d", True, None, dict(depth_strength=0.75, nmb_max_branches=12),
                 ["x", "y"], [9, 10]),
        run_case(ref_engine, "base_multi", False, None, dict(nmb_max_branches=10),
                 ["p0", "p1", "p2", "p3"], [11, 12, 13, 14], transitions=3),
    ]
    # branching table alone over a parameter sweep
    sweep = []
    be = make_ref_engine(ref_engine, False)
    for n in (10, 20, 30, 50):
        be.set_num_inference_steps(n)
        for ds in (0.2, 0.5, 0.8):
            for kw in (dict(nmb_max_branches=5), dict(nmb_max_branches=15), dict(nmb_max_branches=30),
                       dict(t_compute_max_allowed=5.0), dict(t_compute_max_allowed=20.0)):
                idx, stems = be.get_time_based_branching(ds, **kw)
                sweep.append(dict(n=n, depth_strength=ds, kw=kw, idx=[int(v) for v in idx],
                                  stems=[int(v) for v in stems]))
    # guidance dampening + closest idx
    damp = [dict(f=f, g=float(ref_engine.BlendingEngine.set_guidance_mid_dampening(be, f) or be.guidance_scale))
            for f in (0.0, 0.125, 0.5, 0.8, 1.0)]
    be.tree_fracts = [0.0, 0.25, 0.5, 0.75, 1.0]
    closest = [dict(f=f, idx=[int(v) for v in be.get_closest_idx(f)]) for f in (0.1, 0.25, 0.3, 0.6, 0.99)]
    with open(os.path.join(HERE, "tree.json"), "w") as f:
        json.dump(dict(cases=cases, branching_sweep=sweep, damp=damp, closest=closest), f, indent=1)
    print("tree.json:", len(cases), "cases,", len(sweep), "branching rows")


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    ref_utils, ref_engine = import_reference(sys.argv[1])
    golden_slerp(ref_utils)
    golden_tree(ref_engine)
