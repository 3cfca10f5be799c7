"""GPU parity: K1 (slerp/lerp) and K9 (CFG + Euler step) through the C ABI
against the CPU oracle and the reference-generated golden vectors.
Bar: bit-exact (the kernels reproduce the reference's rounding chain)."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")


def test_slerp_golden_bit_exact():
    from latentblending_b200 import utils
    from make_golden import load_slerp_golden
    for k, (p0, p1, f, ref) in enumerate(load_slerp_golden()):
        out = utils.interpolate_spherical(p0.cuda(), p1.cuda(), f).cpu()
        assert out.dtype == ref.dtype
        assert torch.equal(out, ref), f"case {k}: {(out != ref).sum().item()} mismatches"


@pytest.mark.parametrize("n", [8, 1000, 1024, 4 * 64 * 64, 4 * 128 * 128, 4 * 128 * 128 + 8, 4 * 160 * 160, 300001])
@pytest.mark.parametrize("dtype", [torch.float16, torch.float32])
def test_slerp_rows_vs_oracle(n, dtype):
    from latentblending_b200 import ops
    from oracle import mixing
    g = torch.Generator().manual_seed(n)
    rows = 5
    p0 = (torch.randn(rows, n, generator=g) * 3).to(dtype)
    p1 = torch.randn(rows, n, generator=g).to(dtype)
    out = ops.slerp_rows(p0.cuda(), p1.cuda(), 0.37).cpu()
    for r in range(rows):
        ref = mixing.interpolate_spherical(p0[r], p1[r], 0.37)
        if dtype == torch.float16:
            assert torch.equal(out[r], ref), f"row {r}: {(out[r] != ref).sum().item()} mismatches"
        else:
            # fp32 output: the fp64 row sums are accumulated in a different order than torch's, so a
            # result sitting on an fp32 rounding boundary may flip by 1 ulp (torch CPU vs torch CUDA do too)
            bad = out[r] != ref
            assert bad.sum().item() <= max(1, n // 100000), f"row {r}: {bad.sum().item()} mismatches"
            assert torch.allclose(out[r], ref, rtol=2.5e-7, atol=0)


def test_slerp_strided_rows_and_per_row_fract():
    from latentblending_b200 import ops
    from oracle import mixing
    g = torch.Generator().manual_seed(3)
    n = 4 * 32 * 32
    big0 = torch.randn(6, 2, n, generator=g).half()
    big1 = torch.randn(6, 2, n, generator=g).half()
    fr = torch.tensor([0.0, 0.1, 0.5, 0.9, 1.0, 0.33], dtype=torch.float64)
    a, b = big0.cuda()[:, 1], big1.cuda()[:, 0]      # row stride 2n
    out = ops.slerp_rows(a, b, 0.0, fract_rows=fr.cuda()).cpu()
    for r in range(6):
        assert torch.equal(out[r], mixing.interpolate_spherical(big0[r, 1], big1[r, 0], float(fr[r])))


def test_slerp_endpoints_and_empty():
    from latentblending_b200 import ops, utils
    g = torch.Generator().manual_seed(5)
    p0 = torch.randn(1, 4, 16, 16, generator=g).half().cuda()
    p1 = torch.randn(1, 4, 16, 16, generator=g).half().cuda()
    # f=0 -> p0, f=1 -> p1 up to the 1e-7 clamp (<= 1 fp16 ulp)
    assert (utils.interpolate_spherical(p0, p1, 0.0).float() - p0.float()).abs().max() <= 2e-3
    assert (utils.interpolate_spherical(p0, p1, 1.0).float() - p1.float()).abs().max() <= 2e-3
    e = torch.empty(0, 64, dtype=torch.float16, device="cuda")
    assert ops.slerp_rows(e, e, 0.5).shape == (0, 64)


def test_lerp_vs_oracle():
    from latentblending_b200 import utils
    from oracle import mixing
    z = np.load(os.path.join(GOLD, "slerp.npz"))
    a, b = torch.from_numpy(z["lin_a"]), torch.from_numpy(z["lin_b"])
    assert torch.equal(utils.interpolate_linear(a.cuda(), b.cuda(), 0.3).cpu(), torch.from_numpy(z["lin_out"]))
    g = torch.Generator().manual_seed(9)
    for dt in (torch.float16, torch.float32):
        x, y = torch.randn(1, 77, 2048, generator=g).to(dt), torch.randn(1, 77, 2048, generator=g).to(dt)
        for f in (0.0, 0.5, 0.8125, 1.0):
            assert torch.equal(utils.interpolate_linear(x.cuda(), y.cuda(), f).cpu(),
                               mixing.interpolate_linear(x, y, f))


@pytest.mark.parametrize("turbo", [False, True])
@pytest.mark.parametrize("hw", [16, 64, 128, 9])
def test_cfg_euler_step_bit_exact(turbo, hw):
    from latentblending_b200 import ops
    from oracle.schedulers import EulerAncestralDiscrete, EulerDiscrete
    sched = EulerAncestralDiscrete() if turbo else EulerDiscrete()
    N = 4 if turbo else 30
    sched.set_timesteps(N)
    g = torch.Generator().manual_seed(hw + turbo)
    for i in ([0, 1, 3] if turbo else [0, 7, 15, 29]):
        x = (torch.randn(1, 4, hw, hw, generator=g) * float(sched.sigmas[i] + 1)).half()
        eps = torch.randn(2, 4, hw, hw, generator=g).half()
        noise = torch.randn(1, 4, hw, hw, generator=g).half() if turbo else None
        gsc = np.float64(3.37)
        # oracle, op by op (oracle/holder.py loop body)
        x_in_ref = sched.scale_model_input(torch.cat([x] * 2), i)
        e_u, e_t = eps.chunk(2)
        e = e_u + gsc * (e_t - e_u)
        ref = sched.step(e, i, x, noise=noise)
        ref_nocfg = sched.step(eps[:1], i, x, noise=noise)
        # CUDA
        sigma = sched.sigmas[i]
        h = lambda v: float(v.half())      # 0-dim CUDA-tensor scalars reach the fp16 ops rounded to fp16
        div = h((sigma ** 2 + 1) ** 0.5)
        x_in = ops.scale_model_input(x.cuda(), 2, div).cpu()
        assert torch.equal(x_in, x_in_ref)
        if turbo:
            s_up, s_down = sched.sigma_up_down(i)
            dt, sup = h(s_down - sigma), h(s_up)
        else:
            dt, sup = h(sched.sigmas[i + 1] - sigma), 0.0
        traj = torch.empty_like(x).cuda()
        out = ops.cfg_euler_step(x.cuda(), eps.cuda(), gsc, h(sigma), dt, sup,
                                 noise=None if noise is None else noise.cuda(), traj=traj).cpu()
        assert torch.equal(out, ref), f"step {i}: {(out != ref).sum().item()} mismatches"
        assert torch.equal(traj.cpu(), ref)
        out1 = ops.cfg_euler_step(x.cuda(), eps[:1].contiguous().cuda(), 0.0, h(sigma), dt, sup,
                                  noise=None if noise is None else noise.cuda()).cpu()
        assert torch.equal(out1, ref_nocfg)


def test_slerp_certified_fp32_path_equals_exact_fp64_path(monkeypatch):
    """K1 pass 2 evaluates p0*s0 + p1*s1 in split-weight fp32 and certifies the fp16 rounding, falling back to the
    reference's fp64 arithmetic per element (csrc/mix_kernels.cuh).  A/B it against the all-fp64 evaluation
    (LB_SLERP_EXACT=1) on adversarial value families, and against the oracle."""
    from latentblending_b200 import ops
    from oracle import mixing
    g = torch.Generator().manual_seed(11)
    n = 4 * 128 * 128
    fam = []
    a, b = torch.randn(n, generator=g), torch.randn(n, generator=g)
    fam.append((a, b))                                             # typical latents
    fam.append((a * 3e-6, b * 3e-6))                               # fp16 subnormals in and out
    fam.append((a * 9000, b * 9000))                               # near the fp16 overflow threshold
    fam.append((a, a.clone()))                                     # identical rows (dot clamp)
    fam.append((a, -a * 1.0009765625))                             # near-antipodal: heavy cancellation
    z = a.clone(); z[torch.rand(n, generator=g) < 0.75] = 0
    fam.append((z, b * (torch.rand(n, generator=g) < 0.5)))        # exact zeros
    e = torch.randint(-20, 10, (n,), generator=g).float()
    fam.append((a * torch.exp2(e), b * torch.exp2(e.flip(0))))     # 30 binades of magnitude
    fam.append((a * 0.01, b * 100))
    p0 = torch.stack([f[0] for f in fam]).half()
    p1 = torch.stack([f[1] for f in fam]).half()
    for fract in (0.0, 0.25, 0.5, 0.8137, 1.0):
        monkeypatch.delenv("LB_SLERP_EXACT", raising=False)
        fast = ops.slerp_rows(p0.cuda(), p1.cuda(), fract).cpu()
        monkeypatch.setenv("LB_SLERP_EXACT", "1")
        exact = ops.slerp_rows(p0.cuda(), p1.cuda(), fract).cpu()
        monkeypatch.delenv("LB_SLERP_EXACT", raising=False)
        assert torch.equal(fast.view(torch.int16), exact.view(torch.int16)), \
            f"fract {fract}: {(fast.view(torch.int16) != exact.view(torch.int16)).sum().item()} mismatches"
        for r in (0, 2, 6):
            ref = mixing.interpolate_spherical(p0[r], p1[r], fract)
            assert torch.equal(fast[r].view(torch.int16), ref.view(torch.int16)), f"row {r} fract {fract}"
