"""Round-2 CPU tests: the adaptive ODE solver, the oracle's switchable judgement calls, and the pin of the
reference-loop golden (replayed from the rasteriser calls the unmodified reference gs_surfel.py made)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from tests.helpers import cameras, oracle_view, rel_l2, scene

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dopri5_is_adaptive_with_dense_output():
    """ADVICE (medium): the solver must not be clamped to the output grid.  The reference calls
    sample_ode(num_steps=250) with dopri5 (flow_matching_trainer.py:715): tens of steps, not >= 249 x 6 NFE."""
    from gaussiananything_b200.transport.integrators import odeint
    n = [0]

    def f(t, y):
        n[0] += 1
        return -y * (1 + torch.sin(5 * t))

    y0 = torch.tensor([1.0, 2.0, -0.5], dtype=torch.float64)
    ts = torch.linspace(0, 1, 250, dtype=torch.float64)
    ys = odeint(f, y0, ts, method="dopri5", atol=1e-6, rtol=1e-3)
    exact = y0 * torch.exp(-(ts[:, None] + (1 - torch.cos(5 * ts[:, None])) / 5))
    assert ys.shape == (250, 3) and torch.equal(ys[0], y0)
    assert n[0] < 120, n[0]
    assert float((ys - exact).abs().max()) < 3e-3
    n[0] = 0
    ys = odeint(f, y0, ts, method="dopri5", atol=1e-10, rtol=1e-8)
    assert float((ys - exact).abs().max()) < 1e-6 and n[0] < 2500
    # grid states come from the interpolant: a coarser output grid does not change the steps taken
    n[0] = 0
    odeint(f, y0, ts[::83], method="dopri5", atol=1e-6, rtol=1e-3)
    coarse = n[0]
    n[0] = 0
    odeint(f, y0, ts, method="dopri5", atol=1e-6, rtol=1e-3)
    assert n[0] == coarse


def test_dopri5_raises_instead_of_spinning():
    from gaussiananything_b200.transport.integrators import odeint
    y0 = torch.ones(3, dtype=torch.float64)
    ts = torch.linspace(0, 1, 5, dtype=torch.float64)
    with pytest.raises(RuntimeError):
        odeint(lambda t, y: y * float("nan"), y0, ts, method="dopri5")
    with pytest.raises(RuntimeError):                                    # blows up at t = 0.5: step size underflows
        odeint(lambda t, y: 1.0 / (0.5 - t).clamp_min(0.0) ** 2 * torch.ones_like(y), y0, ts, method="dopri5")


def test_sampler_default_method_is_dopri5_and_cheap():
    from gaussiananything_b200 import transport as tr
    s = tr.Sampler(tr.create_transport("GVP", "velocity", None, None, None, "lognorm"))
    n = [0]

    def model(x, t, **kw):
        n[0] += 1
        return -x + t.reshape(-1, 1, 1)

    x = torch.randn(2, 16, 3, dtype=torch.float64)
    traj = s.sample_ode(num_steps=250)(x, model)
    assert traj.shape == (250, 2, 16, 3) and n[0] < 200
    want = s.sample_ode(sampling_method="rk4", num_steps=250)(x, model)[-1]
    assert float((traj[-1] - want).abs().max()) < 1e-3


@pytest.mark.parametrize("radius_formula,quat_norm_grad", [(0, 0), (1, 0), (0, 1), (1, 1)])
def test_oracle_variants_match_torch_autograd(radius_formula, quat_norm_grad):
    """Both settings of the two switchable judgement calls: C oracle == fp64 autograd of the torch restatement."""
    from oracle import surfel_oracle as so
    from oracle import surfel_torch as st
    P, H, W = 120, 40, 48
    g = scene(P, 3, 40.0, 0.004, 0.09)
    g[:, 6:10] *= np.linspace(0.6, 1.7, P, dtype=np.float32)[:, None]            # non-unit quaternions
    vs, ps, _, _ = cameras(1, start=3)
    bg = [1.0, 0.5, 0.2]
    try:
        so.set_variant(radius_formula, quat_norm_grad)
        assert so.get_variant() == (radius_formula, quat_norm_grad)
        st.RADIUS_FORMULA, st.QUAT_NORM_GRAD = radius_formula, quat_norm_grad
        o = oracle_view(g, vs[0], ps[0], bg, H, W)
        T = lambda a: torch.tensor(a, dtype=torch.float64, requires_grad=True)
        m, op, sc, ro, co = T(g[:, 0:3]), T(g[:, 3:4]), T(g[:, 4:6]), T(g[:, 6:10]), T(g[:, 10:13])
        color, radii, allmap = st.rasterize(m, op, sc, ro, co, torch.tensor(vs[0], dtype=torch.float64),
                                            torch.tensor(ps[0], dtype=torch.float64), torch.tensor(bg), H, W)
        assert np.array_equal(radii.numpy(), o["radii"])
        assert rel_l2(o["color"], color.detach().numpy()) < 1e-5
        rng = np.random.default_rng(0)
        gc, ga = rng.standard_normal((3, H, W)), rng.standard_normal((7, H, W))
        ((color * torch.tensor(gc)).sum() + (allmap * torch.tensor(ga)).sum()).backward()
        b = so.rasterize_backward(o, gc, ga)
        for k, t in [("means3D", m), ("opacities", op), ("scales", sc), ("rotations", ro), ("colors", co)]:
            want = t.grad.numpy()
            if k == "rotations" and not quat_norm_grad:
                # variant 0 restates upstream's quat_to_rotmat_vjp: the vjp at q/|q| returned as is (no 1/|q| factor);
                # autograd with a detached normalisation factor carries that factor
                want = want * np.linalg.norm(g[:, 6:10].astype(np.float64), axis=1, keepdims=True)
            assert rel_l2(b[k], want) < 2e-4, k
        if quat_norm_grad:
            assert np.abs((b["rotations"] * g[:, 6:10]).sum(1)).max() < 1e-6 * max(1.0, np.abs(b["rotations"]).max())
    finally:
        so.set_variant(0, 0)
        st.RADIUS_FORMULA, st.QUAT_NORM_GRAD = 0, 0
    if radius_formula:
        o0 = oracle_view(g, vs[0], ps[0], bg, H, W)
        assert (o["radii"] >= o0["radii"]).all() and o["num_rendered"] >= o0["num_rendered"]


def test_reference_loop_golden_reproduces_from_the_unmodified_reference_file():
    """gs_surfel_loop.npz is the unmodified reference gs_surfel.py run over the C oracle behind a rasteriser shim.  Its
    inputs must still come out of tools/synth.py, and every rasteriser call the reference's loop made (recorded in
    gs_surfel_loop_calls.json with digests of what it got back, of which the golden is the reference's own
    post-processing) must still come out of the oracle bit for bit."""
    from tests.golden import make_gs_surfel_golden as mk
    gold = np.load(mk.OUT)
    g, cam = mk.cases()
    assert np.array_equal(g, gold["g"]) and np.float32(cam["tanfov"]) == gold["tanfov"]
    for k in ("view", "proj", "pos"):
        assert np.array_equal(cam[k], gold[k]), k
    with open(mk.CALLS) as f:
        calls = json.load(f)
    assert len(calls) == 2 * 3 + 1 * 2                           # the golden's two renders: B x V = 2 x 3 and 1 x 2
    for i, c in enumerate(calls):
        b, v, n = c["item"], c["view"], c["size"]
        o = oracle_view(gold["g"][b], gold["view"][b, v], gold["proj"][b, v], np.float32(c["bg"]), n, n, c["scale_modifier"])
        for k, want in c["sha256"].items():
            assert mk.digest(o[k]) == want, (i, k)


def test_scene_builders_do_not_need_the_oracle():
    """bench.py's GPU arm builds its inputs from tools/synth.py: importing it must not load the CPU checker."""
    code = ("import sys; sys.path.insert(0, %r); import tools.synth, tests.helpers; "
            "assert not any(m.startswith('oracle') for m in sys.modules), [m for m in sys.modules if m.startswith('oracle')]" % ROOT)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


def test_gemm_tile_width_rule_matches_the_committed_sweep():
    """dit._gemm_config (host logic, no GPU needed) against profiles/r02_gemm_sweep.txt: on every swept DiT shape the width it
    picks is within 3 % of the fastest single-CTA configuration that was measured, and HEADS epilogues stay 128 wide."""
    import os
    import re
    from gaussiananything_b200 import dit
    path = os.path.join(os.path.dirname(__file__), "..", "profiles", "r02_gemm_sweep.txt")
    rows = [l for l in open(path) if l.startswith("M=")]
    assert len(rows) == 9
    for line in rows:
        M, N, K = (int(v) for v in re.match(r"M=(\d+) N=(\d+) K=(\d+)", line).groups())
        us = {int(c): float(t) for c, t in re.findall(r"(\d+):\s+([\d.]+)us", line.split("|", 1)[1])}
        single = {c: t for c, t in us.items() if c in (128, 192, 256)}
        pick = dit._gemm_config(M, N, dit.EPI_BF16)
        assert pick in single, (M, N, pick)
        assert single[pick] <= 1.03 * min(single.values()), (M, N, K, pick, single)
        assert dit._gemm_config(M, N, dit.EPI_HEADS) == 128
