"""CPU tests: pin the oracle (oracle/isdf_oracle.py) against the golden vectors produced by
the unmodified reference (tests/golden/*.pt), and the two oracle formulations against each other."""
import math
import os

import pytest
import torch

from oracle import isdf_oracle as O
from tests.golden import common as C

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def load(name):
    return torch.load(os.path.join(GOLD, name), weights_only=False)


def test_pe_matches_reference_golden():
    gold = load("pe.pt")
    x = (torch.rand(64, 3, generator=C.gen(11)) - 0.5) * torch.tensor([12.0, 4.0, 12.0])
    e = O.pe_encode(x, 0.05937489, 6, None)
    assert e.shape == (64, 255)
    assert torch.allclose(e, gold["plain"], atol=2e-6, rtol=0)
    e = O.pe_encode(x, 0.05937489, 6, C.rigid_transform(5))
    assert torch.allclose(e, gold["rigid"], atol=4e-6, rtol=0)
    e = O.pe_encode(x, 0.04, 9, None)
    assert e.shape == (64, 381)
    assert torch.allclose(e, gold["deg8"], atol=2e-5, rtol=0)


def test_pe_known_answers():
    # SURVEY.md 8c KATs (recorded from the reference)
    e = O.pe_encode(torch.tensor([[1.0, -2.0, 3.0]]), 0.05937489, 6)[0]
    assert torch.allclose(e[:3], torch.tensor([0.05937489, -0.11874978, 0.17812467]), atol=1e-7)
    assert torch.allclose(e[3:9], torch.tensor([0.14365424, 0.28432849, 0.54518676, 0.91407603,
                                                0.74139392, -0.99505454]), atol=2e-6)
    assert abs(float(e.sum()) - 63.66688783) < 2e-4


def test_softplus_kats():
    z = torch.tensor([0.0, -0.05, 0.21])
    sp = O.softplus100(z)
    assert torch.allclose(sp, torch.tensor([0.00693147, 6.7153e-05, 0.21]), atol=1e-7)


@pytest.mark.parametrize("tag,seed,gain,tr", [("g1", 21, 1.0, None), ("g2_rigid", 22, 2.0, 6)])
def test_sdf_and_input_gradient_match_reference(tag, seed, gain, tr):
    gold = load("sdfmap.pt")[tag]
    sd = C.golden_weights(seed, gain=gain)
    layers = O.layers_from_state_dict(sd, 2)
    cfg = O.default_cfg(transform=C.rigid_transform(tr) if tr else None)
    x = ((torch.rand(96, 3, generator=C.gen(12)) - 0.5) * torch.tensor([12.0, 4.0, 12.0])).requires_grad_(True)
    sdf = O.sdf_forward(layers, x, cfg)
    (g,) = torch.autograd.grad(sdf, x, torch.ones_like(sdf))
    scale = gold["sdf"].abs().max()
    assert (sdf - gold["sdf"]).abs().max() / scale < 2e-6
    assert (g - gold["grad"]).abs().max() / gold["grad"].abs().max() < 2e-5


def test_sampling_matches_reference():
    gold = load("sample.pt")
    F, H, W = 3, 32, 48
    depth = torch.stack([C.synthetic_depth(k, H, W, invalid_frac=0.15) for k in range(F)])
    T = torch.stack([C.synthetic_pose(k) for k in range(F)])
    nrm = torch.stack([C.synthetic_normals(H, W, 0.1, 40 + k) for k in range(F)])
    cam = dict(fx=40.0, fy=42.0, cx=23.5, cy=15.5)
    s = O.sample_rays(depth, T, nrm, gold["ib"], gold["ih"], gold["iw"], gold["u"], gold["n_near"],
                      cam, 0.07, 0.1, 19, 8)
    assert torch.equal(s["indices_b"], gold["ib2"])
    assert torch.equal(s["indices_h"], gold["ih2"])
    assert torch.equal(s["indices_w"], gold["iw2"])
    assert torch.equal(s["depth_sample"], gold["depth"])
    assert torch.allclose(s["dirs_C_sample"], gold["dirs_C"], atol=1e-7)
    assert torch.equal(s["norm_sample"], gold["norm"])
    assert torch.allclose(s["z_vals"], gold["z"], atol=1e-6)
    assert torch.allclose(s["pc"], gold["pc"], atol=2e-6)
    assert gold["z"].shape[1] == 27 and gold["z"].shape[0] < 150   # some rays were dropped


CASES = [("c1", 31, 1.0, None, 48, 0.25, "L1"),
         ("c2_rigid_gain2", 32, 2.0, 9, 40, 0.04, "L1"),
         ("c3_L2", 33, 1.5, None, 24, 0.0, "L2")]


def _case(tag, seed, gain, tr, R, nstd, lt, dtype=torch.float32):
    sd = C.golden_weights(seed, gain=gain)
    layers = [(w.to(dtype), b.to(dtype)) for w, b in O.layers_from_state_dict(sd, 2)]
    cfg = O.default_cfg(noise_std=nstd, loss_type=lt,
                        transform=C.rigid_transform(tr) if tr else None)
    batch, noise = C.loss_batch(seed + 100, R)
    batch = {k: v.to(dtype) for k, v in batch.items()}
    return layers, batch, noise.to(dtype), cfg, sd


def _check_against_gold(out, gold, sd, tol_sdf, tol_g, tol_gw):
    assert (out["sdf"] - gold["sdf"]).abs().max() / gold["sdf"].abs().max() < tol_sdf
    assert (out["g"] - gold["grad"]).abs().max() / gold["grad"].abs().max() < tol_g
    tm = out["terms"]["total_mat"]
    assert (tm - gold["total_mat"]).abs().max() / gold["total_mat"].abs().max() < 5e-5
    for k, v in gold["losses"].items():
        assert abs(float(out["losses"][k]) - v) <= 2e-5 * max(1.0, abs(v)), k
    names = list(sd.keys())
    for name, gr in zip(names, out["grads"]):
        nref = float(gold["grad_norm"][name])
        assert abs(float(gr.double().norm()) - nref) <= tol_gw * nref + 1e-9, name
        sub = C.subsample(gr) if gr.numel() > 4096 else gr
        err = (sub.double() - gold["grad_sub"][name].double()).norm() / (gold["grad_sub"][name].double().norm() + 1e-12)
        assert err < tol_gw, (name, float(err))


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_autograd_formulation_matches_reference(case):
    gold = load("step.pt")[case[0]]
    layers, batch, noise, cfg, sd = _case(*case)
    out = O.step_autograd(layers, batch, cfg, noise)
    _check_against_gold(out, gold, sd, 2e-6, 2e-5, 2e-4)


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_sweep_formulation_matches_reference(case):
    gold = load("step.pt")[case[0]]
    layers, batch, noise, cfg, sd = _case(*case, dtype=torch.float64)
    cfg = dict(cfg)
    if cfg.get("transform") is not None:
        cfg["transform"] = cfg["transform"].double()
    out = O.step_sweeps(layers, batch, cfg, noise)
    # fp64 restatement vs the reference's fp32 run: the gap is the reference's own rounding noise
    _check_against_gold(out, gold, sd, 5e-6, 1e-4, 5e-4)


PC_CASES = [("p1", 61, 1.0, None, 48, 0.25, "L1"), ("p2_rigid_L2", 62, 1.5, 9, 32, 0.0, "L2")]


def _case_pc(tag, seed, gain, tr, R, nstd, lt, dtype=torch.float32):
    layers, _, _, cfg, sd = _case(tag, seed, gain, tr, R, nstd, lt, dtype)
    batch, noise = C.loss_batch_pc(seed + 100, R)
    cfg = dict(cfg, bounds_method="pc")
    if dtype == torch.float64 and cfg.get("transform") is not None:
        cfg["transform"] = cfg["transform"].double()
    return layers, {k: v.to(dtype) for k, v in batch.items()}, noise.to(dtype), cfg, sd


@pytest.mark.parametrize("case", PC_CASES, ids=[c[0] for c in PC_CASES])
def test_bounds_pc_matches_reference(case):
    """Row N2: the batch-distance bound and its direction field against loss.bounds_pc (loss.py:56-89)."""
    gold = load("step_pc.pt")[case[0]]
    _, batch, _, cfg, _ = _case_pc(*case)
    bnd, vec = O.bounds_pc(batch["pc"], batch["z_vals"], batch["depth_sample"])
    assert torch.allclose(bnd, gold["bounds"], atol=1e-6, rtol=1e-6)
    nan_gold = gold["grad_vec"][..., 0].isnan()
    assert torch.equal(vec[..., 0].isnan(), nan_gold) and int(nan_gold.sum()) == 1
    assert torch.allclose(vec[~nan_gold], gold["grad_vec"][~nan_gold], atol=2e-6)


@pytest.mark.parametrize("case", PC_CASES, ids=[c[0] for c in PC_CASES])
def test_pc_bound_step_matches_reference(case):
    gold = load("step_pc.pt")[case[0]]
    layers, batch, noise, cfg, sd = _case_pc(*case)
    _check_against_gold(O.step_autograd(layers, batch, cfg, noise), gold, sd, 2e-6, 2e-5, 2e-4)
    layers, batch, noise, cfg, sd = _case_pc(*case, dtype=torch.float64)
    _check_against_gold(O.step_sweeps(layers, batch, cfg, noise), gold, sd, 5e-6, 1e-4, 5e-4)


def test_sweeps_equal_autograd_fp64():
    layers, batch, noise, cfg, sd = _case("c2", 32, 2.0, 9, 40, 0.04, "L1", dtype=torch.float64)
    cfg = dict(cfg, transform=cfg["transform"].double())
    a = O.step_autograd(layers, batch, cfg, noise)
    s = O.step_sweeps(layers, batch, cfg, noise)
    assert (a["sdf"] - s["sdf"]).abs().max() < 1e-12
    assert (a["g"] - s["g"]).abs().max() < 1e-12
    for ga, gs in zip(a["grads"], s["grads"]):
        assert (ga - gs).abs().max() <= 1e-10 * max(1.0, float(ga.abs().max()))


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_frame_avg_matches_reference(case):
    gold = load("step.pt")[case[0]]
    la, fa = O.frame_avg(gold["total_mat"], (4, 16, 24), gold["frame_ib"], gold["frame_ih"], gold["frame_iw"], 8)
    assert torch.allclose(la, gold["loss_approx"], atol=1e-6)
    assert torch.allclose(fa, gold["frame_avg"], atol=1e-6)


def test_adamw_matches_torch():
    gold = load("adamw.pt")["traj"]
    g = C.gen(51)
    p = torch.randn(1000, generator=g)
    m = torch.zeros_like(p)
    v = torch.zeros_like(p)
    for it in range(3):
        gr = torch.randn(1000, generator=g) * 0.01
        p, m, v = O.adamw_update(p, gr, m, v, it + 1, 0.0013, 0.012)
        assert torch.allclose(p, gold[it], atol=1e-6, rtol=1e-6)


LOSS_SETTINGS = [   # (id, n_freqs, block, cfg overrides, batch kind): the settings tests/test_gpu_zz_train_geometry.py uses
    ("orien_loss", 6, 2, dict(orien_loss=True), "ray"),
    ("grad_weight_0", 6, 2, dict(grad_weight=0.0), "ray"),
    ("eik_weight_0", 6, 2, dict(eik_weight=0.0), "ray"),
    ("grad_and_eik_0", 6, 2, dict(grad_weight=0.0, eik_weight=0.0), "ray"),
    ("franka_E465_b3", 11, 3, dict(trunc_weight=30.0, trunc_distance=0.1, noise_std=0.025, dist_behind_surf=0.01), "franka"),
    ("scale_input_0.4_E381", 9, 2, dict(scale_input=0.4), "ray"),
    ("pc_bound_E381", 9, 2, dict(bounds_method="pc"), "pc"),
]


@pytest.mark.parametrize("tag,n_freqs,block,over,kind", LOSS_SETTINGS, ids=[s[0] for s in LOSS_SETTINGS])
def test_oracle_formulations_agree_at_every_loss_setting(tag, n_freqs, block, over, kind):
    """The closed-form adjoints of step_sweeps (orien_loss, switched-off terms, franka truncation, large PE arguments,
    the 'pc' bound) equal autograd of the reference formulation in fp64.  grad_weight 0 runs without normals, as the
    Trainer does."""
    cfg = O.default_cfg(n_freqs=n_freqs, block=block, n_strat=8, n_surf=8, **dict(dict(noise_std=0.08), **over))
    sd = C.golden_weights(7, E=3 + 42 * n_freqs, block=block, gain=1.2)
    layers = [(w.double(), b.double()) for w, b in O.layers_from_state_dict(sd, block)]
    if kind == "pc":
        batch, noise = C.loss_batch_pc(19, 6, S=16)
    else:
        batch, noise = C.loss_batch(19, 6, S=16, dist_behind=cfg["dist_behind_surf"])
    batch = {k: v.double() for k, v in batch.items()}
    if cfg["grad_weight"] == 0:
        batch["norm_sample"] = None
    a = O.step_autograd(layers, batch, cfg, noise.double())
    s = O.step_sweeps(layers, batch, cfg, noise.double())
    assert (a["sdf"] - s["sdf"]).abs().max() < 1e-12 and (a["g"] - s["g"]).abs().max() < 1e-12
    assert set(a["losses"]) == set(s["losses"])
    assert ("grad_loss" in s["losses"]) == (cfg["grad_weight"] != 0)
    assert ("eikonal_loss" in s["losses"]) == (cfg["eik_weight"] != 0)
    for k in a["losses"]:
        assert abs(float(a["losses"][k] - s["losses"][k])) <= 1e-12 * max(1.0, abs(float(a["losses"][k]))), k
    for ga, gs in zip(a["grads"], s["grads"]):
        assert float(ga.abs().max()) > 0
        assert (ga - gs).abs().max() <= 1e-10 * max(1.0, float(ga.abs().max()))


def test_step_sweeps_is_device_generic():
    """step_sweeps builds every constant on the device of its inputs (the GPU tests run the fp64 oracle there): on a
    'meta' batch it must get through without touching a CPU tensor."""
    cfg = O.default_cfg(noise_std=0.08, n_strat=8, n_surf=8, transform=C.rigid_transform(9).double())
    sd = C.golden_weights(7)
    batch, noise = C.loss_batch(19, 4, S=16)
    meta = torch.device("meta")
    layers = [(w.double().to(meta), b.double().to(meta)) for w, b in O.layers_from_state_dict(sd, 2)]
    b = {k: v.double().to(meta) for k, v in batch.items()}
    out = O.step_sweeps(layers, b, dict(cfg, transform=cfg["transform"].to(meta)), noise.double().to(meta))
    assert out["sdf"].device == meta and all(g.device == meta for g in out["grads"])


@pytest.mark.parametrize("n_freqs,block,tr,scale_input", [(6, 2, None, 0.05937489), (6, 3, 9, 0.05937489),
                                                          (9, 2, 9, 0.4), (11, 3, 5, 0.05937489)])
def test_sdf_and_grad_equals_step_sweeps_fp64(n_freqs, block, tr, scale_input):
    """sdf_and_grad (autograd over sdf_forward; the oracle of the forward-only and input-gradient programs) equals the
    sdf and g of the explicit sweeps, with noise, a rigid PE transform and a large scale_input."""
    cfg = O.default_cfg(n_freqs=n_freqs, block=block, noise_std=0.3, scale_input=scale_input,
                        transform=C.rigid_transform(tr).double() if tr else None, n_strat=8, n_surf=8)
    sd = C.golden_weights(13, E=O.embedding_size(n_freqs), block=block, gain=1.2)
    layers = [(w.double(), b.double()) for w, b in O.layers_from_state_dict(sd, block)]
    batch, noise = C.loss_batch(23, 5, S=16)
    batch = {k: v.double() for k, v in batch.items()}
    ref = O.step_sweeps(layers, batch, cfg, noise.double())
    sdf, g = O.sdf_and_grad(layers, batch["pc"], cfg, noise.double())
    assert sdf.shape == (5, 16) and g.shape == (5, 16, 3) and sdf.dtype == torch.float64
    assert float((sdf - ref["sdf"]).abs().max()) < 1e-12 and float((g - ref["g"]).abs().max()) < 1e-12
    sdf0, g0 = O.sdf_and_grad(layers, batch["pc"], cfg)               # noise shifts sdf only
    assert torch.allclose(sdf - sdf0, noise.double() * 0.3 * cfg["scale_output"], rtol=0, atol=1e-12)
    assert torch.equal(g, g0)


@pytest.mark.parametrize("tag,seed,gain,tr", [("g1", 21, 1.0, None), ("g2_rigid", 22, 2.0, 6)])
def test_sdf_and_grad_matches_reference(tag, seed, gain, tr):
    gold = load("sdfmap.pt")[tag]
    sd = C.golden_weights(seed, gain=gain)
    for dt, tol_s, tol_g in ((torch.float32, 2e-6, 2e-5), (torch.float64, 5e-6, 1e-4)):
        layers = [(w.to(dt), b.to(dt)) for w, b in O.layers_from_state_dict(sd, 2)]
        cfg = O.default_cfg(transform=C.rigid_transform(tr).to(dt) if tr else None)
        x = ((torch.rand(96, 3, generator=C.gen(12)) - 0.5) * torch.tensor([12.0, 4.0, 12.0])).to(dt)
        sdf, g = O.sdf_and_grad(layers, x, cfg)
        assert float((sdf - gold["sdf"]).abs().max() / gold["sdf"].abs().max()) < tol_s
        assert float((g - gold["grad"]).abs().max() / gold["grad"].abs().max()) < tol_g


def test_sdf_and_grad_is_device_generic():
    meta = torch.device("meta")
    cfg = O.default_cfg(n_freqs=9, transform=C.rigid_transform(9).double().to(meta))
    sd = C.golden_weights(7, E=O.embedding_size(9))
    layers = [(w.double().to(meta), b.double().to(meta)) for w, b in O.layers_from_state_dict(sd, 2)]
    x = torch.empty(4, 7, 3, dtype=torch.float64, device=meta)
    sdf, g = O.sdf_and_grad(layers, x, cfg, torch.empty(4, 7, dtype=torch.float64, device=meta))
    assert sdf.device == meta and g.device == meta and sdf.shape == (4, 7) and g.shape == (4, 7, 3)


@pytest.mark.parametrize("n_freqs,hidden,block", [(6, 512, 4), (9, 256, 2), (11, 256, 3)])
def test_oracle_formulations_agree_at_other_model_shapes(n_freqs, hidden, block):
    """The shapes of BASELINE configs[4] and of the realsense / franka configs (SURVEY.md appendix A): the explicit
    sweeps equal autograd in fp64 there too (they are the oracle of tests/test_gpu_zz_shapes.py)."""
    cfg = O.default_cfg(n_freqs=n_freqs, hidden=hidden, block=block, noise_std=0.05, n_strat=8, n_surf=8)
    sd = C.golden_weights(5, E=3 + 42 * n_freqs, H=hidden, block=block, gain=1.2)
    layers = [(w.double(), b.double()) for w, b in O.layers_from_state_dict(sd, block)]
    batch, noise = C.loss_batch(9, 6, S=16)
    batch = {k: v.double() for k, v in batch.items()}
    a = O.step_autograd(layers, batch, cfg, noise.double())
    s = O.step_sweeps(layers, batch, cfg, noise.double())
    assert len(a["grads"]) == 2 * (2 * block + 3)
    assert (a["sdf"] - s["sdf"]).abs().max() < 1e-12 and (a["g"] - s["g"]).abs().max() < 1e-12
    for ga, gs in zip(a["grads"], s["grads"]):
        assert (ga - gs).abs().max() <= 1e-10 * max(1.0, float(ga.abs().max()))
