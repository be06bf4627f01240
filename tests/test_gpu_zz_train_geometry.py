"""GPU parity of the fused training step (isdfb_train_fwd_bwd) where the launch plan and the loss settings change, and
of the fast-mode Trainer step (one CUDA graph) on the batch it actually drew -- all against the fp64 oracle, run on
the device in ray chunks.

* Launch geometry: the tensor-core dispatcher (tc_train, isdf_b200/csrc/tc_path.cu) runs each max_points chunk as one
  tile per CTA, as two waves with the first wave's weight gradients on a side stream, or with persistent CTAs that
  loop over several tiles.  Every case states the plan it exercises and asserts it with chunk_plan().
* Loss settings: orien_loss, grad_weight 0 (no normals), eik_weight 0, the franka truncation parameters, a large
  scale_input, the 'pc' bound at a wide embedding, and masked rays carrying what the fused sampler writes for them.
* Fast-mode Trainer step: gradient, loss means, loss matrix and the per-keyframe loss write-back of the replayed graph.

(The file name sorts after the default-shape suites on purpose.)"""
import json
import os

import pytest
import torch

from oracle import isdf_oracle as O
from tests.golden import common as C
from tests.golden import trainer_case as TC
from tests import parity as P
from tests.test_gpu_engine import MODES, TOL

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
TILE = 128                      # points per tensor-core tile (TC_TILE)
GW_SAMPLES = 20000              # batches at least this large use TOL gw, smaller ones gw_small (kink flips ~ 1/N)
PARITY_MODES = [m for m in ("fp32", "bf16x3", "bf16x3g") if m in MODES]
TC_MODES = [m for m in ("bf16x3", "bf16x3g") if m in MODES]
CHUNK_INVARIANCE = {"fp32": 1e-6, "bf16x3": 5e-5, "bf16x3g": 5e-5}     # sdf bound of test_train_properties_full_size


def num_sms():
    return torch.cuda.get_device_properties(DEV).multi_processor_count


def n_dw_jobs(E, block):
    """Weight-gradient jobs of the tensor-core path: two row halves of each 256x256 unit -- the 2*block+2 hidden
    layers, the concat layer's embedding part, and the second embedding halves of layer 0 and the concat layer when
    the padded embedding is wider than 256."""
    return 2 * ((2 * block + 2) + 1 + (2 if E > 256 else 0))


def chunk_plan(n, cap, sms, n_jobs):
    """The launch plan tc_train picks for an n-point batch: one entry per max_points chunk (the engine rounds the
    cap up to whole tiles) with its points, tiles, branch and the grid of the wave-1 weight-gradient launch.
      'single'      tiles <= sms            one tile per CTA, then one dW launch
      'two_wave'    sms < tiles < 2 sms     wave 1 (sms tiles), its dW on a side stream with
                                            grid max(sms - rest, n_jobs) under wave 2 (rest tiles), then wave 2's dW
      'persistent'  tiles >= 2 sms          sms CTAs, several tiles per CTA, then one dW launch"""
    cap = -(-cap // TILE) * TILE
    plan = []
    for p0 in range(0, n, cap):
        nc = min(cap, n - p0)
        tiles = -(-nc // TILE)
        grid = None
        if tiles <= sms:
            branch = "single"
        elif tiles < 2 * sms:
            branch, grid = "two_wave", max(sms - (tiles - sms), n_jobs)
        else:
            branch = "persistent"
        plan.append(dict(points=nc, tiles=tiles, branch=branch, dw_grid=grid))
    return plan


# ------------------------------------------------------------------------------------------ oracle on the device
def _to_dev(batch, dtype):
    return {k: (v.to(device=DEV, dtype=dtype) if v is not None else None) for k, v in batch.items()}


def _oracle_once(sd, batch, noise, cfg, dtype, chunk_points):
    """step_sweeps over ray chunks; each chunk's gradient and loss means weighted by its share of the rays (the loss
    is a mean over samples and every ray has S samples).  The 'pc' bound couples all rays: one chunk."""
    layers = [(w.to(device=DEV, dtype=dtype), b.to(device=DEV, dtype=dtype))
              for w, b in O.layers_from_state_dict(sd, cfg["block"])]
    cfg = dict(cfg)
    if cfg.get("transform") is not None:
        cfg["transform"] = cfg["transform"].to(device=DEV, dtype=dtype)
    b = _to_dev(batch, dtype)
    nz = noise.to(device=DEV, dtype=dtype) if (noise is not None and cfg["noise_std"]) else None
    R, S = b["z_vals"].shape
    ray_chunk = R if cfg.get("bounds_method", "ray") == "pc" else max(1, chunk_points // S)
    grads, losses, sdf, g, lm = None, {}, [], [], []
    for r0 in range(0, R, ray_chunk):
        sl = slice(r0, min(R, r0 + ray_chunk))
        out = O.step_sweeps(layers, {k: (v[sl] if v is not None else None) for k, v in b.items()}, cfg,
                            None if nz is None else nz[sl])
        w = (sl.stop - sl.start) / R
        part = [x * w for x in out["grads"]]
        grads = part if grads is None else [a + p for a, p in zip(grads, part)]
        for k, v in out["losses"].items():
            losses[k] = losses.get(k, 0.0) + w * float(v)
        sdf.append(out["sdf"].cpu()); g.append(out["g"].cpu()); lm.append(out["terms"]["total_mat"].cpu())
        del out
    return dict(sdf=torch.cat(sdf), g=torch.cat(g), loss_mat=torch.cat(lm), losses=losses,
                grads=[x.cpu() for x in grads])


def oracle(sd, batch, noise, cfg, chunk_points=65536):
    """fp64 result plus the 'floor': how far the same restatement in fp32 lands from it.  Tolerances are never
    tighter than 3x that floor (a large scale_input or 11 octaves make fp32 sin() itself lose digits)."""
    ref = _oracle_once(sd, batch, noise, cfg, torch.float64, chunk_points)
    r32 = _oracle_once(sd, batch, noise, cfg, torch.float32, chunk_points)
    ref["floor"] = dict(sdf=P.rel(r32["sdf"], ref["sdf"]), g=P.rel(r32["g"], ref["g"]),
                        loss_mat=P.rel(r32["loss_mat"], ref["loss_mat"]),
                        loss=max(abs(r32["losses"][k] - v) / max(abs(v), 1e-3) for k, v in ref["losses"].items()),
                        gw=max(P.rel_fro(a, b) for a, b in zip(r32["grads"], ref["grads"])))
    torch.cuda.empty_cache()
    return ref


_ORACLE = {}


def memo_oracle(key, *args, **kw):
    if key not in _ORACLE:
        _ORACLE[key] = oracle(*args, **kw)
    return _ORACLE[key]


# ------------------------------------------------------------------------------------------ the kernel side
def run_step(eng, sd, batch, noise, cfg, ray_valid=None):
    """One isdfb_train_fwd_bwd call the way the Trainer makes it: normals only when the normal term is on, the mean
    over the valid samples, the 'pc' bounds from the engine's all-pairs kernel."""
    eng.pack_weights(P.flat_params(sd, DEV))
    eng.zero_grad()
    b = _to_dev(batch, torch.float32)
    R, S = b["z_vals"].shape
    rv = None if ray_valid is None else ray_valid.to(device=DEV, dtype=torch.uint8)
    n_valid = R if rv is None else int(rv.sum())
    pcb = pcv = None
    if cfg.get("bounds_method", "ray") == "pc":
        pcb, pcv = eng.bounds_pc(b["pc"], b["z_vals"], b["depth_sample"], ray_valid=rv)
    lc = P.loss_cfg_from(cfg, n_valid * S, bounds=pcb, grad_vec=pcv)
    nz = noise.to(DEV) if cfg["noise_std"] else None
    nrm = b["norm_sample"] if cfg["grad_weight"] != 0 else None
    sdf, g, lm, sums = eng.train_fwd_bwd(b["pc"], b["z_vals"], b["depth_sample"], b["dirs_C_sample"],
                                         b["T_WC_sample"], nrm, nz, lc, ray_valid=rv)
    grads = P.unflatten(eng.export_grads(), sd)
    torch.cuda.synchronize(DEV)
    return dict(sdf=sdf.cpu(), g=g.cpu(), loss_mat=lm.cpu(), sums=sums.cpu(), grads=[x.cpu() for x in grads],
                n=n_valid * S)


def grad_blocks(name, t, hidden=256):
    """The parts of a gradient tensor that separate weight-gradient jobs write: 128-row halves (a job is one row half
    of one unit), the concat layer's hidden and embedding columns (different units), the output row's column halves
    (w_out rides on the last hidden layer's two jobs)."""
    if t.dim() == 2 and t.shape[0] == 1:
        return {name + "[:, :128]": t[:, :128], name + "[:, 128:]": t[:, 128:]}
    if t.shape[0] != hidden:
        return {name: t}
    out = {}
    for r, rows in (("[:128]", slice(0, 128)), ("[128:]", slice(128, hidden))):
        if name.startswith("cat_layer") and t.dim() == 2:
            out[name + r + "[:, :H]"] = t[rows, :hidden]
            out[name + r + "[:, H:]"] = t[rows, hidden:]
        else:
            out[name + r] = t[rows]
    return out


def compare(out, ref, mode, names, keep=None, orien_weight=None):
    """Errors of a kernel result against the oracle (max-abs / max-abs-ref; relative Frobenius per gradient block),
    asserted against TOL[mode] (never tighter than 3x the fp32 floor).  keep: mask of the rays the oracle ran on."""
    t, fl = TOL[mode], ref["floor"]
    sel = (lambda x: x) if keep is None else (lambda x: x[keep])
    n = out["n"]
    tol = dict(sdf=max(t["sdf"], 3 * fl["sdf"]), g=max(t["g"], 3 * fl["g"]),
               loss=max(t["loss"], 3 * fl["loss"], 3 * fl["loss_mat"]),
               gw=max(t["gw"] if n >= GW_SAMPLES else t["gw_small"], 3 * fl["gw"]))
    e = dict(sdf=P.rel(sel(out["sdf"]), ref["sdf"]), g=P.rel(sel(out["g"]), ref["g"]))
    lm, lm_ref = sel(out["loss_mat"]).double(), ref["loss_mat"].double()
    d = (lm - lm_ref).abs()
    bound = tol["loss"] * float(lm_ref.abs().max())
    if orien_weight is not None:
        # orien_loss is a step of cos(g, u) at 0: a sample within rounding of the step may land on the other side
        flip = d > bound
        assert int(flip.sum()) <= max(2, n // 1000), ("orien flips", int(flip.sum()))
        if bool(flip.any()):
            assert float((d[flip] - orien_weight).abs().max()) < bound
        d = torch.where(flip, torch.zeros_like(d), d)
        e["orien_flips"] = int(flip.sum())
    e["loss_mat"] = float(d.max() / lm_ref.abs().max())
    for i, k in enumerate(("sdf_loss", "grad_loss", "eikonal_loss", "total_loss")):
        got = float(out["sums"][i]) / n
        if k not in ref["losses"]:
            assert float(out["sums"][i]) == 0.0, (k, got)           # term switched off: nothing accumulated
            continue
        e[k] = abs(got - ref["losses"][k]) / max(abs(ref["losses"][k]), 1e-3)
    gb = {}
    for name, a, b in zip(names, out["grads"], ref["grads"]):
        gb[name] = P.rel_fro(a, b)
        for bn, blk in grad_blocks(name, b).items():
            gb[bn] = P.rel_fro(grad_blocks(name, a)[bn], blk)
    e["gw_max"] = max(gb.values())
    bad = {k: v for k, v in gb.items() if not v < tol["gw"]}
    assert e["sdf"] < tol["sdf"] and e["g"] < tol["g"], (e, tol)
    assert e["loss_mat"] < tol["loss"], (e, tol)
    for k in ("sdf_loss", "grad_loss", "eikonal_loss", "total_loss"):
        if k in e:
            assert e[k] < tol["loss"], (k, e, tol)
    assert not bad, ("weight gradients", bad, tol["gw"])
    for k in ("sdf", "g", "loss_mat", "sums"):
        assert bool(torch.isfinite(out[k]).all()), k
    return e


# ------------------------------------------------------------------------------------------ 1. launch geometry
SHAPES = {"E255_b2": (6, 2), "E255_b3": (6, 3), "E381_b2": (9, 2), "E465_b3": (11, 3)}


def _geometry_case(case, N):
    """(rays, samples per ray, max_points, expected branches per chunk) of a case, for N SMs."""
    if case == "1tile_ragged":
        return 3, 27, 32768, ["single"]
    if case == "c4":                                     # bench.py's C4 workload: 20 480 rays x 64, 4 waves per chunk
        R, S, cap = 20480, 64, N * TILE * 4
        n_chunks = -(-(R * S) // cap)
        last = chunk_plan(R * S, cap, N, 14)[-1]["branch"]
        return R, S, cap, ["persistent"] * (n_chunks - 1) + [last]
    if case == "3N_ragged":
        R = (3 * N * TILE) // 27 + 1
        return R, 27, R * 27, ["persistent"]
    if case == "2chunks":                                # 2N tiles, then 2N-5 tiles (two waves, dW grid at the floor)
        return 4 * (2 * N) + 4 * (2 * N - 5), 32, 2 * N * TILE, ["persistent", "two_wave"]
    tiles, branch = {"N": (N, "single"), "N+1": (N + 1, "two_wave"), "2N-5": (2 * N - 5, "two_wave"),
                     "2N-1": (2 * N - 1, "two_wave"), "2N": (2 * N, "persistent")}[case]
    return 4 * tiles, 32, max(32768, 4 * tiles * 32), [branch]     # S = 32: 4 rays per tile exactly


GEOM_CASES = ["1tile_ragged", "N", "N+1", "2N-5", "2N-1", "2N", "3N_ragged", "2chunks"]
GEOM_PARAMS = []
for _s in SHAPES:
    for _c in GEOM_CASES:
        for _m in TC_MODES:
            GEOM_PARAMS.append((_s, _c, _m))
        if "fp32" in PARITY_MODES and (_s == "E255_b2" or _c == "2N-5"):
            GEOM_PARAMS.append((_s, _c, "fp32"))
GEOM_PARAMS += [("E255_b2", "c4", m) for m in PARITY_MODES]


@pytest.mark.parametrize("shape,case,mode", GEOM_PARAMS, ids=["-".join(p) for p in GEOM_PARAMS])
def test_train_step_at_every_launch_plan(shape, case, mode):
    n_freqs, block = SHAPES[shape]
    E = O.embedding_size(n_freqs)
    N = num_sms()
    R, S, cap, branches = _geometry_case(case, N)
    n_jobs = n_dw_jobs(E, block)
    plan = chunk_plan(R * S, cap, N, n_jobs)
    assert [c["branch"] for c in plan] == branches, (case, plan)
    if case == "1tile_ragged":
        assert plan[0]["tiles"] == 1 and R * S % TILE
    if case == "2N":
        assert plan[0]["tiles"] == 2 * N                  # two tiles per persistent CTA
    if case == "3N_ragged":
        assert plan[0]["tiles"] >= 3 * N and R * S % TILE
    if case in ("2N-5", "2N-1", "2chunks"):               # wave 1's dW grid is the floor: one CTA per job
        assert plan[-1]["dw_grid"] == n_jobs and N - (plan[-1]["tiles"] - N) < n_jobs
    cfg = O.default_cfg(n_freqs=n_freqs, block=block, noise_std=0.08, n_strat=S - 8, n_surf=8)
    sd = C.golden_weights(31 + block, E=E, block=block, gain=1.2)
    batch, noise = C.loss_batch(1000 + R, R, S=S)
    ref = memo_oracle(("geom", shape, case), sd, batch, noise, cfg)
    eng = P.make_engine(DEV, cfg, mode, max_points=cap)
    out = run_step(eng, sd, batch, noise, cfg)
    e = compare(out, ref, mode, list(sd.keys()))
    print("geometry %s %s %s: points=%d chunks=%s errs=%s" % (shape, case, mode, R * S,
                                                               [(c["tiles"], c["branch"]) for c in plan], e))
    if case == "2N-1":
        # the same batch cut into two one-tile-per-CTA chunks instead of two waves: equal up to summation order
        cap2 = N * TILE
        assert [c["branch"] for c in chunk_plan(R * S, cap2, N, n_jobs)] == ["single", "single"]
        out2 = run_step(P.make_engine(DEV, cfg, mode, max_points=cap2), sd, batch, noise, cfg)
        assert P.rel(out2["sdf"], out["sdf"]) < CHUNK_INVARIANCE[mode]
        assert max(P.rel_fro(a, b) for a, b in zip(out2["grads"], out["grads"])) < max(1e-4, 0.1 * TOL[mode]["gw"])


# ------------------------------------------------------------------------------------------ 2. loss settings
LOSS_SETTINGS = {
    # name: (n_freqs, block, cfg overrides, batch kind)
    "orien_loss": (6, 2, dict(orien_loss=True), "ray"),
    "grad_weight_0": (6, 2, dict(grad_weight=0.0), "ray"),
    "eik_weight_0": (6, 2, dict(eik_weight=0.0), "ray"),
    "grad_and_eik_0": (6, 2, dict(grad_weight=0.0, eik_weight=0.0), "ray"),
    "franka_E465_b3": (11, 3, dict(trunc_weight=30.0, trunc_distance=0.1, noise_std=0.025, dist_behind_surf=0.01), "franka"),
    "scale_input_0.4_E381": (9, 2, dict(scale_input=0.4), "ray"),
    "pc_bound_E381": (9, 2, dict(bounds_method="pc"), "pc"),
    "masked_rays": (6, 2, {}, "masked"),
}
LOSS_PARAMS = [(s, R, m) for s in LOSS_SETTINGS for R in (1000, 40) for m in PARITY_MODES]


def mask_rays(batch, noise, frac, seed, min_depth=0.07, dist_behind=0.1):
    """Mask a fraction of the rays the way the fused sampler writes rays without depth (sample.cu): depth 0, the
    surface sample at z = 0, near-surface and stratified samples squeezed into [min_depth, dist_behind], NaN normals."""
    g = C.gen(seed)
    R, S = batch["z_vals"].shape
    masked = torch.rand(R, generator=g) < frac
    b = {k: v.clone() for k, v in batch.items()}
    n_strat, n_surf = S - 8, 8
    far = torch.full((R,), dist_behind)
    near = (0.1 * torch.randn(R, n_surf - 1, generator=g)).clamp(min_depth, dist_behind)
    edges = torch.linspace(0, 1, n_strat + 1)[None, :] * (far - min_depth)[:, None] + min_depth
    z_strat = edges[:, :-1] + torch.rand(R, n_strat, generator=g) * ((far - min_depth)[:, None] / n_strat)
    z0 = torch.cat([torch.zeros(R, 1), near, z_strat], dim=1)
    pc0 = b["T_WC_sample"][:, :3, 3][:, None, :] + b["dirs_W"][:, None, :] * z0[:, :, None]
    b["depth_sample"][masked] = 0.0
    b["z_vals"][masked] = z0[masked]
    b["pc"][masked] = pc0[masked]
    b["norm_sample"][masked] = float("nan")
    return b, (~masked).to(torch.uint8)


@pytest.mark.parametrize("setting,R,mode", LOSS_PARAMS, ids=["%s-%d-%s" % p for p in LOSS_PARAMS])
def test_train_step_at_every_loss_setting(setting, R, mode):
    n_freqs, block, over, kind = LOSS_SETTINGS[setting]
    E = O.embedding_size(n_freqs)
    cfg = O.default_cfg(n_freqs=n_freqs, block=block, **dict(dict(noise_std=0.08), **over))
    sd = C.golden_weights(41 + n_freqs, E=E, block=block, gain=1.2)
    if kind == "pc":
        batch, noise = C.loss_batch_pc(500 + R, R)
    elif kind == "franka":
        batch, noise = C.loss_batch(500 + R, R, dist_behind=cfg["dist_behind_surf"])
    else:
        batch, noise = C.loss_batch(500 + R, R)
    valid = None
    if kind == "masked":
        batch, valid = mask_rays(batch, noise, 0.3, 600 + R)
    plan = chunk_plan(R * 27, 32768, num_sms(), n_dw_jobs(E, block))
    assert [c["branch"] for c in plan] == ["two_wave" if R == 1000 else "single"], plan
    eng = P.make_engine(DEV, cfg, mode, max_points=32768)
    out = run_step(eng, sd, batch, noise, cfg, ray_valid=valid)
    keep = None
    ob, onz = batch, noise
    if valid is not None:
        keep = valid.bool()
        assert float(out["loss_mat"][~keep].abs().max()) == 0.0         # masked rows: exactly nothing
        assert bool(torch.isfinite(out["sdf"]).all() and torch.isfinite(out["g"]).all())
        assert all(bool(torch.isfinite(x).all()) for x in out["grads"])
        ob, onz = {k: v[keep] for k, v in batch.items()}, noise[keep]
    if cfg["grad_weight"] == 0:
        ob = dict(ob, norm_sample=None)                                  # the oracle must not need them either
    ref = memo_oracle(("loss", setting, R), sd, ob, onz, cfg)
    e = compare(out, ref, mode, list(sd.keys()), keep=keep,
                orien_weight=cfg["grad_weight"] if cfg["orien_loss"] else None)
    print("loss setting %s R=%d %s: errs=%s" % (setting, R, mode, e))


# ------------------------------------------------------------------------------------------ 3. fast-mode Trainer step
@pytest.fixture(scope="module")
def seq200(tmp_path_factory):
    root = tmp_path_factory.mktemp("isdf_seq200")
    s = TC.write_sequence(str(root))
    cfg = TC.config(s)
    cfg["sample"]["n_rays"] = 200                # 5 window frames x 200 rays x 27 samples: a two-wave batch
    cfg_path = os.path.join(str(root), "cfg.json")
    json.dump(cfg, open(cfg_path, "w"))
    return cfg_path


@pytest.mark.parametrize("mode", MODES)
def test_fast_mode_graph_step_matches_oracle_on_its_batch(seq200, mode):
    """The replayed fast-mode step (window, fused sampler, two-wave K4, step_finish, AdamW as one graph) against the
    fp64 oracle on the batch that replay drew, with the parameters it started from."""
    from isdf.modules import trainer
    torch.manual_seed(11)
    tr = trainer.Trainer("cuda:0", seq200, precision=mode, rng_mode="fast")
    for k in range(TC.N_FRAMES):
        tr.last_is_keyframe = True
        tr.add_data(tr.get_data([k]))
    for _ in range(3):                           # eager, capture (+ replay), replay
        tr.step()
    assert tr._graph, "the fast-mode step was not captured"
    flat0 = tr.sdf_map.flat_parameters().detach().clone()
    losses, _ = tr.step()                        # the replay under test
    torch.cuda.synchronize(DEV)
    pts, lc = tr._last_pts
    fmap = tr.active_idxs.clone()
    n_win = fmap.numel()
    assert n_win == tr.window_size and not torch.equal(fmap.cpu(), torch.arange(n_win))
    grads = tr.sdf_map.engine().export_grads().cpu()
    means = {k: float(v) for k, v in losses.items()}
    favg = tr.frames.frame_avg_losses.detach().cpu().clone()
    f = tr.frames
    ib, ih, iw = pts["indices_b"], pts["indices_h"], pts["indices_w"]
    R, S = pts["z_vals"].shape
    assert R == n_win * tr.n_rays and R * S > 148 * TILE
    # the sampler's gathers: depth through the window map, normals by window slot (fix_normal_window = 0)
    assert torch.equal(pts["depth_sample"], f.depth_batch[fmap[ib], ih, iw])
    assert not tr.fix_normal_window
    assert torch.equal(torch.nan_to_num(pts["norm_sample"], nan=7.0), torch.nan_to_num(f.normal_batch[ib, ih, iw], nan=7.0))
    keep = pts["ray_valid"].bool()
    n_valid = int(keep.sum())
    assert 0 < n_valid < R                       # the synthetic depth has holes: the mask is exercised
    sd_names = list(tr.sdf_map.state_dict().keys())
    sd_shapes = {k: v.shape for k, v in tr.sdf_map.state_dict().items()}
    sd = {k: t for k, t in zip(sd_names, P.unflatten(flat0.cpu(), {k: torch.empty(s) for k, s in sd_shapes.items()}))}
    cfg = O.default_cfg(n_freqs=tr.n_embed_funcs + 1, block=tr.hidden_layers_block, hidden=tr.hidden_feature_size,
                        scale_input=tr.scale_input, scale_output=tr.scale_output,
                        transform=tr.sdf_map.positional_encoding.transform, noise_std=lc.noise_std,
                        loss_type=tr.loss_type, trunc_weight=tr.trunc_weight, trunc_distance=tr.trunc_distance,
                        eik_weight=tr.eik_weight, eik_apply_dist=tr.eik_apply_dist, grad_weight=tr.grad_weight,
                        orien_loss=bool(tr.orien_loss))
    if cfg["transform"] is not None:
        cfg["transform"] = cfg["transform"].cpu()
    T = pts["T_WC_sample"]
    batch = dict(pc=pts["pc"], z_vals=pts["z_vals"], depth_sample=pts["depth_sample"],
                 dirs_C_sample=pts["dirs_C_sample"], T_WC_sample=T, norm_sample=pts["norm_sample"],
                 dirs_W=(T[:, :3, :3] * pts["dirs_C_sample"][:, None, :]).sum(-1))
    batch = {k: v[keep].cpu() for k, v in batch.items()}
    ref = oracle(sd, batch, pts["noise"][keep].cpu(), cfg)
    t = TOL[mode]
    n = n_valid * S
    gw = t["gw"] if n >= GW_SAMPLES else t["gw_small"]
    got = P.unflatten(grads, sd)
    errs = {k: P.rel_fro(a, b) for k, a, b in zip(sd_names, got, ref["grads"])}
    assert max(errs.values()) < gw, errs
    for k, v in ref["losses"].items():
        assert abs(means[k] - v) <= t["loss"] * max(abs(v), 1e-3), (k, means[k], v)
    lm = tr.last_loss_mat.detach().cpu()
    assert float(lm[~keep.cpu()].abs().max()) == 0.0
    assert P.rel(lm[keep.cpu()], ref["loss_mat"]) < t["loss"]
    # per-keyframe losses written back through the window map: K5 of this step's loss matrix on the valid rays
    kc = keep.cpu()
    ibv, ihv, iwv = ib.cpu()[kc], ih.cpu()[kc], iw.cpu()[kc]
    _, fa = O.frame_avg(lm[kc].double(), (n_win, tr.H, tr.W), ibv, ihv, iwv, tr.loss_approx_factor)
    assert torch.allclose(favg[fmap.cpu()].double(), fa, rtol=1e-5, atol=1e-7), (favg[fmap.cpu()], fa)
    _, fa_ref = O.frame_avg(ref["loss_mat"], (n_win, tr.H, tr.W), ibv, ihv, iwv, tr.loss_approx_factor)
    assert P.rel(favg[fmap.cpu()], fa_ref) < t["loss"]
    print("fast-mode step %s: valid samples=%d max grad rel_fro=%.3g" % (mode, n, max(errs.values())))
