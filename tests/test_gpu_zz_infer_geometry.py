"""GPU parity of the forward-only program (K2: sdf) and the forward+input-gradient program (K3: sdf, d sdf / d x) of
tc_chain_kernel, of the lattice get_sdf_grid generates inside the kernel, and of the Trainer calls built on them
(grad_fn, get_sdf_grid, the frozen map of the keyframe decision, render_depth_normals) -- all against the fp64
oracle (oracle.isdf_oracle.sdf_and_grad), run on the device in point chunks.

* Launch plans: tc_forward_impl (isdf_b200/csrc/tc_path.cu) cuts n points into max_points chunks and launches each
  with min(tiles, sms) CTAs; a CTA loops over tiles b, b + grid, ...  The per-tile step count of K2 is odd at every
  shape (7, 9, 9, 11), and the TMEM ping-pong index and the d_full barrier phases keep counting across the tiles of
  a CTA, so a CTA's second tile starts on the other accumulator and the other parity.  Every case states the plan it
  exercises, asserts it with forward_plan(), and reports the error over second-and-later tiles separately.
* Outputs are written into buffers pre-filled with a NaN-payload sentinel: a tile that is never computed cannot pass
  by reusing an earlier result, and writes past n show up bit-exactly.
* Lattice: the kernel rounds the coordinates term by term, so its points may differ from torch's by one ulp; the
  tolerance floor is measured by moving every coordinate by one ulp and re-running the oracle.

(The file name sorts after the default-shape suites on purpose.)"""
import ctypes as CT
import json
import os
import re
import time

import numpy as np
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
ORACLE_CHUNK = 65536            # points per oracle call on the device
TC_MODES = [m for m in ("bf16x3", "bf16x3g") if m in MODES]
SHAPES = {"E255_b2": (6, 2), "E255_b3": (6, 3), "E381_b2": (9, 2), "E465_b3": (11, 3)}
SENTINEL = 0x7FC0DEAD           # a quiet NaN with a payload no float arithmetic produces
PAD = 256                       # sentinel elements past n (x3 for g): longer than a tile


def num_sms():
    return torch.cuda.get_device_properties(DEV).multi_processor_count


def forward_plan(n, cap, sms):
    """The launch plan tc_forward_impl picks for n points: the engine rounds max_points up to whole tiles; per chunk
    the grid is min(tiles, sms) and CTA b runs tiles b, b + grid, ... (per_cta = ceil(tiles / grid) for CTA 0)."""
    cap = -(-cap // TILE) * TILE
    plan = []
    for p0 in range(0, n, cap):
        nc = min(cap, n - p0)
        tiles = -(-nc // TILE)
        grid = min(tiles, sms)
        plan.append(dict(p0=p0, points=nc, tiles=tiles, grid=grid, per_cta=-(-tiles // grid)))
    return plan


def tile_round(plan, n):
    """Per point: the round in which its CTA computes its tile (tile // grid); 0 = the CTA's first tile."""
    out = torch.empty(n, dtype=torch.int64)
    for c in plan:
        out[c["p0"]:c["p0"] + c["points"]] = (torch.arange(c["points"]) // TILE) // c["grid"]
    return out


# ------------------------------------------------------------------------------------------ oracle on the device
def _oracle_points(sd, cfg, x, noise, dtype):
    layers = [(w.to(device=DEV, dtype=dtype), b.to(device=DEV, dtype=dtype))
              for w, b in O.layers_from_state_dict(sd, cfg["block"])]
    cfg = dict(cfg)
    if cfg.get("transform") is not None:
        cfg["transform"] = torch.as_tensor(cfg["transform"]).to(device=DEV, dtype=dtype)
    sdf, g = [], []
    for p0 in range(0, x.shape[0], ORACLE_CHUNK):
        xs = x[p0:p0 + ORACLE_CHUNK].to(device=DEV, dtype=dtype)
        nz = None if noise is None else noise[p0:p0 + ORACLE_CHUNK].to(device=DEV, dtype=dtype)
        s, gg = O.sdf_and_grad(layers, xs, cfg, nz)
        sdf.append(s.cpu())
        g.append(gg.cpu())
    return torch.cat(sdf), torch.cat(g)


def oracle(sd, cfg, x, noise=None):
    """fp64 sdf and g at x [n, 3] plus the 'floor': how far the same computation in fp32 lands from it.  Tolerances are
    never tighter than 3x that floor (a large scale_input or 11 octaves make fp32 sin() itself lose digits)."""
    sdf, g = _oracle_points(sd, cfg, x, noise, torch.float64)
    s32, g32 = _oracle_points(sd, cfg, x, noise, torch.float32)
    torch.cuda.empty_cache()
    return dict(sdf=sdf, g=g, floor=dict(sdf=P.rel(s32, sdf), g=P.rel(g32, g)))


def lattice_oracle(sd, cfg, pc):
    """oracle() at fp32 lattice points, with the floor also covering a one-ulp move of every coordinate (the kernel
    rounds R g + t term by term; torch's matmul may fuse or reorder)."""
    ref = oracle(sd, cfg, pc)
    moved = torch.nextafter(pc, torch.full_like(pc, float("inf")))
    s_ulp, _ = _oracle_points(sd, cfg, moved, None, torch.float64)
    ref["floor"]["ulp"] = P.rel(s_ulp, ref["sdf"])
    return ref


_ORACLE = {}


def memo(key, fn, *args):
    if key not in _ORACLE:
        _ORACLE[key] = fn(*args)
    return _ORACLE[key]


def points(seed, n, half_width=6.0):
    """Points spread over +-half_width (the top octaves of the encoding wrap many times) and unit normal noise."""
    g = C.gen(seed)
    return (torch.rand(n, 3, generator=g) - 0.5) * (2 * half_width), torch.randn(n, generator=g)


# ------------------------------------------------------------------------------------------ the kernel side
def sentinel(n):
    return torch.full((n,), SENTINEL, dtype=torch.int32, device=DEV).view(torch.float32)


def tail_intact(buf, start):
    return bool((buf[start:].view(torch.int32) == SENTINEL).all())


def _ptr(t):
    return CT.c_void_p(t.data_ptr() if t is not None else 0)


def _stream():
    return CT.c_void_p(torch.cuda.current_stream(DEV).cuda_stream)


def abi_forward(eng, x, noise, noise_std, want_grad, pad=0):
    """isdfb_mlp_forward(_grad) through the C ABI into sentinel-filled outputs `pad` elements (x3 for g) longer than n."""
    x = x.to(DEV).contiguous()
    n = x.shape[0]
    nz = None if noise is None else noise.to(DEV).contiguous()
    sdf = sentinel(n + pad)
    g = sentinel(3 * (n + pad)) if want_grad else None
    if want_grad:
        rc = eng.lib.isdfb_mlp_forward_grad(eng._ctx, _ptr(x), _ptr(nz), float(noise_std), n, _ptr(sdf), _ptr(g),
                                            _stream())
    else:
        rc = eng.lib.isdfb_mlp_forward(eng._ctx, _ptr(x), _ptr(nz), float(noise_std), n, _ptr(sdf), _stream())
    eng._ck(rc)
    torch.cuda.synchronize(DEV)
    return sdf, g


def abi_forward_grid(eng, lin, scale, transform, pad=0):
    dim = lin.numel()
    out = sentinel(dim ** 3 + pad)
    sc = None if scale is None else (CT.c_float * 3)(*[float(v) for v in scale])
    tr = None if transform is None else (CT.c_float * 12)(*torch.as_tensor(transform)[:3, :4].reshape(-1).tolist())
    eng._ck(eng.lib.isdfb_mlp_forward_grid(eng._ctx, _ptr(lin), dim, sc, tr, _ptr(out), _stream()))
    torch.cuda.synchronize(DEV)
    return out


def compare(got, ref, mode, rounds=None, extra_floor=0.0):
    """Errors (max-abs / max-abs-ref) of sdf and, if present, g against the oracle, asserted against TOL[mode] (never
    tighter than 3x the fp32 floor or extra_floor).  rounds: per-point tile round; the error over rounds >= 1 is
    reported separately so that a failure confined to a CTA's later tiles says so."""
    t, fl = TOL[mode], ref["floor"]
    tol = dict(sdf=max(t["sdf"], 3 * fl["sdf"], 3 * extra_floor), g=max(t["g"], 3 * fl["g"]))
    e = {}
    for k, a in got.items():
        if a is None:
            continue
        b = ref[k].double()
        a = a.detach().cpu().double().reshape(b.shape)
        d = torch.nan_to_num((a - b).abs(), nan=float("inf")).reshape(b.shape[0], -1).amax(dim=1)
        scale = float(b.abs().max())
        e[k] = float(d.max()) / scale
        if rounds is not None and bool((rounds >= 1).any()):
            e[k + "@round0"] = float(d[rounds == 0].max()) / scale
            e[k + "@round1+"] = float(d[rounds >= 1].max()) / scale
    assert all(e[k] < tol[k] for k in got if got[k] is not None), (e, tol)
    return e, tol


# ------------------------------------------------------------------------------------------ 1. launch plans
LAUNCH_CASES = ["1tile", "N", "N+1", "2N-1", "2N", "3N_ragged", "2chunks_ragged"]


def launch_case(case, N):
    """(point counts, max_points) of a case for N SMs."""
    if case == "1tile":
        return [1, 127], 32768
    if case == "2chunks_ragged":                  # 2N, 2N, then N+6 tiles (ragged, two tiles on CTAs 0..5)
        cap = 2 * N * TILE
        return [2 * cap + (N + 5) * TILE + 45], cap
    n = {"N": N * TILE, "N+1": N * TILE + 77, "2N-1": (2 * N - 1) * TILE, "2N": 2 * N * TILE,
         "3N_ragged": 3 * N * TILE - 50}[case]
    return [n], max(32768, n)


def check_launch_plan(case, plan, n, N):
    last = plan[-1]
    if case == "1tile":
        assert len(plan) == 1 and last["tiles"] == 1 and last["grid"] == 1
    elif case == "N":
        assert len(plan) == 1 and last["tiles"] == N and last["per_cta"] == 1
    elif case == "N+1":                           # CTA 0 runs tiles 0 and N; tile N is ragged
        assert len(plan) == 1 and last["tiles"] == N + 1 and last["grid"] == N and last["per_cta"] == 2 and n % TILE
    elif case == "2N-1":                          # every CTA but the last runs two tiles
        assert len(plan) == 1 and last["tiles"] == 2 * N - 1 and last["grid"] == N and last["per_cta"] == 2
    elif case == "2N":
        assert len(plan) == 1 and last["tiles"] == 2 * N and last["per_cta"] == 2
    elif case == "3N_ragged":                     # three tiles per CTA (an odd count of an odd-length program)
        assert len(plan) == 1 and last["tiles"] == 3 * N and last["per_cta"] == 3 and n % TILE
    else:
        assert len(plan) >= 3 and all(c["tiles"] == 2 * N and c["per_cta"] == 2 for c in plan[:-1])
        assert last["points"] % TILE and last["per_cta"] == 2


def launch_cfg(shape, case):
    """Half of the cases carry a rigid PE transform (alternating over shape and case); the 2N case at E381 uses
    scale_input 0.4; the multi-chunk case carries noise (its chunks must read noise from their own offset)."""
    n_freqs, block = SHAPES[shape]
    over = {}
    if (list(SHAPES).index(shape) + LAUNCH_CASES.index(case)) % 2:
        over["transform"] = C.rigid_transform(50 + LAUNCH_CASES.index(case))
    if shape == "E381_b2" and case == "2N":
        over["scale_input"] = 0.4
    noisy = case == "2chunks_ragged"
    return O.default_cfg(n_freqs=n_freqs, block=block, noise_std=0.3 if noisy else 0.0, **over), noisy


LAUNCH_PARAMS = []
for _s in SHAPES:
    for _c in LAUNCH_CASES:
        for _p in ("fwd", "fwd_grad"):
            _modes = list(TC_MODES)
            if "fp32" in MODES and (_s == "E255_b2" or _c == "N+1"):
                _modes.append("fp32")
            if "bf16" in MODES and _s == "E255_b2" and _c == "N+1":
                _modes.append("bf16")
            LAUNCH_PARAMS += [(_s, _c, _p, _m) for _m in _modes]


@pytest.mark.parametrize("shape,case,program,mode", LAUNCH_PARAMS, ids=["-".join(p) for p in LAUNCH_PARAMS])
def test_forward_programs_at_every_launch_plan(shape, case, program, mode):
    N = num_sms()
    n_freqs, block = SHAPES[shape]
    sizes, cap = launch_case(case, N)
    cfg, noisy = launch_cfg(shape, case)
    sd = C.golden_weights(60 + n_freqs + block, E=O.embedding_size(n_freqs), block=block, gain=1.2)
    eng = P.make_engine(DEV, cfg, mode, max_points=cap)
    eng.pack_weights(P.flat_params(sd, DEV))
    for n in sizes:
        plan = forward_plan(n, cap, N)
        check_launch_plan(case, plan, n, N)
        x, noise = points(700 + n, n)
        nz = noise if noisy else None
        ref = memo(("launch", shape, case, n), oracle, sd, cfg, x, nz)
        sdf, g = abi_forward(eng, x, nz, cfg["noise_std"], program == "fwd_grad")
        e, tol = compare(dict(sdf=sdf, g=g), ref, mode, rounds=tile_round(plan, n))
        print("launch %s %s %s %s: n=%d plan=%s errs=%s tol=%s" % (
            shape, case, program, mode, n, [(c["tiles"], c["grid"], c["per_cta"]) for c in plan], e, tol))


# ------------------------------------------------------------------------------------------ 2. no writes past n
@pytest.mark.parametrize("mode", [m for m in ("bf16x3g", "fp32") if m in MODES])
def test_no_writes_past_n(mode):
    """Ragged n on a multi-chunk plan whose last chunk puts two tiles on some CTAs; outputs 256 elements (x3 for g)
    longer than n, pre-filled with a NaN-payload sentinel: the tails come back bit-identical."""
    N = num_sms()
    cap = (N + 9) * TILE
    n = 2 * cap + (N + 7) * TILE + 45
    plan = forward_plan(n, cap, N)
    assert len(plan) == 3 and plan[-1]["points"] % TILE and plan[-1]["per_cta"] == 2
    cfg = O.default_cfg(noise_std=0.3, transform=C.rigid_transform(3))
    eng = P.make_engine(DEV, cfg, mode, max_points=cap)
    eng.pack_weights(P.flat_params(C.golden_weights(81, gain=1.2), DEV))
    x, noise = points(82, n)
    xd, nd = x.to(DEV), noise.to(DEV)
    for want_grad in (False, True):
        sdf, g = abi_forward(eng, xd, nd, 0.3, want_grad, pad=PAD)
        assert tail_intact(sdf, n), ("sdf written past n", want_grad)
        assert bool(torch.isfinite(sdf[:n]).all())
        ref = eng.forward(xd, noise=nd, noise_std=0.3, want_grad=want_grad)     # the Engine's exact-size outputs
        assert P.rel(sdf[:n].cpu(), (ref[0] if want_grad else ref).cpu()) < 1e-6
        if want_grad:
            assert tail_intact(g, 3 * n), "g written past n"
            assert bool(torch.isfinite(g[:3 * n]).all())
            assert P.rel(g[:3 * n].cpu(), ref[1].reshape(-1).cpu()) < 1e-6
    dim = next(d for d in range(8, 200) if d ** 3 > 2 * cap and (d ** 3 % cap) % TILE)
    gplan = forward_plan(dim ** 3, cap, N)
    assert len(gplan) >= 3 and gplan[-1]["points"] % TILE
    lin = torch.linspace(-1.0, 1.0, dim, device=DEV)
    out = abi_forward_grid(eng, lin, [5.1, 1.8, 3.9], C.rigid_transform(4), pad=PAD)
    assert tail_intact(out, dim ** 3), "lattice sdf written past dim^3"
    assert bool(torch.isfinite(out[:dim ** 3]).all())


# ------------------------------------------------------------------------------------------ 3. in-kernel lattice
GRID_CASES = ["1tile", "N+k", "chunks"]


def grid_case(case, N):
    """(dim, max_points) of a lattice case for N SMs."""
    if case == "1tile":
        return 5, 32768
    if case == "N+k":                             # the first dim past N tiles: one chunk, two tiles on some CTAs
        d = next(d for d in range(2, 400) if d ** 3 > N * TILE)
        return d, max(32768, d ** 3)
    cap = (N + 7) * TILE                          # several chunks of N+7 tiles (chunk offset p0 enters i, j, k)
    return next(d for d in range(2, 400) if d ** 3 > 2 * cap and (d ** 3 % cap) % TILE), cap


def check_grid_plan(case, plan, N):
    last = plan[-1]
    if case == "1tile":
        assert len(plan) == 1 and last["tiles"] == 1 and last["points"] % TILE
    elif case == "N+k":
        assert len(plan) == 1 and N < last["tiles"] <= 2 * N and last["per_cta"] == 2
    else:
        assert len(plan) >= 3 and last["points"] % TILE and plan[0]["per_cta"] == 2


GRID_PARAMS = []
for _s in SHAPES:
    for _c in GRID_CASES:
        for _v in ("plain", "box"):
            _modes = list(TC_MODES) + (["fp32"] if "fp32" in MODES and _s in ("E255_b2", "E465_b3") else [])
            GRID_PARAMS += [(_s, _c, _v, _m) for _m in _modes]
BOX_SCALE = [5.1, 1.8, 3.9]                       # anisotropic: the lattice spans +-5 m along x


@pytest.mark.parametrize("shape,case,variant,mode", GRID_PARAMS, ids=["-".join(p) for p in GRID_PARAMS])
def test_lattice_generated_in_kernel(shape, case, variant, mode):
    """isdfb_mlp_forward_grid against the fp64 oracle at the transform.make_3D_grid points; 'box' adds a box transform,
    an anisotropic scale and a rigid PE transform."""
    from isdf.geometry import transform
    N = num_sms()
    n_freqs, block = SHAPES[shape]
    dim, cap = grid_case(case, N)
    plan = forward_plan(dim ** 3, cap, N)
    check_grid_plan(case, plan, N)
    box = variant == "box"
    cfg = O.default_cfg(n_freqs=n_freqs, block=block, transform=C.rigid_transform(14) if box else None)
    sd = C.golden_weights(90 + n_freqs + block, E=O.embedding_size(n_freqs), block=block, gain=1.2)
    T_box = C.rigid_transform(3) if box else None
    scale = torch.tensor(BOX_SCALE) if box else None
    pc = transform.make_3D_grid([-1.0, 1.0], dim, DEV, transform=None if T_box is None else T_box.to(DEV),
                                scale=None if scale is None else scale.to(DEV)).reshape(-1, 3).cpu()
    ref = memo(("grid", shape, case, variant), lattice_oracle, sd, cfg, pc)
    eng = P.make_engine(DEV, cfg, mode, max_points=cap)
    eng.pack_weights(P.flat_params(sd, DEV))
    lin = torch.linspace(-1.0, 1.0, dim, device=DEV)
    out = abi_forward_grid(eng, lin, None if scale is None else scale.tolist(), T_box)
    e, tol = compare(dict(sdf=out), ref, mode, rounds=tile_round(plan, dim ** 3), extra_floor=ref["floor"]["ulp"])
    got = eng.forward_grid(lin, scale=scale, transform=T_box)          # the Engine's call: same values, its shape
    assert got.shape == (dim, dim, dim) and P.rel(got.reshape(-1).cpu(), out.cpu()) < 1e-6
    print("lattice %s %s %s %s: dim=%d plan=%s floor=%s errs=%s tol=%s" % (
        shape, case, variant, mode, dim, [(c["tiles"], c["grid"], c["per_cta"]) for c in plan], ref["floor"], e, tol))


def test_lattice_past_2_31_points():
    """dim = 1291: 2 151 685 171 points (8.6 GB of sdf), past int32 indexing; every value finite and ~4 k points, among
    them the last tile and both sides of index 2^31, equal to the oracle."""
    if "bf16x3g" not in MODES:
        pytest.skip("bf16x3g not among the tested modes")
    from isdf.geometry import transform
    N = num_sms()
    dim = 1291
    n = dim ** 3
    assert n > 2 ** 31
    cap = N * TILE * 8
    cfg = O.default_cfg(transform=C.rigid_transform(14))
    sd = C.golden_weights(95, gain=1.2)
    eng = P.make_engine(DEV, cfg, "bf16x3g", max_points=cap)
    eng.pack_weights(P.flat_params(sd, DEV))
    T_box = C.rigid_transform(3)
    scale = torch.tensor(BOX_SCALE)
    lin = torch.linspace(-1.0, 1.0, dim, device=DEV)
    eng.forward_grid(lin[:5], scale=scale, transform=T_box)          # module load, outside the timing
    torch.cuda.synchronize(DEV)
    t0 = time.perf_counter()
    sdf = eng.forward_grid(lin, scale=scale, transform=T_box).view(-1)
    torch.cuda.synchronize(DEV)
    secs = time.perf_counter() - t0
    assert bool(torch.isfinite(sdf).all())
    g = C.gen(96)
    idx = torch.cat([torch.randint(0, n, (3500,), generator=g), torch.arange(n - 2 * TILE, n),
                     torch.arange(2 ** 31 - 200, 2 ** 31 + 200), torch.arange(0, 64)])
    i, j, k = idx // (dim * dim), (idx // dim) % dim, idx % dim
    lc = lin.cpu()
    grid = torch.stack([lc[i], lc[j], lc[k]], dim=-1)[:, None, None, :].to(DEV)
    pc = transform.transform_3D_grid(grid, transform=T_box.to(DEV), scale=scale.to(DEV)).reshape(-1, 3).cpu()
    ref = lattice_oracle(sd, cfg, pc)
    got = sdf[idx.to(DEV)].cpu()
    del sdf
    torch.cuda.empty_cache()
    e, tol = compare(dict(sdf=got), ref, "bf16x3g", extra_floor=ref["floor"]["ulp"])
    print("lattice dim=%d (%d points, %d chunks): %.2f s = %.1f M points/s on %s; floor=%s errs=%s tol=%s" % (
        dim, n, len(forward_plan(n, cap, N)), secs, n / secs / 1e6, torch.cuda.get_device_name(DEV), ref["floor"], e,
        tol))


# ------------------------------------------------------------------------------------------ 4. Trainer surface
@pytest.fixture(scope="module")
def seq(tmp_path_factory):
    root = tmp_path_factory.mktemp("isdf_seq_infer_geometry")
    s = TC.write_sequence(str(root))
    cfg_path = os.path.join(str(root), "cfg.json")
    json.dump(TC.config(s), open(cfg_path, "w"))
    return cfg_path


def _snapshot(m):
    return {k: v.detach().cpu().clone() for k, v in m.state_dict().items()}


def _map_cfg(tr):
    tf = tr.sdf_map.positional_encoding.transform
    return O.default_cfg(n_freqs=tr.n_embed_funcs + 1, block=tr.hidden_layers_block, hidden=tr.hidden_feature_size,
                         scale_input=tr.scale_input, scale_output=tr.scale_output,
                         transform=None if tf is None else torch.as_tensor(tf).detach().cpu().float())


@pytest.mark.parametrize("mode", [m for m in ("bf16x3g", "fp32") if m in MODES])
def test_trainer_inference_surface_on_oracle(seq, mode, capsys):
    from isdf.modules import trainer, render
    from isdf.geometry import transform
    np.random.seed(3)
    torch.manual_seed(3)
    tr = trainer.Trainer("cuda:0", seq, precision=mode, grid_dim=24)
    for k in range(2):
        tr.add_frame(tr.get_data([k]))
        tr.last_is_keyframe = True
        tr.optim_frames = 5
        for _ in range(5):
            tr.step()
    x, _ = points(101, 3000, half_width=3.0)

    # grad_fn / sdf_fn on the trained weights
    sd = _snapshot(tr.sdf_map)
    cfg = _map_cfg(tr)
    ref = oracle(sd, cfg, x)
    e_fn, _ = compare(dict(sdf=torch.from_numpy(tr.sdf_fn(x.numpy())), g=torch.from_numpy(tr.grad_fn(x.numpy()))),
                      ref, mode)

    # get_sdf_grid over the scene box: the in-kernel lattice, then a caller-supplied point set
    T_box = C.rigid_transform(14).numpy().astype(np.float64)
    tr.set_scene_properties(T_extent_to_scene=T_box, bounds_extents=np.array([6.0, 2.5, 4.0]))
    cfg = _map_cfg(tr)
    assert cfg["transform"] is not None
    pc = transform.make_3D_grid([-1.0, 1.0], 24, DEV, transform=tr.bounds_transform,
                                scale=tr.scene_scale).reshape(-1, 3).contiguous()
    gref = lattice_oracle(sd, cfg, pc.cpu())
    grid = tr.get_sdf_grid()
    assert grid.shape == (24, 24, 24)
    e_grid, _ = compare(dict(sdf=grid), gref, mode, extra_floor=gref["floor"]["ulp"])
    tr.grid_pc = pc.clone()
    grid_pc = tr.get_sdf_grid()
    e_grid_pc, _ = compare(dict(sdf=grid_pc), gref, mode, extra_floor=gref["floor"]["ulp"])

    # frozen map: add_frame after a keyframe snapshots the map; later steps change the live map only
    tr.last_is_keyframe = True                    # what check_keyframe_latest leaves after a keyframe
    sd_frozen = _snapshot(tr.sdf_map)
    tr.add_frame(tr.get_data([2]))
    for _ in range(3):
        tr.step()
    sd_live = _snapshot(tr.sdf_map)
    with torch.no_grad():
        f_sdf = tr.frozen_sdf_map(x.to(DEV))
        l_sdf = tr.sdf_map(x.to(DEV))
    ref_f = oracle(sd_frozen, cfg, x)
    ref_l = oracle(sd_live, cfg, x)
    e_frozen, tol = compare(dict(sdf=f_sdf), ref_f, mode)
    e_live, _ = compare(dict(sdf=l_sdf), ref_l, mode)
    moved = P.rel(ref_l["sdf"], ref_f["sdf"])
    assert moved > 10 * tol["sdf"], ("three steps did not move the live map away from the frozen one", moved)

    # the keyframe decision: the proportion is_keyframe prints, recomputed from the oracle.  After a few steps the map's
    # sdf has no zero crossing on most rays (every ray renders depth 0 and fails), so the frozen map is given weights
    # whose sdf changes sign along the rays, and kf_dist_th is put into the widest gap of the oracle's relative depth
    # errors on a first draw; the decision is then taken again on the same samples.
    sd_kf = C.golden_weights(97, gain=1.2)
    tr.frozen_sdf_map.load_state_dict(sd_kf)
    eng = tr.frozen_sdf_map.engine()
    calls, drawn = [], []
    fwd, sample_points = eng.forward, tr.sample_points

    def rec_forward(xx, noise=None, noise_std=0.0, want_grad=False):
        out = fwd(xx, noise=noise, noise_std=noise_std, want_grad=want_grad)
        calls.append((xx.detach().clone(), None if noise is None else noise.clone(), float(noise_std), out.clone()))
        return out

    def rec_sample(*a, **kw):
        if drawn:
            return drawn[0]                       # the replay: the samples of the first draw
        drawn.append(sample_points(*a, **kw))
        return drawn[0]

    def decide():
        capsys.readouterr()
        tr.is_keyframe(tr.frames.T_WC_batch[-1].unsqueeze(0), tr.frames.depth_batch[-1].unsqueeze(0))
        return float(re.search(r"Proportion of loss below threshold (\S+)", capsys.readouterr().out).group(1))

    def oracle_decision(call):
        xx, noise, noise_std, got = call
        assert noise is not None and noise_std == tr.noise_std
        kref = oracle(sd_kf, dict(cfg, noise_std=noise_std), xx.reshape(-1, 3).cpu(), noise.reshape(-1).cpu())
        e, ktol = compare(dict(sdf=got.reshape(-1)), kref, mode)
        pts = drawn[0]
        R, S = pts["z_vals"].shape
        sdf_ref = kref["sdf"].view(R, S)
        z, order = pts["z_vals"].cpu().double().sort(dim=-1)
        view_depth = render.sdf_render_depth(z, torch.gather(sdf_ref, 1, order))
        depth = pts["depth_sample"].cpu().double()
        valid = torch.ones(R, dtype=torch.bool) if pts.get("ray_valid") is None else pts["ray_valid"].cpu().bool()
        return e, ktol, sdf_ref, depth, (view_depth - depth).abs() / depth, valid

    th0 = tr.kf_dist_th
    eng.forward, tr.sample_points = rec_forward, rec_sample
    try:
        decide()
        _, _, _, _, err0, valid0 = oracle_decision(calls[0])
        v = err0[valid0].sort().values
        assert v.numel() >= 8 and float(v[-1] - v[0]) > 0.05, ("no spread of rendered depths", v)
        lo, hi = v.numel() // 4, (3 * v.numel()) // 4
        i = lo + int((v[lo + 1:hi + 1] - v[lo:hi]).argmax())
        tr.kf_dist_th = float(v[i] + v[i + 1]) / 2
        prop = decide()
    finally:
        del eng.forward, tr.sample_points
        th, tr.kf_dist_th = tr.kf_dist_th, th0
    assert len(calls) == 2 and len(drawn) == 1
    e_kf, ktol, sdf_ref, depth, err, valid = oracle_decision(calls[1])
    n_valid = int(valid.sum())
    k_ref = int(((err < th) & valid).sum())
    k_got = int(round(prop * n_valid))
    assert 0 < k_ref < n_valid
    # a ray with a sample within tolerance of the surface may render another sample index (or land on the other side
    # of the threshold): only such rays may differ
    tol_abs = ktol["sdf"] * float(sdf_ref.abs().max())
    ambiguous = ((sdf_ref.abs() <= tol_abs).any(dim=1) | ((err - th).abs() <= 2 * tol_abs / depth)) & valid
    n_amb = int(ambiguous.sum())
    assert abs(k_got - k_ref) <= n_amb, (prop, k_got, k_ref, n_valid, n_amb)
    assert n_amb <= max(2, n_valid // 20), (n_amb, n_valid)

    # render_depth_normals: normals = -g / (|g| + 1e-4) of the oracle at the kernel's own rendered depths, in camera frame
    T = tr.frames.T_WC_batch_np[-1]
    depth_r, normals = tr.render_depth_normals(T)
    assert bool(torch.isfinite(normals).all())
    T_WC = torch.as_tensor(T, dtype=torch.float32, device=DEV).reshape(1, 4, 4)
    R_WC = T_WC[:, :3, :3]
    dirs_W = (R_WC * tr.dirs_C_vis_up[..., None, :]).sum(dim=-1).view(-1, 3)
    pc_r = (T_WC[:, :3, -1].view(-1, 3) + dirs_W * depth_r.flatten()[:, None]).cpu()     # the points K3 ran at
    nref = oracle(sd_live, cfg, pc_r)
    g = nref["g"]
    gn = g.norm(dim=1, keepdim=True)
    n_C = (-g / (gn + 1e-4)) @ R_WC[0].cpu().double()                    # R^T n_W, row-vector form
    ntol = max(TOL[mode]["g"], 3 * nref["floor"]["g"])
    bound = 2 * ntol * float(gn.max()) / (gn[:, 0] + 1e-4) + 1e-5        # |d n| <~ 2 |d g| / |g|
    dn = (normals.reshape(-1, 3).cpu().double() - n_C).abs().amax(dim=1)
    assert bool((dn <= bound).all()), (float(dn.max()), float((dn / bound).max()))
    print("trainer surface %s: fn=%s grid=%s grid_pc=%s frozen=%s live=%s (moved %.3g) kf=%s prop=%.4f "
          "th=%.4f k=%d/%d ref=%d ambiguous=%d normals max|dn|/bound=%.3g" % (
              mode, e_fn, e_grid, e_grid_pc, e_frozen, e_live, moved, e_kf, prop, th, k_got, n_valid, k_ref, n_amb,
              float((dn / bound).max())))
