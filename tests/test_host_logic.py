"""CPU tests of the host-side mirror (no kernels): render / grid helpers and the checkpoint format against
fixtures produced by the unmodified reference (tests/golden/make_golden_infer.py)."""
import io
import os

import torch

from tests.golden import common as C
describe = C.describe

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def load(name):
    return torch.load(os.path.join(GOLD, name), weights_only=False)


def test_sdf_render_depth_matches_reference():
    from isdf_b200.modules import render
    g = load("infer.pt")["render_depth"]
    assert torch.equal(render.sdf_render_depth(g["z"], g["sdf"]), g["depth"])


def test_make_3d_grid_matches_reference():
    from isdf_b200.geometry import transform
    g = load("infer.pt")["grid"]
    T_box = C.rigid_transform(14)
    scale = g["extents"] / (2.0 * 0.9)
    pc = transform.make_3D_grid([-1.0, 1.0], 12, "cpu", transform=torch.inverse(T_box), scale=scale).view(-1, 3)
    assert torch.allclose(pc, g["grid_pc"], atol=1e-6)


def test_checkpoint_structure_matches_reference_files():
    """Row N4: what Trainer.save_checkpoint writes has exactly the nested keys / shapes / dtypes of the file the
    reference driver writes (train.py:207-219), so either side loads the other's checkpoints."""
    from isdf_b200.modules import embedding, fc_map
    from isdf_b200.modules.trainer import FusedAdamW
    gold = load("infer.pt")["checkpoint"]
    pe = embedding.PostionalEncoding(min_deg=0, max_deg=5, scale=0.05937489)
    m = fc_map.SDFMap(pe, 256, 2, 0.14)
    m.load_state_dict(C.golden_weights(73))
    opt = FusedAdamW(m, lr=0.0013, weight_decay=0.012)
    opt.step_count = 2
    ck = {"step": 7.5, "model_state_dict": m.state_dict(), "optimizer_state_dict": opt.state_dict(), "loss": 0.25}
    buf = io.BytesIO()
    torch.save(ck, buf)
    mine = describe(torch.load(io.BytesIO(buf.getvalue()), weights_only=False))
    assert mine == gold["structure"]
    # and torch's own AdamW accepts it (what the reference's optimiser.load_state_dict would do)
    ref_opt = torch.optim.AdamW(m.parameters(), lr=0.5, weight_decay=0.5)
    ref_opt.load_state_dict(ck["optimizer_state_dict"])
    assert ref_opt.param_groups[0]["lr"] == 0.0013 and float(ref_opt.state[list(m.parameters())[0]]["step"]) == 2.0


# ---- host helpers vs the reference (tests/golden/make_golden_host.py) ---------------------------------------------
def _close(a, b, tol=1e-6):
    a = torch.as_tensor(a)
    b = torch.as_tensor(b)
    assert a.shape == b.shape, (a.shape, b.shape)
    nan = torch.isnan(b)
    assert torch.equal(torch.isnan(a), nan)
    assert torch.allclose(a[~nan].double(), b[~nan].double(), atol=tol, rtol=tol)


def test_transform_helpers_match_reference():
    import numpy as np
    from isdf_b200.geometry import transform as T
    g = load("host.pt")
    H, W, cam = 12, 16, (20.0, 21.0, 7.5, 5.5)
    _close(T.ray_dirs_C(2, H, W, *cam, "cpu", "z"), g["ray_dirs_z"])
    _close(T.ray_dirs_C(1, H, W, *cam, "cpu", "euclidean"), g["ray_dirs_e"])
    dirs = g["ray_dirs_z"].view(2, -1, 3)[0, :40]
    Tw = torch.stack([C.synthetic_pose(k % 5) for k in range(40)])
    for mine, ref in zip(T.origin_dirs_W(Tw, dirs), g["origin_dirs_W"]):
        _close(mine, ref)
    for mine, ref in zip(T.origin_dirs_W(Tw[3:4], g["ray_dirs_z"].view(2, -1, 3)[:1]), g["origin_dirs_W_one_pose"]):
        _close(mine, ref)
    depth = C.synthetic_depth(2, H, W)
    depth[3, 4] = float("nan")
    _close(T.pointcloud_from_depth_torch(depth, *cam), g["pc_torch"])
    _close(T.pointcloud_from_depth_torch(depth, *cam, depth_type="euclidean", skip=2), g["pc_torch_e_skip2"])
    _close(T.pointcloud_from_depth(depth.numpy(), *cam), g["pc_np"])
    _close(T.backproject_pointclouds(np.stack([depth.numpy(), 2 * depth.numpy()]), *cam), g["backproject"])
    pts = torch.randn(50, 3, generator=C.gen(81))      # the golden script's first draw from gen(81)
    ext, cen = T.pc_bounds(pts.numpy())
    _close(ext, g["pc_bounds"][0]); _close(cen, g["pc_bounds"][1])
    n = T.estimate_pointcloud_normals(T.pointcloud_from_depth_torch(C.synthetic_depth(1, 24, 32), 30., 30., 15.5, 11.5))
    _close(n, g["normals"], tol=1e-5)
    _close(T.normalize(np.array([3.0, -4.0, 12.0])), g["normalize"])


def test_loss_and_render_helpers_match_reference():
    from isdf_b200.modules import loss as L, render as R, sample as S
    g = load("host.pt")
    batch, _ = C.loss_batch(82, 20)
    b, gv = L.bounds_ray(batch["depth_sample"], batch["z_vals"], batch["dirs_C_sample"], batch["T_WC_sample"], True)
    _close(b, g["bounds_ray"][0]); _close(gv, g["bounds_ray"][1])
    sdf = g["sdf"]
    for lt in ("L1", "L2"):
        mat, free = L.sdf_loss(sdf, b, 0.29365022, loss_type=lt)
        _close(mat, g["sdf_loss_" + lt][0]); assert torch.equal(free, g["sdf_loss_" + lt][1])
    for mine, ref in zip(L.full_sdf_loss(sdf, b), g["full_sdf_loss"]):
        _close(mine, ref)
    for mine, ref in zip(L.tsdf_loss(sdf, b, 0.3), g["tsdf_loss"]):
        _close(mine, ref)
    gq = C.gen(81)
    torch.randn(50, 3, generator=gq); torch.randn(20, 27, generator=gq)         # replay the golden script's draws
    gl, ek = torch.rand(20, 27, generator=gq), torch.rand(20, 27, generator=gq)
    mat, free = L.sdf_loss(sdf, b, 0.29365022, loss_type="L1")
    tot, tot_mat, losses = L.tot_loss(mat.clone(), gl, ek, free, b, 0.1, 5.38344020, 0.018, 0.268)
    _close(tot, g["tot_loss"][0]); _close(tot_mat, g["tot_loss"][1])
    assert list(losses) == list(g["tot_loss"][2])                                  # same keys, same order (train.py:138,215)
    for k, v in g["tot_loss"][2].items():
        assert abs(float(losses[k]) - v) < 1e-6
    full, masks = torch.rand(3, 16, 24, generator=gq), (torch.rand(3, 16, 24, generator=gq) < 0.2).float()
    _close(L.approx_loss(full * masks, masks.clone(), 24, 16, 8), g["approx_loss"])
    w, v = torch.rand(5, 9, generator=gq), torch.rand(5, 9, generator=gq)
    _close(R.render_weighted(w, v), g["render_weighted"][0]); _close(R.render_weighted(w, v, normalise=True), g["render_weighted"][1])
    torch.manual_seed(9)
    _close(S.stratified_sample(0.07, 5.0, 6, "cpu", 11), g["strat_scalar"])
    torch.manual_seed(9)
    _close(S.stratified_sample(0.07, torch.linspace(1, 3, 6), 6, "cpu", 11), g["strat_tensor"])


def test_framedata_append_and_replace_match_reference():
    import numpy as np
    from isdf_b200.datasets.data_util import FrameData
    g = load("host.pt")["framedata"]
    fd = FrameData()
    for (k, rep), ref in zip(((0, False), (1, False), (2, True), (3, False), (4, True)), g):
        d_ = FrameData(frame_id=np.array([k]), im_batch=torch.full((1, 2, 3, 3), float(k)), im_batch_np=np.full((1, 2, 3, 3), k, np.uint8),
                       depth_batch=torch.full((1, 2, 3), float(k)), depth_batch_np=np.full((1, 2, 3), k, np.float32),
                       T_WC_batch=torch.eye(4)[None] * k, T_WC_batch_np=np.eye(4, dtype=np.float32)[None] * k,
                       normal_batch=torch.full((1, 2, 3, 3), float(k)))
        fd.add_frame_data(d_, replace=rep)
        n, fid, dep, im, favg, tnp = ref
        assert len(fd) == n and np.array_equal(fd.frame_id, fid)
        assert torch.equal(fd.depth_batch[:, 0, 0], dep) and np.array_equal(fd.im_batch_np[:, 0, 0, 0], im)
        assert torch.equal(fd.frame_avg_losses, favg) and np.array_equal(fd.T_WC_batch_np[:, 0, 0], tnp)
        assert fd.normal_batch.shape == (n, 2, 3, 3) and fd.im_batch.shape == (n, 2, 3, 3)


def test_scannet_reader_and_intrinsics(tmp_path):
    """configs[2] (ScanNet): the reader of the reference's on-disk layout (datasets/dataset.py:74-121) and the
    depth-camera intrinsics parser (trainer.py:335-346); depth in metres, far values zeroed (image_transforms.py)."""
    import cv2
    import numpy as np
    from isdf_b200.datasets import dataset as ds
    root = tmp_path / "scene0010_00"
    (root / "frames" / "color").mkdir(parents=True)
    (root / "frames" / "depth").mkdir(parents=True)
    rng = np.random.default_rng(3)
    depths, poses = [], []
    for i in range(3):
        d = rng.integers(0, 6000, size=(48, 64)).astype(np.uint16)
        d[0, 0] = 20000                                               # 20 m -> zeroed by the depth filter (max 12 m)
        cv2.imwrite(str(root / "frames" / "depth" / ("%d.png" % i)), d)
        cv2.imwrite(str(root / "frames" / "color" / ("%d.jpg" % i)), np.full((96, 128, 3), (10 * i, 100, 200), np.uint8))
        depths.append(d)
        poses.append(C.synthetic_pose(i).numpy().reshape(-1))
    np.savetxt(str(root / "traj.txt"), np.array(poses))
    (root / "scene0010_00.txt").write_text("colorHeight = 968\ncolorWidth = 1296\ndepthHeight = 480\ndepthWidth = 640\n"
                                           "fx_depth = 577.870605\nfy_depth = 577.870605\nmx_depth = 319.5\nmy_depth = 239.5\n")
    assert ds.read_scannet_intrinsics(str(root / "scene0010_00.txt")) == (577.870605, 577.870605, 319.5, 239.5, 480, 640)
    rd = ds.ScanNetDataset(str(root), str(root / "traj.txt"), rgb_transform=ds.bgr_to_rgb,
                           depth_transform=ds.depth_scale_filter(1.0 / 1000.0, 12.0))
    assert len(rd) == 3
    s = rd[2]
    ref = depths[2].astype(np.float32) / 1000.0
    ref[ref > 12.0] = 0.0
    assert s["depth"].dtype == np.float32 and np.allclose(s["depth"], ref) and s["depth"][0, 0] == 0.0
    assert s["image"].shape == (96, 128, 3) and abs(int(s["image"][5, 5, 0]) - 200) <= 3       # BGR -> RGB
    assert np.allclose(s["T"], C.synthetic_pose(2).numpy())


# A stand-in for an upstream iSDF checkout: its layout (`isdf` is a namespace package; the sub-packages the drivers
# import) with just enough code for what the two tests below drive, so that they need nothing outside this repository.
# The Trainer takes the driver's calls (train.py:102-136) and reports the mean depth of its frames as `total_loss`.
_STUB_TRAINER = '''import json
import cv2
import numpy as np
import torch


class Trainer:
    def __init__(self, device, config_file, chkpt_load_file=None, incremental=True):
        ds = json.load(open(config_file))["dataset"]
        self.seq_dir, self.depth_scale = ds["seq_dir"], ds["depth_scale"]
        self.last_is_keyframe = False
        self.depths = []

    def get_data(self, idxs):
        return [cv2.imread(self.seq_dir + "results/depth%06d.png" % k, cv2.IMREAD_UNCHANGED) / self.depth_scale
                for k in idxs]

    def add_data(self, data):
        self.depths += data

    def step(self):
        return {"total_loss": torch.tensor(float(np.mean(self.depths)))}, 0.0
'''
_STUB_REFERENCE = {
    "isdf/modules/__init__.py": "", "isdf/modules/trainer.py": _STUB_TRAINER, "isdf/modules/fc_map.py": "",
    "isdf/modules/embedding.py": "", "isdf/modules/sample.py": "", "isdf/modules/loss.py": "",
    "isdf/modules/render.py": "",
    "isdf/geometry/__init__.py": "", "isdf/geometry/transform.py": "def to_trimesh(transform=None):\n    return None\n",
    "isdf/datasets/__init__.py": "", "isdf/datasets/data_util.py": "", "isdf/datasets/sdf_util.py": "",
    "isdf/eval/__init__.py": "", "isdf/eval/plot_utils.py": "",
    "isdf/eval/metrics.py": "def accuracy_comp(gt_points, rec_points):\n    return 0.0\n",
    "isdf/visualisation/__init__.py": "",
}


def _stub_reference(root):
    for rel, text in _STUB_REFERENCE.items():
        os.makedirs(os.path.join(root, os.path.dirname(rel)), exist_ok=True)
        with open(os.path.join(root, rel), "w") as f:
            f.write(text)
    return str(root)


def test_alias_package_layers_over_the_reference_checkout(tmp_path):
    """INTEGRATION.md section 1: with this repo BEFORE the reference on sys.path, the drivers' imports resolve --
    replaced modules here, everything else (isdf.visualisation, isdf.eval.plot_utils, missing names) in the reference."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    ref = _stub_reference(tmp_path / "reference")
    res = subprocess.run([sys.executable, os.path.join(root, "tools", "dropin_check.py")], capture_output=True, text=True,
                         timeout=300, env=dict(os.environ, ISDF_REFERENCE=ref))
    assert res.returncode == 0, res.stdout + res.stderr
    out = res.stdout
    assert "trainer from %s" % os.path.join(root, "isdf_b200", "modules", "trainer.py") in out
    assert "visualisation from %s" % os.path.join(ref, "isdf", "visualisation", "__init__.py") in out
    assert "accuracy_comp (fallback): isdf_reference.eval.metrics" in out
    assert "to_trimesh (fallback): isdf_reference.geometry.transform" in out
    assert "isdf.eval.plot_utils from %s" % os.path.join(ref, "isdf", "eval", "plot_utils.py") in out


def test_reference_copy_is_verbatim_and_steps_on_cpu(tmp_path, monkeypatch):
    """oracle/make_ref.py + oracle/ref_step.py: the CPU arm of bench.py.  The copy under oracle/_ref must be byte-identical
    to the checkout (SHA-256 manifest) and leave out what is not source, import through the shim without this repo's `isdf`
    alias getting in the way, and its Trainer must be driven like train.py does, on the sequence ref_step writes."""
    import hashlib
    import json
    import subprocess
    import sys
    import numpy as np
    from oracle import make_ref
    src = _stub_reference(tmp_path / "reference")
    os.makedirs(os.path.join(src, "isdf", "modules", "__pycache__"))
    open(os.path.join(src, "isdf", "modules", "__pycache__", "trainer.cpython-312.pyc"), "wb").write(b"\0")
    open(os.path.join(src, "isdf", "visualisation", "100x100.png"), "wb").write(b"\x89PNG")
    monkeypatch.setattr(make_ref, "SRC", src)
    monkeypatch.setattr(make_ref, "DST", str(tmp_path / "_ref"))
    assert make_ref.populate()
    man = json.load(open(os.path.join(make_ref.DST, "MANIFEST.json")))
    assert sorted(man["files"]) == sorted(_STUB_REFERENCE)
    assert not os.path.exists(os.path.join(make_ref.DST, "isdf", "modules", "__pycache__"))
    assert not os.path.exists(os.path.join(make_ref.DST, "isdf", "visualisation", "100x100.png"))
    for rel, digest in man["files"].items():
        for root in (make_ref.SRC, make_ref.DST):
            assert hashlib.sha256(open(os.path.join(root, rel), "rb").read()).hexdigest() == digest, (root, rel)
    # a tiny config through the same stepper bench.py uses, in a fresh interpreter (the shim evicts `isdf*` modules)
    code = (
        "import sys, json; sys.path.insert(0, %r)\n"
        "import torch; torch.set_num_threads(4)\n"
        "import bench\n"
        "from oracle import ref_step\n"
        "wl = dict(bench.WORKLOADS['default']); wl.update(H=120, W=160, fx=100.0, fy=100.0, cx=79.5, cy=59.5, n_rays=16)\n"
        "st = ref_step.RefTrainerStepper(bench.make_config(wl, 'fp32', 'reference'), n_keyframes=6)\n"
        "a = st.step(); b = st.step()\n"
        "print(json.dumps({'file': st.trainer_file, 'pts': st.points_per_step, 'loss': [a[0], b[0]]}))\n"
        % os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600,
                         env=dict(os.environ, ISDF_REFERENCE_ROOT=make_ref.DST))
    assert res.returncode == 0, res.stderr[-2000:]
    out = json.loads(res.stdout.strip().splitlines()[-1])
    assert out["file"] == os.path.join(make_ref.DST, "isdf", "modules", "trainer.py")
    # the six keyframes of ref_step.write_sequence, read back from its 1 mm PNGs
    v, u = np.arange(120.0)[:, None], np.arange(160.0)[None, :]
    mean_depth = np.mean([2.0 + 0.5 * np.sin(u / 80.0 + 0.1 * k) + 0.3 * np.cos(v / 60.0) for k in range(6)])
    assert out["pts"] == 16 * 5 * 27 and all(abs(x - mean_depth) < 1e-3 for x in out["loss"])


def test_bench_cpu_thread_count_is_one_per_physical_core():
    import bench
    n = bench.host_threads()
    assert 1 <= n <= (os.cpu_count() or 1) and torch.get_num_threads() == n


def test_bench_cpu_arm_falls_back_to_the_port_without_the_reference(monkeypatch):
    """bench.make_cpu_stepper: with neither /root/reference nor oracle/_ref the CPU arm times the committed restatement
    (kind 'port') instead of failing; with the reference it reports kind 'reference'."""
    import bench
    from oracle import ref_shim
    wl = dict(bench.WORKLOADS["default"])
    wl.update(H=64, W=96, fx=60.0, fy=60.0, cx=47.5, cy=31.5, n_rays=8)
    monkeypatch.setattr(ref_shim, "available", lambda: False)
    st, kind, what = bench.make_cpu_stepper(wl, 5, None)
    assert kind == "port" and "cpu_step" in what
    dt, pts, per = bench.time_cpu(st, 0, 1)
    assert pts == 8 * 5 * 27 and dt > 0 and len(per) == 1
