"""Host-side logic that needs no GPU: module/state-dict layout, option plumbing, ray sharding and the
world_size-2 gather (gloo)."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import neuman_b200 as nb
from neuman_b200 import sharding

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_state_dict_layout_matches_reference_names():
    coarse, fine = nb.build_nerf(nb.default_opt(use_cuda=False))
    sd = coarse.state_dict()
    shapes = {k: tuple(v.shape) for k, v in sd.items()}
    assert shapes["nerf.pts_linears.0.weight"] == (256, 63)
    assert shapes["nerf.pts_linears.5.weight"] == (256, 319)
    assert shapes["nerf.views_linears.0.weight"] == (128, 283)
    assert shapes["nerf.feature_linear.weight"] == (256, 256)
    assert shapes["nerf.alpha_linear.weight"] == (1, 256)
    assert shapes["nerf.rgb_linear.weight"] == (3, 128)
    assert sum(v.numel() for v in sd.values()) == 595844            # SURVEY.md §8a row 7
    h = nb.HumanNeRF(nb.default_opt(use_cuda=False))
    keys = list(h.state_dict())
    assert any(k.startswith("coarse_bkg_net.nerf.") for k in keys)
    assert any(k.startswith("fine_bkg_net.nerf.") for k in keys)
    assert any(k.startswith("coarse_human_net.nerf.") for k in keys)
    assert h.coarse_human_net.pos_pe.mapping == "rotate" and h.coarse_bkg_net.pos_pe.mapping == "posenc"


def test_state_dict_keys_equal_reference():
    """The seeded background nets have the reference's keys, shapes and default-init values (tests/golden/reference.npz)."""
    from oracle import scenes
    from tests import util
    g = util.golden("reference.npz")
    pc, pf = scenes.seed_nets(nb.build_nerf, nb.default_opt(use_cuda=False), 1)
    util.assert_state_dict_is_the_references(pc.state_dict(), g, "bsd_coarse")
    util.assert_state_dict_is_the_references(pf.state_dict(), g, "bsd_fine")


@pytest.mark.parametrize("scale_type", ["linear", "tanh", "no"])
def test_offset_net_equals_reference(scale_type):
    """neuman_b200.OffsetNet (library-GEMM forward, models/vanilla.py:169-205) against the reference's OffsetNet with the
    same seeded weights (tests/golden/reference.npz): bit-equal on the CPU, gradients included (sampled)."""
    from tests import util
    g = util.golden("reference.npz")
    opt = nb.default_opt(use_cuda=False, num_offset_nets=1, offset_scale=0.7, offset_scale_type=scale_type)
    torch.manual_seed(3)
    mine = nb.build_offset_net(opt)
    assert list(mine.state_dict()) == [str(k) for k in g[f"off_{scale_type}_sd_keys"]]
    assert [k for k, _ in mine.named_parameters()] == [str(k) for k in g[f"off_{scale_type}_keys"]]
    x = torch.from_numpy(g[f"off_{scale_type}_x"])
    a = mine(x)
    assert a.shape == (40, 6, 3) and torch.equal(a, torch.from_numpy(g[f"off_{scale_type}_y"]))
    a.square().sum().backward()
    for i, (k, p) in enumerate(mine.named_parameters()):
        idx = util.pick(p.grad.numel(), g[f"off_{scale_type}_grads"].shape[1], 200 + i)
        q = torch.from_numpy(g[f"off_{scale_type}_grads"][i, :len(idx)])
        assert torch.allclose(p.grad.reshape(-1)[torch.from_numpy(idx)], q, rtol=1e-5, atol=1e-7), k
        assert abs(p.grad.double().norm().item() - g[f"off_{scale_type}_norms"][i]) <= 1e-5 * g[f"off_{scale_type}_norms"][i] + 1e-7, k


@pytest.mark.parametrize("posenc", ["posenc", "rotate"])
def test_module_interface_layer_by_layer_equals_reference(posenc):
    """SURVEY.md 8b lists Embedder.forward and NeRF.forward among the signatures to preserve: the mirrors evaluate them with
    library ops (the fused kernels serve Joiner.forward); bit-equal to the reference's modules on the CPU, and
    NeRF(Embedder(x), Embedder(v)) == the reference's Joiner (tests/golden/reference.npz)."""
    from oracle import scenes
    from tests import util
    g = {k[len(f"mi_{posenc}_"):]: v for k, v in util.golden("reference.npz").items() if k.startswith(f"mi_{posenc}_")}
    torch.manual_seed(2)
    mine, _ = nb.build_nerf(nb.default_opt(use_cuda=False, posenc=posenc))
    assert abs(scenes.net_checksum(mine) - g["sum"]) <= 1e-9 * g["sum"]
    x, v = torch.from_numpy(g["x"]), torch.from_numpy(g["v"])
    e, d = mine.pos_pe(x), mine.dir_pe(v)
    assert torch.equal(e, torch.from_numpy(g["pos"])) and torch.equal(d, torch.from_numpy(g["dir"]))
    assert e.shape[-1] == 63 and d.shape[-1] == 27
    assert torch.equal(mine.nerf(e, d), torch.from_numpy(g["out"]))


def test_offset_net_joiner_form_stays_on_the_modules_device():
    """Device placement of models.offset_joiner_weights without a GPU: on the `meta` device every intermediate must be
    created on the module's device (mixing in a CPU tensor raises there exactly as it would with CUDA); the architecture
    constants are built once per device and reused; a tensor time works like a float."""
    from neuman_b200 import models
    net = nb.build_offset_net(nb.default_opt(use_cuda=False, num_offset_nets=1, offset_scale_type='tanh'))
    meta = copy_to(net, 'meta')
    for t in (0.3, torch.tensor(0.3, device='meta')):
        W = models.offset_joiner_weights(meta, t)
        assert all(v.device.type == 'meta' for v in W.values())
    j = models.offset_shadow_joiner(meta)
    assert all(p.device.type == 'meta' and not p.requires_grad for p in j.parameters())
    W1, W2 = models.offset_joiner_weights(net, 0.25), models.offset_joiner_weights(net, torch.tensor(0.25))
    assert all(torch.equal(W1[k], W2[k]) for k in W1)
    assert W1['views_linears.0.weight'] is W2['views_linears.0.weight'] and W1['rgb_linear.weight'] is W2['rgb_linear.weight']
    assert not W1['rgb_linear.weight'].requires_grad and W1['feature_linear.weight'].requires_grad
    fresh = nb.build_offset_net(nb.default_opt(use_cuda=False, num_offset_nets=1))
    with torch.inference_mode():                      # constants first built inside inference mode must stay usable by autograd
        models.offset_joiner_weights(fresh, 0.1)
    Wf = models.offset_joiner_weights(fresh, 0.1)
    torch.autograd.grad(sum((v * v).sum() for v in Wf.values() if v.requires_grad), list(fresh.nerf.parameters()))


def copy_to(module, device):
    import copy
    return copy.deepcopy(module).to(device)


def test_shard_ranges_cover_every_pixel_once():
    for n, world in ((921600, 8), (4096, 3), (10, 4), (7, 8), (0, 2)):
        seen = np.zeros(n, dtype=np.int32)
        sizes = []
        for r in range(world):
            p0, cnt = sharding.shard_range(n, r, world)
            seen[p0:p0 + cnt] += 1
            sizes.append(cnt)
        assert (seen == 1).all() and max(sizes) - min(sizes) <= 1


def test_gather_world_size_2_gloo(tmp_path):
    """Two gloo ranks each 'render' their shard (CPU stand-in), all_gather reassembles the frame."""
    script = tmp_path / "w.py"
    script.write_text(f"""
import os, sys, numpy as np, torch, torch.distributed as dist
sys.path.insert(0, {ROOT!r})
from neuman_b200 import sharding
dist.init_process_group('gloo')
rank, world = dist.get_rank(), dist.get_world_size()
n = 1001
p0, cnt = sharding.shard_range(n, rank, world)
local = torch.arange(p0, p0 + cnt, dtype=torch.float32)[:, None].repeat(1, 5)     # fake rgb,depth,acc
frame = sharding.gather_frame(local, n, rank, world)
assert frame.shape == (n, 5) and torch.equal(frame[:, 0], torch.arange(n, dtype=torch.float32))
dist.destroy_process_group()
print('ok', rank)
""")
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                          "--master-addr", "127.0.0.1", "--master-port", "29533", str(script)],
                         capture_output=True, text=True, timeout=300, env=env)
    assert out.returncode == 0, out.stderr[-2000:]
    assert out.stdout.count("ok") == 2


def test_tile_partition_covers_every_pixel_once():
    """SURVEY.md §8e: interleaved 16x16 tiles dealt round-robin; every pixel in exactly one shard, shards balanced to within
    one tile, edge tiles clipped."""
    from neuman_b200 import sharding
    for (H, W) in ((720, 1280), (512, 512), (72, 100), (5, 7)):
        for world in (1, 2, 3, 8):
            seen = np.zeros(H * W, np.int32)
            sizes = []
            for r in range(world):
                p = sharding.tile_pixels(H, W, r, world)
                assert p.dtype == np.int32 and (p >= 0).all() and (p < H * W).all()
                seen[p] += 1
                sizes.append(p.size)
            assert (seen == 1).all()
            if (H, W) in ((720, 1280), (512, 512)) and world != 3:
                assert max(sizes) == min(sizes)                          # BASELINE.json's frames split evenly over 1/2/4/8 GPUs
            assert max(sizes) - min(sizes) <= 2 * sharding.TILE * sharding.TILE
    # a tile is 16 consecutive pixels of 16 consecutive rows
    p = sharding.tile_pixels(720, 1280, 3, 8)
    assert p[0] == 3 * 16 and p[15] == 3 * 16 + 15 and p[16] == 1280 + 3 * 16


def test_tile_shards_gather_world_size_2_gloo(tmp_path):
    """Two gloo ranks fill their tile shards (CPU stand-in for the renderers), ONE all_gather of the equal-sized shards
    moves them, and the pixel lists put every value back (the CPU restatement of nm_assemble_frame)."""
    script = tmp_path / "w.py"
    script.write_text(f"""
import os, sys, numpy as np, torch, torch.distributed as dist
sys.path.insert(0, {ROOT!r})
from neuman_b200 import sharding
dist.init_process_group('gloo')
rank, world = dist.get_rank(), dist.get_world_size()
H, W, planes = 72, 100, 5
lists = [sharding.tile_pixels(H, W, r, world) for r in range(world)]
per = max(x.size for x in lists)
mine = torch.from_numpy(lists[rank]).long()
shard = torch.zeros(planes * per)
n = mine.numel()
shard[:3 * per][:3 * n].view(n, 3)[:] = torch.stack([mine * 3.0, mine * 3.0 + 1, mine * 3.0 + 2], 1)      # fake rgb
shard[3 * per:4 * per][:n] = mine + 0.25                                                                 # fake depth
shard[4 * per:5 * per][:n] = mine + 0.5                                                                  # fake acc
gathered = torch.empty(world * planes * per)
dist.all_gather_into_tensor(gathered, shard)
rgb, depth, acc = torch.full((H * W, 3), -1.0), torch.full((H * W,), -1.0), torch.full((H * W,), -1.0)
for r in range(world):
    base = gathered[r * planes * per:(r + 1) * planes * per]
    idx = torch.from_numpy(lists[r]).long()
    m = idx.numel()
    rgb[idx] = base[:3 * per][:3 * m].view(m, 3)
    depth[idx] = base[3 * per:4 * per][:m]
    acc[idx] = base[4 * per:5 * per][:m]
pix = torch.arange(H * W, dtype=torch.float32)
assert torch.equal(rgb, torch.stack([pix * 3, pix * 3 + 1, pix * 3 + 2], 1)) and torch.equal(depth, pix + 0.25) and torch.equal(acc, pix + 0.5)
dist.destroy_process_group()
print('ok', rank)
""")
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                          "--master-addr", "127.0.0.1", "--master-port", "29534", str(script)],
                         capture_output=True, text=True, timeout=300, env=env)
    assert out.returncode == 0, out.stderr[-2000:]
    assert out.stdout.count("ok") == 2


@pytest.mark.reference
def test_install_rebinds_reference_modules():
    from oracle import ref_import
    ref_import.load()
    mods = nb.install()
    assert mods["render_utils"].render_vanilla.__name__ == "render_vanilla"
    # CPU tensors keep using the reference implementation (training / CPU path untouched)
    raw, z, d = torch.randn(3, 5, 4), torch.sort(torch.rand(3, 5))[0], torch.randn(3, 3)
    from oracle import neuman_oracle as no
    out = mods["render_utils"].raw2outputs(raw, z, d)
    exp = no.raw2outputs(raw, z, d)
    assert torch.allclose(out[0], exp[0])


@pytest.mark.reference
def test_install_train_switch_keeps_cpu_paths_on_the_reference():
    """install(train=True) wraps the trainers' entry points (Joiner.forward, raw2outputs, the samplers,
    warp_samples_to_canonical_diff); with CPU tensors / grads every wrapper must fall through to the reference code."""
    from oracle import ref_import, ref_opts
    ref = ref_import.load()
    mods = nb.install(train=True)
    ru, ry, mv = mods["render_utils"], mods["ray_utils"], mods["vanilla"]
    assert ry.warp_samples_to_canonical_diff.__name__ == "warp_samples_to_canonical_diff"
    torch.manual_seed(0)
    raw = torch.randn(3, 5, 4, requires_grad=True)
    z, d = torch.sort(torch.rand(3, 5))[0], torch.randn(3, 3)
    rgb = ru.raw2outputs(raw, z, d)[0]
    rgb.sum().backward()                                  # reference torch ops: autograd works on the CPU
    assert raw.grad is not None and torch.isfinite(raw.grad).all()
    coarse, _ = mv.build_nerf(ref_opts.default_opt(use_cuda=False))
    out = coarse(torch.randn(7, 3), torch.randn(7, 3))
    assert out.shape == (7, 4) and out.requires_grad
    batch = {'origin': torch.zeros(4, 3), 'direction': torch.randn(4, 3), 'near': torch.ones(4, 1) * 0.5, 'far': torch.ones(4, 1) * 2}
    pts, dirs, zv = ry.ray_to_samples(batch, 6)
    assert pts.shape == (4, 6, 3) and zv.shape == (4, 6)


def test_frame_metrics_match_the_oracle(tmp_path):
    """neuman_b200.metrics (render_test_views.py:27-41,88) against the scipy restatement of the scikit-image formulas."""
    from neuman_b200 import metrics
    from oracle import metrics_oracle as mo
    rng = np.random.RandomState(0)
    gt = rng.randint(0, 256, (37, 53, 3)).astype(np.uint8)
    noise = rng.normal(0, 12, gt.shape)
    pred = np.clip(gt.astype(np.float64) + noise, 0, 255).astype(np.uint8)
    assert abs(metrics.psnr(gt, pred) - mo.peak_signal_noise_ratio(gt, pred)) < 1e-9
    assert abs(metrics.ssim(pred, gt) - mo.structural_similarity(pred, gt)) < 1e-9
    assert abs(metrics.ssim(gt, gt) - 1.0) < 1e-12
    f = rng.uniform(-0.1, 1.1, (5, 7, 3)).astype(np.float32)
    u = metrics.to_uint8(f).numpy()
    assert u.dtype == np.uint8 and np.array_equal(u, np.floor(np.clip(f.astype(np.float64), 0, 1) * 255 + 0.5).astype(np.uint8))
    metrics.save_png(str(tmp_path / "a.png"), f)
    from PIL import Image
    assert np.array_equal(np.asarray(Image.open(tmp_path / "a.png")), u)
    r = metrics.eval_metrics([gt, gt], [pred, gt])
    assert set(r) == {"ssim", "psnr"} and np.isinf(r["psnr"])


def test_frame_metrics_against_opencv(tmp_path):
    """Third-party pins available in this image (scikit-image / imageio are not): OpenCV's own PSNR for uint8 frames
    (cv2.PSNR, R = 255) and its PNG decoder on the file save_png wrote; SSIM's window means against cv2.blur's box filter
    (an independent implementation of the uniform window the scikit-image formula averages over)."""
    cv2 = pytest.importorskip("cv2")
    from neuman_b200 import metrics
    rng = np.random.RandomState(1)
    gt = rng.randint(0, 256, (41, 57, 3)).astype(np.uint8)
    pred = np.clip(gt.astype(np.float64) + rng.normal(0, 9, gt.shape), 0, 255).astype(np.uint8)
    assert abs(metrics.psnr(gt, pred) - cv2.PSNR(gt, pred)) < 1e-9
    f = rng.uniform(0, 1, (9, 11, 3)).astype(np.float32)
    metrics.save_png(str(tmp_path / "b.png"), f)
    bgr = cv2.imread(str(tmp_path / "b.png"), cv2.IMREAD_COLOR)
    assert np.array_equal(bgr[..., ::-1], metrics.to_uint8(f).numpy())
    # SSIM of one channel from cv2's box filter (BORDER_REFLECT_101 borders are cropped away exactly as scikit-image crops)
    x, y = pred[..., 0].astype(np.float64), gt[..., 0].astype(np.float64)
    box = lambda a: cv2.blur(a, (7, 7))[3:-3, 3:-3]
    ux, uy = box(x), box(y)
    cn = 49 / 48.0
    vx, vy, vxy = cn * (box(x * x) - ux * ux), cn * (box(y * y) - uy * uy), cn * (box(x * y) - ux * uy)
    C1, C2 = (0.01 * 255) ** 2, (0.03 * 255) ** 2
    S = ((2 * ux * uy + C1) * (2 * vxy + C2)) / ((ux ** 2 + uy ** 2 + C1) * (vx + vy + C2))
    assert abs(metrics.ssim(pred[..., :1], gt[..., :1]) - S.mean()) < 1e-9


def test_lpips_restatement_structure_and_formula():
    """neuman_b200.metrics.LPIPS (render_test_views.py:19,36-38; trainers/human_nerf_trainer.py:152,432-435).  The package
    and its weights are absent (parity UNPINNED); what can be checked here: the package's parameter names, the feature
    stack against torchvision's AlexNet with the same weights, the distance against a numpy restatement of the published
    formula, and the two call sites' tensor conventions."""
    torchvision = pytest.importorskip("torchvision")
    from neuman_b200 import metrics
    m = metrics.LPIPS()
    keys = list(m.state_dict())
    want = ['scaling_layer.shift', 'scaling_layer.scale']
    for sl, idx in ((1, 0), (2, 3), (3, 6), (4, 8), (5, 10)):
        want += [f'net.slice{sl}.{idx}.weight', f'net.slice{sl}.{idx}.bias']
    want += [f'lin{k}.model.1.weight' for k in range(5)] + [f'lins.{k}.model.1.weight' for k in range(5)]
    assert keys == want and not m.training and not m.pretrained
    torch.manual_seed(0)
    alex = torchvision.models.alexnet(weights=None).eval()
    lin = {f'lin{k}.model.1.weight': torch.rand(1, c, 1, 1) for k, c in enumerate(metrics.LPIPS.CHNS)}
    m.load_pretrained(alex.state_dict(), lin)
    assert m.pretrained
    x, y = torch.rand(2, 3, 64, 48) * 2 - 1, torch.rand(2, 3, 64, 48) * 2 - 1
    # feature stack == torchvision's features at its five ReLUs
    h, taps = m.scaling_layer(x), []
    for i, layer in enumerate(alex.features[:12]):
        h = layer(h)
        if i in (1, 4, 7, 9, 11):
            taps.append(h)
    for a, b in zip(m.net(m.scaling_layer(x)), taps):
        assert torch.equal(a, b)
    # distance == the published formula, restated in numpy
    with torch.no_grad():
        got = m(x, y).numpy()
        fx, fy = [t.numpy() for t in m.net(m.scaling_layer(x))], [t.numpy() for t in m.net(m.scaling_layer(y))]
    val = np.zeros((2, 1, 1, 1))
    for k in range(5):
        ux = fx[k] / (np.sqrt((fx[k] ** 2).sum(1, keepdims=True)) + 1e-10)
        uy = fy[k] / (np.sqrt((fy[k] ** 2).sum(1, keepdims=True)) + 1e-10)
        w = lin[f'lin{k}.model.1.weight'].numpy()[0][None]
        val += (((ux - uy) ** 2) * w).sum(1, keepdims=True).mean((2, 3), keepdims=True)
    assert np.abs(got - val).max() < 1e-6
    with torch.no_grad():
        assert float(m(x, x).abs().max()) == 0.0
        assert torch.allclose(m((x + 1) / 2, (y + 1) / 2, normalize=True), m(x, y), atol=1e-6)
    # the trainer's patch term: first 1024 rays of the batch, unbatched [3,32,32] tensors (:432-435)
    rgb, col = torch.rand(1400, 3, requires_grad=True), torch.rand(1400, 3)
    loss = metrics.lpips_patch_loss(m, rgb, col)
    assert loss.dim() == 0 and loss.requires_grad
    loss.backward()
    assert rgb.grad[:1024].abs().max() > 0 and rgb.grad[1024:].abs().max() == 0
    # the evaluation script's call (uint8 frames -> /127.5 - 1)
    rng = np.random.RandomState(0)
    gt = rng.randint(0, 256, (40, 56, 3)).astype(np.uint8)
    pred = np.clip(gt + rng.normal(0, 10, gt.shape), 0, 255).astype(np.uint8)
    r = metrics.eval_metrics([gt], [pred], lpips_fn=m)
    with torch.no_grad():
        ref_val = float(m(torch.from_numpy(pred).permute(2, 0, 1)[None].float() / 127.5 - 1,
                          torch.from_numpy(gt).permute(2, 0, 1)[None].float() / 127.5 - 1)[0, 0, 0, 0])
    assert set(r) == {"ssim", "psnr", "lpips"} and abs(r["lpips"] - ref_val) < 1e-7 and r["lpips"] > 0


def test_batchers_host_logic_equals_the_reference_datasets(monkeypatch):
    """The host logic of neuman_b200.data (segment plan, patch window, gathers, near/far cache lookup, dtypes) on CPU
    tensors against the batches the UNMODIFIED reference datasets produced (tests/golden/batches.npz): the ray kernel
    (ops.shot_rays -> nm_raygen) is substituted by the oracle here; tests/test_gpu_train.py runs the same comparison
    through the CUDA library."""
    import numpy as np
    import torch
    from neuman_b200 import data as nd, ops
    from oracle import neuman_oracle as no
    from tests import test_gpu_train as T, util

    def oracle_shot_rays(cap, xy, device=None):
        o, d = no.shot_rays(cap.intrinsic_matrix, cap.cam_pose.camera_to_world, xy.cpu().numpy())
        return torch.from_numpy(np.asarray(o, dtype=np.float32)), torch.from_numpy(np.asarray(d, dtype=np.float32))
    g = util.golden("batches.npz")
    B, H = nd.BackgroundRayBatcher, nd.HumanRayBatcher
    monkeypatch.setattr(ops, "shot_rays", oracle_shot_rays)
    monkeypatch.setattr(torch.Tensor, "cuda", lambda self, *a, **k: self)
    monkeypatch.setattr(nd, "BackgroundRayBatcher", lambda opt, caps: B(opt, caps, device="cpu"))
    monkeypatch.setattr(nd, "HumanRayBatcher", lambda opt, caps, nf: H(opt, caps, nf, device="cpu"))
    monkeypatch.setattr(nd, "near_far_cache_device",
                        lambda cap, verts, thr: torch.from_numpy(g["hu_cap%d_cache" % (0 if cap.image.shape[0] == 48 else 1)]))
    T.test_background_batches_equal_the_reference_dataset()
    T.test_human_batches_equal_the_reference_dataset()


@pytest.mark.parametrize("t", [0.0, 3 / 11, 0.97])
def test_offset_net_as_joiner_weights_are_equivalent(t):
    """models.offset_joiner_weights: for a fixed time the offset network IS a Joiner on (x, y, z) -- time channels folded
    into the layer-0 / skip-layer biases, output_linear carried through the non-negative head as relu(y) - relu(-y).  The
    oracle's Joiner on the synthesized weights must reproduce the library forward, gradients to the offset net's own
    parameters included (autograd through the synthesis)."""
    from neuman_b200 import models
    from oracle import neuman_oracle as no
    opt = nb.default_opt(use_cuda=False, num_offset_nets=1, offset_scale=0.7, offset_scale_type='tanh', pos_min_freq=0)
    torch.manual_seed(5)
    net = nb.build_offset_net(opt)
    assert net.tc_supported()
    x = torch.randn(300, 3)
    lib = net(torch.cat([x, torch.full((300, 1), t)], -1))
    W = net.joiner_weights(t)
    j = models.offset_shadow_joiner(net)
    assert sorted(W) == sorted(k for k, _ in j.nerf.named_parameters())
    assert all(tuple(W[k].shape) == tuple(p.shape) for k, p in j.nerf.named_parameters())
    assert len(net.state_dict()) == 18 and not any("shadow" in k for k in net.state_dict())      # checkpoints unchanged
    P = no.NetParams(sd={'nerf.' + k: v for k, v in W.items()},
                     pos_pe=no.PESpec(kind='posenc', min_freq=0.0, max_freq=9.0, n_freqs=10, include_input=True))
    raw = no.net_forward(P, x, torch.zeros_like(x))
    out = models._offset_scaled(net, raw[:, :3])
    assert (out - lib).abs().max() < 1e-6
    w = torch.randn(300, 3)
    params = list(net.nerf.parameters())
    g1 = torch.autograd.grad((lib * w).sum(), params, retain_graph=True)
    g2 = torch.autograd.grad((out * w).sum(), params)
    for a, b in zip(g1, g2):
        assert (a - b).abs().max() < 1e-5 * (1 + a.abs().max())
    xyz, tt = models.offset_channel_split(10)
    assert sorted(xyz + tt) == list(range(84)) and len(xyz) == 63
