"""Generates tests/golden/reference.npz: what the UNMODIFIED reference computes on exactly the inputs of
tests/test_oracle_vs_reference.py and of the reference comparisons in tests/test_host.py, so that those tests compare the
oracle and the host mirrors against the reference without importing it.  Run where the reference tree is readable:

    python tools/make_golden_reference.py

Inputs drawn from a random generator are stored next to the outputs.  Networks are not stored (too large): the tests
rebuild them with the host mirrors (neuman_b200.models) from the same seeds, and the fixture holds, per tensor, the
float64 sum, the float64 sum of absolute values and the values at 32 seeded positions of the reference's own weights.
Arrays that are larger than the comparison needs (per-vertex SMPL outputs) are stored as a seeded sample of rows.
"""
import contextlib
import io
import os
import sys
import tempfile

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_import, ref_opts, scenes, synth_smpl      # noqa: E402
from tests.util import pick                                      # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "reference.npz")
N_PICK = 32          # sampled values per weight tensor or gradient (tests/util.py: pick)
N_ROWS = 128         # sampled rows of per-vertex arrays


def quiet(fn, *a, **k):
    with contextlib.redirect_stdout(io.StringIO()):
        return fn(*a, **k)


def cap_of(ref, K, c2w, H, W, near=0.0, far=3.14):
    cam = ref.pinhole_camera.PinholeCamera(W, H, K[0, 0], K[1, 1], K[0, 2], K[1, 2])
    pose = ref.camera_pose.CameraPose.from_camera_to_world(c2w.astype(np.float64))
    cap = ref.captures.BasePinholeCapture(cam, pose)
    cap.near, cap.far = {"bkg": near}, {"bkg": far}
    return cap


def camera(H, W, f=None, seed=0):
    """The camera of tests/test_oracle_vs_reference.py."""
    rng = np.random.RandomState(seed)
    f = f or 1000.0 * W / 1280
    K = np.array([[f, 0, W / 2], [0, f, H / 2], [0, 0, 1.0]])
    a = rng.uniform(-0.2, 0.2)
    R = np.array([[np.cos(a), 0, np.sin(a)], [0, 1, 0], [-np.sin(a), 0, np.cos(a)]])
    c2w = np.eye(4)
    c2w[:3, :3] = R
    c2w[:3, 3] = [0.1, -0.05, -1.5]
    return K, c2w


def state_digest(g, prefix, sd):
    """Keys, shapes, float64 sum / abs-sum and N_PICK seeded values (NaN-padded) of every tensor of a state dict."""
    keys = list(sd)
    g[f"{prefix}_keys"] = np.array(keys)
    g[f"{prefix}_shapes"] = np.array(["x".join(map(str, sd[k].shape)) for k in keys])
    g[f"{prefix}_sums"] = np.array([[sd[k].double().sum().item(), sd[k].double().abs().sum().item()] for k in keys])
    vals = np.full((len(keys), N_PICK), np.nan, dtype=np.float32)
    for i, k in enumerate(keys):
        v = sd[k].detach().cpu().reshape(-1)
        idx = pick(v.numel(), N_PICK, i)
        vals[i, :len(idx)] = v[torch.from_numpy(idx)].numpy()
    g[f"{prefix}_vals"] = vals


def human_net(ref):
    """tests/test_oracle_vs_reference.py::_reference_human_net."""
    torch.manual_seed(1)
    net = quiet(ref.human_nerf.HumanNeRF, ref_opts.default_opt(num_offset_nets=1))
    rng = np.random.RandomState(6)
    pose, betas = rng.normal(0, 0.3, (1, 72)).astype(np.float32), rng.normal(0, 1, (1, 10)).astype(np.float32)
    align = np.eye(4, dtype=np.float32)
    align[:3, :3] = np.array([[np.cos(0.2), 0, np.sin(0.2)], [0, 1, 0], [-np.sin(0.2), 0, np.cos(0.2)]])
    align = align.T.copy()
    align[3, :3] = (0.3, -0.1, 2.0)
    P = torch.nn.Parameter
    net.poses, net.betas, net.alignments, net.scale = P(torch.from_numpy(pose)), P(torch.from_numpy(betas)), P(torch.from_numpy(align[None])), 0.4
    pk = os.path.join(tempfile.mkdtemp(), "SMPL_NEUTRAL.pkl")
    synth_smpl.write_pickle(pk, 0)
    net.body_model = ref.smpl.SMPL(pk, gender="neutral", device=torch.device("cpu"))
    da = torch.zeros(24, 3)
    da[1, 2], da[2, 2] = 1.0, -1.0
    net.da_smpl = P(da.reshape(1, -1), requires_grad=False)
    return net


def oracle_vs_reference(ref, g):
    # rays
    H, W = 12, 20
    K, c2w = camera(H, W)
    cap = cap_of(ref, K, c2w, H, W)
    g["rays_K"], g["rays_c2w"] = cap.intrinsic_matrix, cap.cam_pose.camera_to_world
    xy = np.argwhere(np.ones((H, W)))[:, ::-1]
    g["rays_o"], g["rays_d"] = ref.ray_utils.shot_rays(cap, xy)
    g["rays_all_o"], g["rays_all_d"] = ref.ray_utils.shot_all_rays(cap)

    # sampling / composite
    torch.manual_seed(0)
    R, S, N = 37, 24, 16
    o, d = torch.randn(R, 3), torch.nn.functional.normalize(torch.randn(R, 3), dim=-1)
    near, far = torch.rand(R, 1), 2 + torch.rand(R, 1)
    batch = {"origin": o, "direction": d, "near": near, "far": far}
    p, v, z = ref.ray_utils.ray_to_samples(batch, S)
    raw = torch.randn(R, S, 4) * 3
    out = ref.render_utils.raw2outputs(raw, z, d, white_bkg=True)
    ip, _, iz = ref.ray_utils.ray_to_importance_samples(batch, z, out[3], N)
    torch.manual_seed(5)
    _, _, zp = ref.ray_utils.ray_to_samples(batch, S, perturb=1.0)
    g.update(sc_o=o.numpy(), sc_d=d.numpy(), sc_near=near.numpy(), sc_far=far.numpy(), sc_raw=raw.numpy(),
             sc_pts=p.numpy(), sc_views=v.numpy(), sc_z=z.numpy(), sc_imp_pts=ip.numpy(), sc_imp_z=iz.numpy(),
             sc_z_perturb=zp.numpy())
    for name, t in zip(("rgb", "disp", "acc", "w", "depth"), out):
        g[f"sc_{name}"] = t.numpy()

    # networks
    torch.manual_seed(1)
    coarse, fine = ref.vanilla.build_nerf(ref_opts.default_opt())
    human, _ = ref.vanilla.build_nerf(ref_opts.default_opt(posenc="rotate"))
    pts, views = torch.randn(50, 7, 3), torch.nn.functional.normalize(torch.randn(50, 7, 3), dim=-1)
    g.update(net_pts=pts.numpy(), net_views=views.numpy())
    with torch.no_grad():
        for name, net in (("coarse", coarse), ("fine", fine), ("human", human)):
            g[f"net_{name}_out"] = net(pts, views).numpy()
            g[f"net_{name}_sum"] = np.float64(scenes.net_checksum(net))

    # near / far
    rng = np.random.RandomState(0)
    V = rng.normal(0, 0.3, size=(500, 3)).astype(np.float32)
    o = np.tile(np.array([[0, 0, -2.0]], dtype=np.float32), (64, 1))
    d = rng.normal(0, 0.3, size=(64, 3)).astype(np.float32) + np.array([0, 0, 1], dtype=np.float32)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    g["nf_near_np"], g["nf_far_np"] = ref.ray_utils.geometry_guided_near_far(o, d, V, 0.1)
    n, f = ref.ray_utils.geometry_guided_near_far(torch.from_numpy(o), torch.from_numpy(d), torch.from_numpy(V), 0.1)
    g["nf_near_t"], g["nf_far_t"] = n.numpy(), f.numpy()

    # SMPL
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "SMPL_NEUTRAL.pkl")
        synth_smpl.write_pickle(path)
        body = ref.smpl.SMPL(path, gender="neutral", device=torch.device("cpu"))
    rng = np.random.RandomState(3)
    pose = torch.from_numpy(rng.normal(0, 0.3, (1, 72))).float()
    betas = torch.from_numpy(rng.normal(0, 1, (1, 10))).float()
    v_r, T_r = body.verts_transformations(pose, betas, concat_joints=True)
    verts_r, joints_r = body(pose, betas, return_joints=True)
    rows = pick(T_r.shape[1], N_ROWS, 100)
    vrows = pick(verts_r.shape[1], N_ROWS, 101)
    g.update(smpl_pose=pose.numpy(), smpl_betas=betas.numpy(), smpl_T=T_r[0].numpy()[rows],
             smpl_v=v_r[0].numpy()[rows], smpl_verts=verts_r[0].numpy()[vrows], smpl_joints=joints_r[0].numpy())

    # warp
    b = synth_smpl.random_body(seed=2)
    rng = np.random.RandomState(0)
    pw = (b["verts"].mean(0) + rng.normal(0, 0.25, size=(6, 9, 3))).astype(np.float32)
    faces6 = np.concatenate([b["faces"], b["faces"]], 1)
    g["warp_pts"] = pw
    g["warp_can"], g["warp_dirs"], g["warp_closest"] = ref.ray_utils.warp_samples_to_canonical(pw, b["verts"], faces6, b["Ts"])

    # frame drivers
    torch.manual_seed(1)
    coarse, fine = ref.vanilla.build_nerf(ref_opts.default_opt())
    g["rv_sum"] = np.array([scenes.net_checksum(coarse), scenes.net_checksum(fine)])
    H, W = 6, 9
    K, c2w = camera(H, W)
    cap = cap_of(ref, K, c2w, H, W)
    g["rv_K"], g["rv_c2w"] = cap.intrinsic_matrix, cap.cam_pose.camera_to_world
    g["rv_rgb"], g["rv_depth"] = quiet(ref.render_utils.render_vanilla, coarse, cap, fine_net=fine, rays_per_batch=32,
                                       samples_per_ray=16, importance_samples_per_ray=8, return_depth=True)
    torch.manual_seed(1)
    net = quiet(ref.human_nerf.HumanNeRF, ref_opts.default_opt())
    scenes.boost_density(net.coarse_human_net)
    g["hum_sum"] = np.array([scenes.net_checksum(j) for j in (net.coarse_bkg_net, net.fine_bkg_net, net.coarse_human_net)])
    body = synth_smpl.random_body(seed=1, center=(0.1, 0.0, 0.3))
    body2 = synth_smpl.random_body(seed=4, center=(-0.2, 0.0, 0.5))
    H, W = 10, 8
    K, c2w = camera(H, W, f=14.0)
    cap = cap_of(ref, K, c2w, H, W)
    g["hum_K"], g["hum_c2w"] = cap.intrinsic_matrix, cap.cam_pose.camera_to_world
    faces, geo = body["faces"], body["geo_threshold"]
    for can in (True, False):
        r, dd, a = quiet(ref.render_utils.render_smpl_nerf, net, cap, body["verts"], faces, body["Ts"], rays_per_batch=32,
                         samples_per_ray=12, render_can=can, geo_threshold=geo, return_depth=True, return_mask=True,
                         interval_comp=0.7)
        g.update({f"hum_smpl{int(can)}_rgb": r, f"hum_smpl{int(can)}_depth": dd, f"hum_smpl{int(can)}_acc": a})
    g["hum_hyb_rgb"], g["hum_hyb_depth"] = quiet(ref.render_utils.render_hybrid_nerf, net, cap, body["verts"], faces, body["Ts"],
                                                 rays_per_batch=32, samples_per_ray=12, importance_samples_per_ray=8,
                                                 geo_threshold=geo, return_depth=True)
    g["hum_multi_rgb"], g["hum_multi_depth"] = quiet(
        ref.render_utils.render_hybrid_nerf_multi_persons, net, cap, [net, net], [body["verts"], body2["verts"]], [faces, faces],
        [body["Ts"], body2["Ts"]], rays_per_batch=32, samples_per_ray=12, importance_samples_per_ray=8, geo_threshold=geo,
        return_depth=True)

    # HumanNeRF state dict (two offset nets)
    torch.manual_seed(11)
    state_digest(g, "hsd", quiet(ref.human_nerf.HumanNeRF, ref_opts.default_opt(num_offset_nets=2)).state_dict())

    # vertex_forward and its gradients
    net = human_net(ref)
    w_r, T_r = net.vertex_forward(0)
    rng = np.random.RandomState(0)
    g1 = rng.normal(0, 1, tuple(T_r.shape)).astype(np.float32)
    g2 = rng.normal(0, 1, tuple(w_r.shape)).astype(np.float32)
    ((T_r * torch.from_numpy(g1)).sum() + (w_r * torch.from_numpy(g2)).sum()).backward()
    rows = pick(T_r.reshape(-1, 4, 4).shape[0], N_ROWS, 102)
    wrows = pick(w_r.reshape(-1, 3).shape[0], N_ROWS, 103)
    g.update(vf_T=T_r.detach().reshape(-1, 4, 4).numpy()[rows], vf_w=w_r.detach().reshape(-1, 3).numpy()[wrows], vf_T_shape=np.array(tuple(T_r.shape)),
             vf_w_shape=np.array(tuple(w_r.shape)), vf_grad_poses=net.poses.grad.numpy(),
             vf_grad_betas=net.betas.grad.numpy(), vf_grad_alignments=net.alignments.grad.numpy())

    # differentiable warp
    b = synth_smpl.random_body(seed=3)
    V = torch.from_numpy(b["verts"]).float().requires_grad_(True)
    F = np.asarray(b["faces"])[:, :3]
    T = torch.from_numpy(b["Ts"][:6890]).float().requires_grad_(True)
    rng = np.random.RandomState(0)
    P = (b["verts"][rng.randint(0, 6890, 400)] + rng.normal(0, 0.03, (400, 3))).astype(np.float32)
    Ti, f_id, _ = ref.ray_utils.warp_samples_to_canonical_diff(P, V, F, T)
    g["wd_Tinv"], g["wd_face"] = Ti.detach().numpy(), np.asarray(f_id)


def host_mirrors(ref, g):
    # background nets' state dicts (tests/test_host.py::test_state_dict_keys_equal_reference)
    rc, rf = scenes.seed_nets(ref.vanilla.build_nerf, ref_opts.default_opt(), 1)
    state_digest(g, "bsd_coarse", rc.state_dict())
    state_digest(g, "bsd_fine", rf.state_dict())

    # OffsetNet forward and gradients on the host mirror's seeded weights
    import neuman_b200 as nb
    for st in ("linear", "tanh", "no"):
        opt = nb.default_opt(use_cuda=False, num_offset_nets=1, offset_scale=0.7, offset_scale_type=st)
        torch.manual_seed(3)
        mine = nb.build_offset_net(opt)
        theirs = ref.vanilla.build_offset_net(opt)
        theirs.load_state_dict(mine.state_dict())
        x = torch.randn(40, 6, 4)
        y = theirs(x)
        y.square().sum().backward()
        g[f"off_{st}_x"], g[f"off_{st}_y"] = x.numpy(), y.detach().numpy()
        g[f"off_{st}_sd_keys"] = np.array(list(theirs.state_dict()))
        g[f"off_{st}_keys"] = np.array([k for k, _ in theirs.named_parameters()])
        params = list(theirs.parameters())
        grads = np.full((len(params), N_PICK), np.nan, dtype=np.float32)
        for i, p in enumerate(params):
            idx = pick(p.grad.numel(), N_PICK, 200 + i)
            grads[i, :len(idx)] = p.grad.reshape(-1)[torch.from_numpy(idx)].numpy()
        g[f"off_{st}_grads"] = grads
        g[f"off_{st}_norms"] = np.array([p.grad.double().norm().item() for p in params])

    # Embedder / NeRF / Joiner layer by layer
    for posenc in ("posenc", "rotate"):
        torch.manual_seed(2)
        theirs, _ = ref.vanilla.build_nerf(ref_opts.default_opt(posenc=posenc))
        for pe in (theirs.pos_pe, theirs.dir_pe):
            if hasattr(pe, "bvals"):
                pe.bvals = pe.bvals.cpu()
        x, v = torch.randn(7, 5, 3), torch.randn(7, 5, 3)
        with torch.no_grad():
            g.update({f"mi_{posenc}_x": x.numpy(), f"mi_{posenc}_v": v.numpy(), f"mi_{posenc}_pos": theirs.pos_pe(x).numpy(),
                      f"mi_{posenc}_dir": theirs.dir_pe(v).numpy(), f"mi_{posenc}_out": theirs(x, v).numpy()})
        g[f"mi_{posenc}_sum"] = np.float64(scenes.net_checksum(theirs))


def main():
    ref = ref_import.load()
    g = {}
    oracle_vs_reference(ref, g)
    host_mirrors(ref, g)
    np.savez_compressed(OUT, **g)
    print(OUT, os.path.getsize(OUT) // 1024, "KiB,", len(g), "arrays")


if __name__ == "__main__":
    main()
