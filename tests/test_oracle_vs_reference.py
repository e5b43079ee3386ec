"""The oracle restatement (oracle/neuman_oracle.py) against what the UNMODIFIED reference computed on the same inputs
(tests/golden/reference.npz, written by tools/make_golden_reference.py).  Networks are rebuilt with the host mirrors
from the reference's seeds; their weights are first checked against the reference's (checksums, sampled values)."""
import numpy as np
import torch

import neuman_b200 as nb
from oracle import neuman_oracle as no
from oracle import scenes, synth_smpl
from tests import util

G = util.golden("reference.npz")
ROWS = 128                                   # tools/make_golden_reference.py: N_ROWS


def test_rays_match():
    H, W = 12, 20
    xy = no.all_pixel_coords(H, W)
    assert np.array_equal(xy, np.argwhere(np.ones((H, W)))[:, ::-1])
    o, d = no.shot_rays(G["rays_K"], G["rays_c2w"], xy)
    assert np.array_equal(o, G["rays_o"]) and np.array_equal(d, G["rays_d"])
    o, d = no.shot_all_rays(G["rays_K"], G["rays_c2w"], H, W)
    assert np.array_equal(o, G["rays_all_o"]) and np.array_equal(d, G["rays_all_d"])


def test_sampling_composite_match():
    t = {k[3:]: torch.from_numpy(v) for k, v in G.items() if k.startswith("sc_")}
    S, N = t["z"].shape[1], t["imp_z"].shape[1] - t["z"].shape[1]
    p, v, z = no.ray_to_samples(t["o"], t["d"], t["near"], t["far"], S)
    assert torch.equal(p, t["pts"]) and torch.equal(v, t["views"]) and torch.equal(z, t["z"])
    out = no.raw2outputs(t["raw"], z, t["d"], white_bkg=True)
    for name, a in zip(("rgb", "disp", "acc", "w", "depth"), out):
        assert torch.equal(a, t[name]), name
    p, v, z2 = no.ray_to_importance_samples(t["o"], t["d"], z, out[3], N)
    assert torch.equal(z2, t["imp_z"]) and torch.equal(p, t["imp_pts"])
    # stratified: the reference drew its offsets from the global RNG right after torch.manual_seed(5)
    torch.manual_seed(5)
    _, _, zp = no.ray_to_samples(t["o"], t["d"], t["near"], t["far"], S, perturb=1.0)
    assert torch.equal(zp, t["z_perturb"])


def test_nets_match():
    torch.manual_seed(1)
    coarse, fine = nb.build_nerf(nb.default_opt(use_cuda=False))
    human, _ = nb.build_nerf(nb.default_opt(use_cuda=False, posenc="rotate"))
    pts, views = torch.from_numpy(G["net_pts"]), torch.from_numpy(G["net_views"])
    for name, net in (("coarse", coarse), ("fine", fine), ("human", human)):
        assert abs(scenes.net_checksum(net) - G[f"net_{name}_sum"]) <= 1e-9 * G[f"net_{name}_sum"], name
        with torch.no_grad():
            y = no.net_forward(no.net_params_from_joiner(net), pts, views)
        y_r = torch.from_numpy(G[f"net_{name}_out"])
        assert torch.allclose(y, y_r, atol=1e-6, rtol=0), (y - y_r).abs().max()


def test_near_far_match():
    rng = np.random.RandomState(0)
    V = rng.normal(0, 0.3, size=(500, 3)).astype(np.float32)
    o = np.tile(np.array([[0, 0, -2.0]], dtype=np.float32), (64, 1))
    d = rng.normal(0, 0.3, size=(64, 3)).astype(np.float32) + np.array([0, 0, 1], dtype=np.float32)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    n_r, f_r = G["nf_near_np"], G["nf_far_np"]
    n, f = no.geometry_guided_near_far(o, d, V, 0.1)
    # the discriminant thr^2-(|ov|^2-z0^2) cancels catastrophically; numpy and torch round it
    # differently (reference noise floor ~4e-6), so the two branches agree to 2e-5, same hit set
    assert np.array_equal(np.isinf(n), np.isinf(n_r))
    hit = ~np.isinf(n)
    assert np.allclose(n[hit], n_r[hit], atol=2e-5) and np.allclose(f[hit], f_r[hit], atol=2e-5)
    n_r, f_r = torch.from_numpy(G["nf_near_t"]), torch.from_numpy(G["nf_far_t"])
    n, f = no.geometry_guided_near_far(torch.from_numpy(o), torch.from_numpy(d), torch.from_numpy(V), 0.1)
    assert torch.allclose(n, n_r, atol=1e-6) and torch.allclose(f, f_r, atol=1e-6)
    assert torch.equal(torch.isinf(n), torch.isinf(n_r))


def test_smpl_match():
    model = synth_smpl.torch_model()
    pose, betas = torch.from_numpy(G["smpl_pose"]), torch.from_numpy(G["smpl_betas"])
    T, v = no.smpl_lbs(model, pose, betas, concat_joints=True)
    rows = torch.from_numpy(util.pick(T.shape[0], ROWS, 100))
    assert torch.allclose(T[rows], torch.from_numpy(G["smpl_T"]), atol=1e-6)
    assert torch.allclose(v[rows], torch.from_numpy(G["smpl_v"]), atol=1e-6)
    verts, joints = no.smpl_forward_verts(model, pose, betas)
    vrows = torch.from_numpy(util.pick(verts.shape[1], ROWS, 101))
    assert torch.allclose(verts[0, vrows], torch.from_numpy(G["smpl_verts"]), atol=1e-5)
    assert torch.allclose(joints[0], torch.from_numpy(G["smpl_joints"]), atol=1e-5)


def test_warp_match():
    body = synth_smpl.random_body(seed=2)
    faces6 = np.concatenate([body["faces"], body["faces"]], 1)       # 6-column faces like read_obj
    c, d, cl = no.warp_samples_to_canonical(G["warp_pts"], body["verts"], faces6, body["Ts"])
    assert np.allclose(c, G["warp_can"], atol=1e-12) and np.allclose(d, G["warp_dirs"], atol=1e-9)
    assert np.allclose(cl, G["warp_closest"])


def test_render_vanilla_match():
    coarse, fine = scenes.seed_nets(nb.build_nerf, nb.default_opt(use_cuda=False), 1)
    assert np.allclose([scenes.net_checksum(coarse), scenes.net_checksum(fine)], G["rv_sum"], rtol=1e-9, atol=0)
    H, W = 6, 9
    rgb, dep = no.render_vanilla(no.net_params_from_joiner(coarse), no.net_params_from_joiner(fine),
                                 G["rv_K"], G["rv_c2w"], H, W, 0.0, 3.14,
                                 rays_per_batch=32, samples_per_ray=16, importance_samples_per_ray=8)
    assert np.allclose(rgb.reshape(H, W, 3), G["rv_rgb"], atol=2e-6)
    assert np.allclose(dep.reshape(H, W), G["rv_depth"], atol=2e-6)


def test_render_human_and_hybrid_match():
    torch.manual_seed(1)
    net = nb.HumanNeRF(nb.default_opt(use_cuda=False, num_offset_nets=1))
    scenes.boost_density(net.coarse_human_net)
    sums = [scenes.net_checksum(j) for j in (net.coarse_bkg_net, net.fine_bkg_net, net.coarse_human_net)]
    assert np.allclose(sums, G["hum_sum"], rtol=1e-9, atol=0)
    body = synth_smpl.random_body(seed=1, center=(0.1, 0.0, 0.3))
    H, W = 10, 8
    Kc, c2wc = G["hum_K"], G["hum_c2w"]
    faces = body["faces"]
    hp = no.net_params_from_joiner(net.coarse_human_net)
    cb, fb = no.net_params_from_joiner(net.coarse_bkg_net), no.net_params_from_joiner(net.fine_bkg_net)
    geo = body["geo_threshold"]
    for can in (True, False):
        r_r, d_r, a_r = (G[f"hum_smpl{int(can)}_{k}"] for k in ("rgb", "depth", "acc"))
        r, d, a = no.render_smpl_nerf(hp, Kc, c2wc, H, W, body["verts"], faces, body["Ts"], rays_per_batch=32,
                                      samples_per_ray=12, render_can=can, geo_threshold=geo, interval_comp=0.7)
        assert 0 < (a_r > 0).sum() < a_r.size          # the test must see hits and misses
        assert np.allclose(r.reshape(H, W, 3), r_r, atol=2e-6) and np.allclose(d.reshape(H, W), d_r, atol=2e-6)
        assert np.allclose(a.reshape(H, W), a_r, atol=2e-6)
    r, d, a = no.render_hybrid_nerf(cb, fb, hp, Kc, c2wc, H, W, 0.0, 3.14, body["verts"], faces, body["Ts"],
                                    rays_per_batch=32, samples_per_ray=12, importance_samples_per_ray=8,
                                    geo_threshold=geo)
    assert np.allclose(r.reshape(H, W, 3), G["hum_hyb_rgb"], atol=2e-6) and np.allclose(d.reshape(H, W), G["hum_hyb_depth"], atol=2e-6)
    body2 = synth_smpl.random_body(seed=4, center=(-0.2, 0.0, 0.5))
    r, d = no.render_hybrid_nerf_multi_persons(cb, fb, [hp, hp], Kc, c2wc, H, W, 0.0, 3.14,
                                               [body["verts"], body2["verts"]], [faces, faces],
                                               [body["Ts"], body2["Ts"]], rays_per_batch=32, samples_per_ray=12,
                                               importance_samples_per_ray=8, geo_threshold=geo)
    assert np.allclose(r.reshape(H, W, 3), G["hum_multi_rgb"], atol=2e-6) and np.allclose(d.reshape(H, W), G["hum_multi_depth"], atol=2e-6)


def test_mirror_human_nerf_state_dict_matches_the_reference():
    """The host mirror (neuman_b200.models) creates the reference's parameters -- names, shapes, default-init values in the
    same order -- including the offset nets, so `hybrid_model_state_dict` checkpoints load unchanged (SURVEY.md §8b)."""
    torch.manual_seed(11)
    m = nb.HumanNeRF(nb.default_opt(use_cuda=False, num_offset_nets=2))
    sm = m.state_dict()
    util.assert_state_dict_is_the_references(sm, G, "hsd")
    assert any(k.startswith("offset_nets.1.nerf.output_linear") for k in sm)
    shapes = [tuple(int(n) for n in s.split("x")) if s else () for s in G["hsd_shapes"]]
    m.load_state_dict({str(k): torch.zeros(s) for k, s in zip(G["hsd_keys"], shapes)}, strict=True)


def test_vertex_forward_and_its_gradients_match():
    """oracle.vertex_forward (what the SMPL training kernels and their adjoint are checked against) vs the reference's
    HumanNeRF.vertex_forward (models/human_nerf.py:92-122): values and the gradients loss.backward() sends to
    poses / betas / alignments (the reference's per-frame SMPL parameters of tools/make_golden_reference.py: human_net)."""
    rng = np.random.RandomState(6)
    pose, betas = rng.normal(0, 0.3, (1, 72)).astype(np.float32), rng.normal(0, 1, (1, 10)).astype(np.float32)
    align = np.eye(4, dtype=np.float32)
    align[:3, :3] = np.array([[np.cos(0.2), 0, np.sin(0.2)], [0, 1, 0], [-np.sin(0.2), 0, np.cos(0.2)]])
    align = align.T.copy()
    align[3, :3] = (0.3, -0.1, 2.0)
    model = synth_smpl.torch_model(0)
    po, bo = torch.from_numpy(pose).requires_grad_(True), torch.from_numpy(betas).requires_grad_(True)
    ao = torch.from_numpy(align).requires_grad_(True)
    w_o, T_o = no.vertex_forward(model, po, bo, ao, 0.4)
    assert tuple(T_o.shape) == tuple(G["vf_T_shape"]) and tuple(w_o.shape) == tuple(G["vf_w_shape"])
    T4, w3 = T_o.reshape(-1, 4, 4), w_o.reshape(-1, 3)
    rows, wrows = util.pick(T4.shape[0], ROWS, 102), util.pick(w3.shape[0], ROWS, 103)
    assert (T4[rows] - torch.from_numpy(G["vf_T"])).abs().max() < 1e-6
    assert (w3[wrows] - torch.from_numpy(G["vf_w"])).abs().max() < 1e-6
    rng = np.random.RandomState(0)
    g1 = torch.from_numpy(rng.normal(0, 1, tuple(T_o.shape)).astype(np.float32))
    g2 = torch.from_numpy(rng.normal(0, 1, tuple(w_o.shape)).astype(np.float32))
    ((T_o * g1).sum() + (w_o * g2).sum()).backward()
    for name, b in (("poses", po.grad), ("betas", bo.grad), ("alignments", ao.grad)):
        a = torch.from_numpy(G[f"vf_grad_{name}"]).reshape(b.shape)
        assert (a - b).abs().max() < 1e-5 * (1 + b.abs().max()), name


def test_differentiable_warp_matches_and_its_vertex_gradient_depends_on_the_tie_rule():
    """oracle.warp_diff_Tinv vs the reference's warp_samples_to_canonical_diff (utils/ray_utils.py:69-93) on the same query
    answers.  Then the property that makes libigl's tie rule matter for TRAINING (DESIGN.md §2): where the closest point
    lies on an edge, both adjacent faces give the same inverse transform, but a different gradient with respect to the
    vertices."""
    from oracle import mesh_oracle as mo
    body = synth_smpl.random_body(seed=3)
    V = torch.from_numpy(body["verts"]).float().requires_grad_(True)
    F = np.asarray(body["faces"])[:, :3]
    T = torch.from_numpy(body["Ts"][:6890]).float().requires_grad_(True)
    rng = np.random.RandomState(0)
    P = (body["verts"][rng.randint(0, 6890, 400)] + rng.normal(0, 0.03, (400, 3))).astype(np.float32)
    S, I, C = mo.signed_distance(P, body["verts"], F)
    assert np.array_equal(G["wd_face"], I)
    Ti = no.warp_diff_Tinv(C, I, V, F, T)
    assert (Ti - torch.from_numpy(G["wd_Tinv"])).abs().max() == 0
    # the other face of every edge-region sample
    L = mo.barycentric_coordinates_tri(C, *(body["verts"][F[I, k]].astype(np.float64) for k in range(3)))
    edges = {}
    for f, tri in enumerate(F):
        for e in ((tri[0], tri[1]), (tri[1], tri[2]), (tri[2], tri[0])):
            edges.setdefault((min(e), max(e)), []).append(f)
    I2, flipped = I.copy(), 0
    for r in range(len(I)):
        z = np.flatnonzero(np.abs(L[r]) < 1e-9)
        if len(z) == 1:
            tri = F[I[r]]
            e = (tri[(z[0] + 1) % 3], tri[(z[0] + 2) % 3])
            other = [f for f in edges[(min(e), max(e))] if f != I[r]]
            if other:
                I2[r], flipped = other[0], flipped + 1
    assert flipped > 40                                                    # edge regions are common, not a corner case
    Ti2 = no.warp_diff_Tinv(C, I2, V, F, T)
    assert (Ti2 - Ti).abs().max() < 1e-5 * Ti.abs().max()                 # same transform ...
    w = torch.from_numpy(rng.normal(0, 1, tuple(Ti.shape)).astype(np.float32))
    gV1 = torch.autograd.grad((Ti * w).sum(), V, retain_graph=True)[0]
    gV2 = torch.autograd.grad((Ti2 * w).sum(), V)[0]
    assert (gV1 - gV2).abs().max() > 0.05 * gV1.abs().max()               # ... different gradient to the vertices
