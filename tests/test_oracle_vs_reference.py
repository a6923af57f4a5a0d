"""Pin the oracle and the package's host-side surface against the real reference.

The reference's side of every case is stored in tests/golden/reference_pins.npz (tools/make_golden_reference_pins.py, run
against the unmodified reference): values compared with a tolerance as values (a large output as a fixed seeded sample),
values compared bit for bit as digests.  An output too large to store whole is checked twice: a seeded sample of its elements
at the test's per-element tolerance, and its stored Gaussian projections (_util.projections) against an L2 bound over all of its
elements.  Inputs are regenerated here from the seeds the reference was run with; the case lists are the generator's."""
import json
import os

import numpy as np
import pytest
import torch

import ref_capture
import ref_shim
from make_golden_reference_pins import CAM, FANCY_CASES, GEN_CASES, PDF_CASES, PF_CASES, PF_TESTS, WP_CASES
from oracle import cips3d_oracle as O
from _util import GOLDEN, JL_SLACK, digest, digest_all, digests, projected_l2, sample

PINS = np.load(os.path.join(GOLDEN, "reference_pins.npz"))


def pin(key):
    return torch.from_numpy(PINS[key])


def pin_json(key):
    return json.loads(str(PINS[key]))


def constructor_init_generator(seed, frozen=False):
    """This package's generator as its constructor initialises it under `seed`: the reference's init, bit for bit
    (test_boundary_cpu.py::test_constructor_init_matches_reference_bitwise)."""
    from _util import build_generator
    torch.manual_seed(seed)
    return build_generator("cpu", frozen=frozen)


@pytest.mark.parametrize("noise,kw", GEN_CASES)
def test_generator_bitwise_vs_reference(noise, kw):
    i = GEN_CASES.index((noise, kw))
    sd = {k: v.clone() for k, v in constructor_init_generator(1234).state_dict().items()}     # reference-constructor init
    assert digests(sd) == pin_json("G_init_1234")
    torch.manual_seed(11)
    zs = {"z_nerf": torch.randn(2, 256), "z_inr": torch.randn(2, 512)}                # GeneratorNerfINR.get_zs(2)
    assert {k: digest(v) for k, v in zs.items()} == pin_json(f"gen{i}_zs")
    args = dict(ref_shim.G_KWARGS)
    args.update(kw)
    log = []
    for kind, shape, dg in pin_json(f"gen{i}_draw_spec"):       # the reference forward's draws, in its order
        t = (torch.rand if kind == "rand" else torch.randn)(shape)
        assert digest(t) == dg
        log.append((kind, t))
    draws = ref_capture.draws_from_log(log, hierarchical=args["hierarchical_sample"])
    draws.setdefault("noise_c", None)
    draws.setdefault("pdf_u", None)
    with torch.no_grad():
        img2, py2 = O.generator_forward(sd, zs, draws, img_size=12, nerf_noise=noise,
                                        return_aux_img=True, **args)
    img = pin(f"gen{i}_img")
    assert img2.shape == img.shape
    assert (img - img2).abs().max().item() < 1e-6
    assert torch.equal(pin(f"gen{i}_pitch_yaw"), py2)


def test_draw_order_matches_reference():
    """oracle.draw_randoms replays the reference's RNG call sequence (SURVEY.md §7 hard part 4)."""
    torch.manual_seed(5)
    d = O.draw_randoms(2, 8, 12)
    d_ref = pin_json("draw_order")
    assert list(d) == list(d_ref)
    for k in d:
        assert digest(d[k]) == d_ref[k], k


def test_discriminator_vs_reference():
    import cips3d_b200
    torch.manual_seed(3)
    D = cips3d_b200.Discriminator_MultiScale_Aux(**ref_shim.D_CFG)
    sd = {k: v.clone() for k, v in D.state_dict().items()}
    del D
    assert digest_all(sd) == str(PINS["D_init_3"])                   # the reference's constructor init under this seed
    x = torch.randn(4, 3, 32, 32)
    assert digest(x) == str(PINS["disc_x"])
    with torch.no_grad():
        b = O.discriminator_forward(sd, x, use_aux_disc=True, alpha=0.6)
    a = pin("disc_out")
    assert a.shape == b.shape and (a - b).abs().max().item() < 1e-6


def test_optimiser_tail_vs_torch_and_reference_ema():
    """oracle.clip_adam_ema_step == clip_grad_norm_ + torch.optim.Adam.step + the reference's EMA.update, bit for bit."""
    torch.manual_seed(0)
    net = torch.nn.Sequential(torch.nn.Linear(19, 33), torch.nn.Tanh(), torch.nn.Linear(33, 7))
    opt = torch.optim.Adam(params=[{'params': net.parameters(), 'initial_lr': 2e-3}], lr=2e-3, betas=(0.0, 0.999),
                           weight_decay=0, foreach=False)
    P = [p.detach().clone() for p in net.parameters()]
    M = [torch.zeros_like(p) for p in P]
    V = [torch.zeros_like(p) for p in P]
    E = [p.clone() for p in P]
    ema_ref = pin_json("ema_steps")          # the reference EMA's parameters after each step (decay 0.999, start_itr 2)
    for it in range(5):
        x = torch.randn(8, 19)
        opt.zero_grad()
        net(x).square().mean().mul(1e3).backward()
        grads = [p.grad.detach().clone() for p in net.parameters()]
        n_ref = torch.nn.utils.clip_grad_norm_(net.parameters(), 10.0)
        opt.step()
        n = O.clip_adam_ema_step(P, grads, M, V, E, step=it + 1, lr=2e-3, betas=(0.0, 0.999), max_norm=10.0,
                                 ema_decay=0.999 if it >= 2 else None)
        assert torch.equal(n, n_ref)
        for a, b in zip(P, net.parameters()):
            assert torch.equal(a, b.detach())
        assert [digest(a) for a in E] == ema_ref[it]


@pytest.mark.parametrize("cls_name", ["SPATIALSIRENBASELINE", "TALLSIREN"])
def test_pigan_surface_constructor_state_dict_and_field_vs_reference(cls_name):
    """cips3d_b200.pigan vs the real piGAN_lib classes: same state_dict keys / shapes / order, same constructor
    initialisation bit for bit under one seed (same RNG call order), same mapping network and field outputs."""
    import cips3d_b200
    torch.manual_seed(123)
    mine = cips3d_b200.pigan.ImplicitGenerator3d(getattr(cips3d_b200.pigan, cls_name), z_dim=256)
    sm = mine.state_dict()
    sr = pin_json(f"pigan_{cls_name}_init")
    assert list(sr.keys()) == list(sm.keys())
    assert {k: tuple(v.shape) for k, v in sm.items()} == {k: tuple(v) for k, v in O.pigan_template().items()}
    assert digests(sm) == sr
    bits = pin_json(f"pigan_{cls_name}_bits")
    z = torch.randn(3, 256)
    pts, dirs = torch.randn(3, 50, 3) * 0.1, torch.nn.functional.normalize(torch.randn(3, 50, 3), dim=-1)
    assert (digest(z), digest(pts), digest(dirs)) == (bits["z"], bits["pts"], bits["dirs"])
    o_r = pin(f"pigan_{cls_name}_field")
    with torch.no_grad():
        fr_m, ph_m = mine.siren.mapping_network(z)
        assert digest(fr_m) == bits["fr"] and digest(ph_m) == bits["ph"]
        o_m = mine.siren.forward_with_frequencies_phase_shifts(pts, fr_m, ph_m, ray_directions=dirs)
        o_o = O.pigan_siren(sm, pts, dirs, fr_m, ph_m, gridwarp=cls_name == "SPATIALSIRENBASELINE")
    assert o_m.shape == o_r.shape
    assert (o_r - o_m).abs().max().item() < 1e-6 and (o_r - o_o).abs().max().item() < 1e-6
    # generate_avg_frequencies draws the same 10000 latents
    mine.device = mine.siren.device = "cpu"
    torch.manual_seed(7)
    a_m = mine.generate_avg_frequencies()
    assert digest(a_m[0]) == bits["avg_fr"] and digest(a_m[1]) == bits["avg_ph"]


@pytest.mark.parametrize("clamp,last_back,white_back,noise_std,T,Cn", FANCY_CASES)
def test_native_fancy_integration_vs_the_real_function(clamp, last_back, white_back, noise_std, T, Cn):
    """ops.fancy_integration (csrc/integrate_ops.cu on the CPU emulation) against the UNMODIFIED exp/pigan/pigan_utils.py
    function: same signature, same RNG draw (identical seed -> identical noise), same three outputs, same gradient."""
    from _emu import emulated
    i = FANCY_CASES.index((clamp, last_back, white_back, noise_std, T, Cn))
    g = torch.Generator().manual_seed(T * 100 + Cn)
    rs = torch.randn(2, 29, T, Cn + 1, generator=g)
    rs[..., Cn] = (rs[..., Cn] + 0.3) * 8
    z = torch.sort(0.88 + 0.24 * torch.rand(2, 29, T, 1, generator=g), -2).values
    d_rgb = torch.randn(2, 29, Cn, generator=g)
    rgb0, depth0, w0 = pin(f"fancy{i}_rgb"), pin(f"fancy{i}_depth"), pin(f"fancy{i}_weights")
    with emulated(async_mode=0) as pkg:
        r1 = rs.clone().requires_grad_()
        torch.manual_seed(77)
        rgb1, depth1, w1 = pkg.ops.fancy_integration(r1, z, device="cpu", dim_rgb=Cn, noise_std=noise_std, last_back=last_back,
                                                     white_back=white_back, clamp_mode=clamp)
        (g1,) = torch.autograd.grad(rgb1, r1, d_rgb)
        with pytest.raises(AssertionError):
            pkg.ops.fancy_integration(r1, z, device="cpu", dim_rgb=Cn, clamp_mode=None)       # pigan_utils.py:252-253
    assert str(PINS["fancy_clamp_none_raises"]) == "AssertionError"
    assert rgb1.shape == rgb0.shape and depth1.shape == depth0.shape and w1.shape == w0.shape
    assert (w1 - w0).abs().max().item() < 1e-6
    assert (rgb1.detach() - rgb0).abs().max().item() < 1e-5
    assert (depth1 - depth0).abs().max().item() < 1e-5
    g0_sample, g0_max = pin(f"fancy{i}_grad_sample"), pin(f"fancy{i}_grad_absmax").item()
    tol = 1e-4 * g0_max + 1e-6
    assert (sample(g1, g0_sample.numel()) - g0_sample).abs().max().item() < tol
    assert projected_l2(g1, pin(f"fancy{i}_grad_proj")) < JL_SLACK * tol * g1.numel() ** 0.5     # the same bound, in L2
    with emulated(async_mode=0) as pkg:
        torch.manual_seed(77)
        pkg.ops.fancy_integration(rs, z, device="cpu", dim_rgb=Cn, noise_std=noise_std, clamp_mode=clamp)
        b = torch.rand(4)
    assert torch.equal(pin(f"fancy{i}_rand_after"), b)     # both consumed the same amount of the torch RNG stream


@pytest.mark.parametrize("n,k,det", PDF_CASES)
def test_native_sample_pdf_vs_the_real_function(n, k, det):
    """ops.sample_pdf (emulation): the reference function's signature, its torch.rand / linspace draw and its output."""
    from _emu import emulated
    i = PDF_CASES.index((n, k, det))
    g = torch.Generator().manual_seed(n * 10 + k)
    w = torch.rand(41, n, generator=g) + 1e-5
    edges = torch.sort(0.88 + 0.24 * torch.rand(41, n + 2, generator=g), -1).values
    bins = 0.5 * (edges[:, :-1] + edges[:, 1:])
    want = pin(f"pdf{i}_samples")
    with emulated(async_mode=0) as pkg:
        torch.manual_seed(3)
        got = pkg.ops.sample_pdf(bins, w, k, det=det)
        b = torch.rand(2)
    assert got.shape == want.shape and (got - want).abs().max().item() < 2e-6
    assert torch.equal(pin(f"pdf{i}_rand_after"), b)      # same RNG consumption (none in det mode)


@pytest.mark.parametrize("frozen,backend,case", PF_TESTS)
def test_points_forward_vs_reference(monkeypatch, frozen, backend, case):
    """GeneratorNerfINR[_freeze_NeRF].points_forward (generator.py:1659-1762 / 1972-2078; reference signature) against the
    UNMODIFIED method on identical weights, points and seed -- same three RNG draws, same images, same parameter gradients;
    with the torch ops and with the native integration / resampling / merge ops (CPU emulation).  The reference's
    gradients are stored as N_PROJ Gaussian projections of each parameter's whole gradient, with its max |g| and L2 norm
    (and, for the torch backend's per-element bound, a seeded sample of its elements)."""
    import cips3d_b200
    from _emu import emulated
    i = PF_CASES.index((frozen, case))
    hier, noise, kw = case
    monkeypatch.setattr(cips3d_b200.generator, "_require_cuda", lambda *a, **k: None)
    G = constructor_init_generator(21, frozen=frozen).train()
    assert digest_all(G.state_dict()) == str(PINS[f"pf{i}_init"])     # the reference's weights
    G.train_integrate = backend
    b, n, s = 2, 37, 12
    g = torch.Generator().manual_seed(5)
    origins = torch.randn(b, n, 3, generator=g) * 0.05 + torch.tensor([0., 0., 1.])
    dirs = torch.nn.functional.normalize(torch.randn(b, n, 3, generator=g) * 0.05 + torch.tensor([0., 0., -1.]), dim=-1)
    z_vals = torch.sort(0.88 + 0.24 * torch.rand(b, n, s, 1, generator=g), -2).values
    points = origins[:, :, None] + dirs[:, :, None] * z_vals
    dirs_exp = dirs[:, :, None].expand(-1, -1, s, -1).contiguous()
    idx = torch.randperm(n, generator=g)[:29]
    zs = {"z_nerf": torch.randn(b, 256, generator=g), "z_inr": torch.randn(b, 512, generator=g)}
    args = dict(transformed_points=points, transformed_ray_directions_expanded=dirs_exp, num_steps=s, hierarchical_sample=hier,
                z_vals=z_vals, nerf_noise=noise, transformed_ray_origins=origins, transformed_ray_directions=dirs,
                return_aux_img=True, idx_grad=idx, **kw)
    G.zero_grad()
    with emulated(async_mode=0):
        style = G.mapping_network(**zs)
        torch.manual_seed(99)
        inr, aux = G.points_forward(style_dict=style, **args)
        after = torch.rand(3)
        (inr.square().mean() + (aux.square().mean() if aux.requires_grad else 0)).backward()
    new = {k: p.grad.clone() for k, p in G.named_parameters() if p.grad is not None}
    inr_ref, aux_ref = pin(f"pf{i}_inr"), pin(f"pf{i}_aux")
    assert torch.equal(after, pin(f"pf{i}_rand_after"))                       # same RNG consumption
    assert inr.shape == inr_ref.shape and aux.shape == aux_ref.shape
    assert (inr.detach() - inr_ref).abs().max().item() < 2e-5 and (aux.detach() - aux_ref).abs().max().item() < 2e-5
    keys = pin_json(f"pf{i}_grad_keys")
    assert new.keys() == set(keys)
    assert any(k.startswith("siren.") for k in keys) == (not frozen)
    proj = pin(f"pf{i}_grad_proj").view(len(keys), -1)
    absmax, norm = pin(f"pf{i}_grad_absmax").tolist(), pin(f"pf{i}_grad_norm").tolist()
    samples = pin(f"pf{i}_grad_sample").split([min(16, new[k].numel()) for k in keys]) if backend == "torch" else None
    for j, k in enumerate(keys):
        if backend == "torch":                  # identical arithmetic to the reference's
            assert (sample(new[k], 16, seed=j) - samples[j]).abs().max().item() < 1e-3 * absmax[j] + 1e-7, k
        # ~1e-6 differences of pixels_fea flip LeakyReLU gates of |z| ~ 0 units in the CIPS MLP (29 pixels): compare in L2,
        # over the whole gradient through its projections
        assert projected_l2(new[k], proj[j], seed=j) < JL_SLACK * (1e-2 * norm[j] + 1e-7), k
        assert abs(new[k].norm().item() - norm[j]) < 1e-2 * norm[j] + 1e-7, k


@pytest.mark.parametrize("lock,cam", WP_CASES)
def test_get_world_points_and_direction_vs_reference(lock, cam):
    """cips3d_b200.comm_utils.get_world_points_and_direction against exp/comm/comm_utils.py:682-763: same signature, the same
    seven outputs, the same RNG order (jitter, then the camera draws), also with a given camera and lock_view_dependence."""
    import cips3d_b200
    i = WP_CASES.index((lock, cam))
    kw = dict(batch_size=2, num_steps=12, img_size=9, fov=12, ray_start=0.88, ray_end=1.12, h_stddev=0.3, v_stddev=0.155,
              h_mean=1.5707963, v_mean=1.5707963, sample_dist="gaussian", lock_view_dependence=lock, device="cpu")
    if cam:
        kw.update(CAM)
    torch.manual_seed(8)
    got = cips3d_b200.comm_utils.get_world_points_and_direction(**kw)
    b = torch.rand(3)
    shapes = pin_json(f"wp{i}_shapes")
    assert torch.equal(pin(f"wp{i}_rand_after"), b) and len(got) == len(shapes) == 7
    for j, (g_, shape) in enumerate(zip(got, shapes)):
        assert list(g_.shape) == shape, j
        assert (sample(g_, 256, seed=j) - pin(f"wp{i}_out{j}")).abs().max().item() < 2e-6, j
        assert projected_l2(g_, pin(f"wp{i}_proj{j}"), seed=j) < JL_SLACK * 2e-6 * g_.numel() ** 0.5, j    # the same bound, in L2
    probe = torch.arange(got[2].numel(), dtype=torch.float32).reshape(got[2].shape)
    assert digest(cips3d_b200.comm_utils.gather_points(probe, torch.tensor([3, 1]))) == str(PINS[f"wp{i}_gather"])


def test_host_helpers_of_the_inference_scripts_vs_reference():
    """comm_utils camera trajectories (bit for bit) and inr_layer_swapping (same parameters touched, same blend)."""
    import cips3d_b200
    from _util import build_generator
    cu = cips3d_b200.comm_utils
    for j, a in enumerate((cu.get_circle_camera_pos_and_lookup(r=1.1, alpha=0.4, num_samples=7, periods=2),
                           cu.get_circle_camera_pos_and_lookup(),
                           cu.get_yaw_camera_pos_and_lookup(r=1, num_samples=9))):
        assert len(a) == len([k for k in PINS.files if k.startswith(f"traj{j}_")])
        for m, x in enumerate(a):
            y = PINS[f"traj{j}_{m}"]
            assert x.dtype == y.dtype and np.array_equal(x, y)
    assert np.array_equal(np.array(cu.get_yaw_pitch_by_xyz(0.3, -0.2, 0.9), dtype=np.float64), PINS["yaw_pitch_by_xyz"])
    torch.manual_seed(2)
    A = build_generator("cpu").inr_net
    T = build_generator("cpu").inr_net                      # different random init
    cu.inr_layer_swapping(A, T, 0.3, ["64", "1024"], verbose=False)
    assert digests(A.state_dict()) == pin_json("inr_swap")


def test_camera_space_ray_functions_vs_reference():
    """comm_utils.get_initial_rays_trig / perturb_points: reference signatures, bit-identical outputs and RNG consumption."""
    import cips3d_b200
    cu = cips3d_b200.comm_utils
    for res in ((7, 7), (6, 9)):
        a = cu.get_initial_rays_trig(bs=2, num_steps=12, fov=12, resolution=res, ray_start=0.88, ray_end=1.12, device="cpu")
        assert [digest(x) for x in a] == pin_json(f"rays_{res[0]}x{res[1]}")
    torch.manual_seed(4)
    p1, z1 = cu.perturb_points(a[0], a[1], a[2], "cpu")
    r1 = torch.rand(2)
    assert [digest(p1), digest(z1), digest(r1)] == pin_json("perturb")


@pytest.mark.parametrize("cam", [False, True])
def test_transform_sampled_points_vs_reference(cam):
    import cips3d_b200
    cu = cips3d_b200.comm_utils
    i = int(cam)
    pts, z, d = cu.get_initial_rays_trig(bs=2, num_steps=12, fov=12, resolution=(5, 5), ray_start=0.88, ray_end=1.12, device="cpu")
    kw = dict(h_stddev=0.3, v_stddev=0.155, h_mean=1.5707963, v_mean=1.5707963, mode="gaussian", device="cpu")
    if cam:
        kw.update(CAM)
    torch.manual_seed(6)
    got = cu.transform_sampled_points(pts, z, d, **kw)
    r2 = torch.rand(2)
    assert torch.equal(pin(f"tsp{i}_rand_after"), r2)
    shapes = pin_json(f"tsp{i}_shapes")
    assert len(got) == len(shapes)
    for j, (g_, shape) in enumerate(zip(got, shapes)):
        assert list(g_.shape) == shape and (g_ - pin(f"tsp{i}_out{j}")).abs().max().item() < 1e-6, j


def test_pigan_lib_function_surface_vs_reference():
    """cips3d_b200.pigan.fancy_integration / sample_pdf against piGAN_lib/generators/volumetric_rendering.py (emulation)."""
    import cips3d_b200
    from _emu import emulated
    g = torch.Generator().manual_seed(12)
    rs = torch.randn(2, 21, 24, 4, generator=g)
    rs[..., 3] = (rs[..., 3] + 0.3) * 8
    z = torch.sort(0.88 + 0.24 * torch.rand(2, 21, 24, 1, generator=g), -2).values
    want = [pin(k) for k in sorted(k for k in PINS.files if k.startswith("vr_fancy_out"))]
    w = torch.rand(19, 10, generator=g) + 1e-5
    bins = torch.sort(0.88 + 0.24 * torch.rand(19, 11, generator=g), -1).values
    want_pdf = pin("vr_sample_pdf")
    with emulated(async_mode=0):
        torch.manual_seed(1)
        got = cips3d_b200.pigan.fancy_integration(rs, z, device="cpu", noise_std=0.4, last_back=True, white_back=True, clamp_mode="relu")
        got_pdf = cips3d_b200.pigan.sample_pdf(bins, w, 12, det=False)
        with pytest.raises(TypeError):
            cips3d_b200.pigan.fancy_integration(rs, z, device="cpu")
    assert str(PINS["vr_fancy_no_kwargs_raises"]) == "TypeError"
    assert len(got) == len(want)
    for a, b in zip(got, want):
        assert a.shape == b.shape and (a - b).abs().max().item() < 1e-5
    assert got_pdf.shape == want_pdf.shape and (got_pdf - want_pdf).abs().max().item() < 2e-6
