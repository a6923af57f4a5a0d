"""Host-side contract tests that need no GPU: state_dict contract, constructor-init parity with the
reference, C-ABI exports, fail-loud behaviour, RNG-order parity of the torch-side helpers."""
import ctypes
import json
import os
import re

import numpy as np
import pytest
import torch

import ref_shim
from oracle import cips3d_oracle as O
from _util import GOLDEN, JL_SLACK, digest, projected_l2, sample

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PINS = np.load(os.path.join(GOLDEN, "reference_pins.npz"))     # the reference's side of the parity tests


@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__ as g
    g.build()
    import cips3d_b200
    return cips3d_b200


def _contract():
    with open(os.path.join(GOLDEN, "state_dict_contract.json")) as f:
        return json.load(f)


def test_generator_state_dict_contract(pkg):
    G = pkg.GeneratorNerfINR(**O.G_CFG, device="cpu")
    c = _contract()["generator"]
    sd = G.state_dict()
    assert list(sd.keys()) == list(c.keys())
    assert all(list(sd[k].shape) == c[k] for k in sd)
    Gf = pkg.GeneratorNerfINR_freeze_NeRF(**O.G_CFG, device="cpu")
    assert list(Gf.state_dict().keys()) == list(c.keys())
    for attr in ("siren", "inr_net", "mapping_network_nerf", "mapping_network_inr", "aux_to_rbg", "filters",
                 "epoch", "step", "z_dim", "device"):
        assert hasattr(G, attr)


def test_discriminator_state_dict_contract(pkg):
    D = pkg.Discriminator_MultiScale_Aux(diffaug=False, max_size=1024, channel_multiplier=2,
                                         first_downsample=False, stddev_group=0)
    c = _contract()["discriminator"]
    sd = D.state_dict()
    assert list(sd.keys()) == list(c.keys())
    assert all(list(sd[k].shape) == c[k] for k in sd)
    assert sum(p.numel() for p in D.parameters()) == 37518914          # BASELINE.md section 2


def test_constructor_init_matches_reference_bitwise(pkg):
    """Both constructors initialise like the reference's under the same seed: digests of the reference's state_dicts
    (tests/golden/reference_pins.npz, tools/make_golden_reference_pins.py)."""
    torch.manual_seed(1234)
    mine = pkg.GeneratorNerfINR(**O.G_CFG, device="cpu").state_dict()
    ref = json.loads(str(PINS["G_init_1234"]))
    assert list(ref) == list(mine)
    for k in ref:
        assert digest(mine[k]) == ref[k], k
    torch.manual_seed(77)
    myd = pkg.Discriminator_MultiScale_Aux(**ref_shim.D_CFG).state_dict()
    refd = json.loads(str(PINS["D_init_77"]))
    assert list(refd) == list(myd)
    for k in refd:
        assert digest(myd[k]) == refd[k], k


def test_library_exports_every_declared_symbol(pkg):
    hdr = open(os.path.join(ROOT, "include", "cips3d_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    names = set(re.findall(r"\b(c3d_\w+)\s*\(", hdr))
    assert {"c3d_ray_siren_fwd", "c3d_cips_fwd", "c3d_bias_act", "c3d_upfirdn2d"} <= names
    lib = ctypes.CDLL(pkg._lib.LIB_PATH)
    for n in names:
        assert hasattr(lib, n), n
    assert set(pkg._lib.EXPORTS) == names
    assert lib.c3d_version() >= 100


def test_no_cpu_fallback(pkg):
    G = pkg.GeneratorNerfINR(**O.G_CFG, device="cpu")
    zs = {"z_nerf": torch.randn(1, 256), "z_inr": torch.randn(1, 512)}
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        G(zs, img_size=8, **O.G_KWARGS)
    with pytest.raises(Exception, match="CUDA"):
        pkg.ops.bias_act(torch.randn(2, 3, 4, 4), torch.randn(3))
    D = pkg.Discriminator_MultiScale_Aux(diffaug=False, max_size=64)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        D(torch.randn(2, 3, 32, 32))


def test_product_never_imports_oracle():
    pkg_dir = os.path.join(ROOT, "cips-3d_b200")
    for fn in os.listdir(pkg_dir):
        if fn.endswith(".py"):
            src = open(os.path.join(pkg_dir, fn)).read()
            assert "oracle" not in src.replace("the CPU oracle", ""), fn


def test_get_zs_and_draw_order(pkg):
    """get_zs + the forward's draw order consume torch's RNG like the reference (generator.py:1774-1794)."""
    G = pkg.GeneratorNerfINR(**O.G_CFG, device="cpu")
    torch.manual_seed(3)
    zs = G.get_zs(4)
    torch.manual_seed(3)
    assert torch.equal(zs["z_nerf"], torch.randn(4, 256)) and torch.equal(zs["z_inr"], torch.randn(4, 512))
    parts = G.get_zs(4, batch_split=2)
    assert len(parts) == 2 and parts[0]["z_nerf"].shape == (2, 256)


@pytest.mark.parametrize("mode", ["uniform", "normal", "gaussian", "truncated_gaussian", "spherical_uniform", "mean", "hybrid"])
def test_camera_sampling_matches_reference(pkg, mode):
    import random
    kw = dict(bs=5, r=1, horizontal_stddev=0.3, vertical_stddev=0.155, horizontal_mean=1.2, vertical_mean=1.7, mode=mode)
    a = [torch.from_numpy(PINS[k]) for k in sorted(k for k in PINS.files if re.fullmatch(f"cam_{mode}_[0-9]+", k))]
    torch.manual_seed(9); random.seed(4)
    b = pkg.comm_utils.sample_camera_positions("cpu", **kw)
    assert len(a) == len(b)
    for x, y in zip(a, b):
        assert x.shape == y.shape and torch.allclose(x, y, atol=1e-6), mode
    m_ref = torch.from_numpy(PINS[f"cam_{mode}_cam2world"])
    m = pkg.comm_utils.create_cam2world_matrix(-b[0], b[0], device="cpu")
    assert torch.allclose(m_ref, m, atol=1e-6)


def test_diffaugment_matches_reference(pkg):
    """The reference's DiffAugment output on the same input and seeds.  Stored: a fixed sample of each output's elements,
    checked at allclose's per-element bound, and Gaussian projections of the whole output, checked against that bound in L2."""
    x = torch.randn(6, 3, 32, 32, generator=torch.Generator().manual_seed(31))
    for seed in range(5):
        torch.manual_seed(seed)
        b = pkg.DiffAugment(x, policy="color,translation,cutout")
        assert list(b.shape) == PINS[f"diffaug{seed}_shape"].tolist()
        assert torch.allclose(torch.from_numpy(PINS[f"diffaug{seed}_sample"]), sample(b, 1024, seed=seed), atol=1e-6), seed
        assert projected_l2(b, torch.from_numpy(PINS[f"diffaug{seed}_proj"]), seed=seed) < JL_SLACK * float(PINS[f"diffaug{seed}_tol_l2"]), seed


def test_scatter_points_roundtrip(pkg):
    idx = torch.randperm(20)
    pts = torch.randn(2, 20, 3)
    out = pkg.comm_utils.scatter_points(idx[:7], pts[:, idx[:7]], idx[7:], pts[:, idx[7:]], 20)
    assert torch.equal(out, pts)
