"""Shared helpers for the parity tests (golden loading, oracle replay, error metrics)."""
import ast
import json
import os

import numpy as np
import torch

from oracle import cips3d_oracle as O

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
GEN_CASES = ("r16_synth", "r16_trained_noise", "r8_softplus_backs", "r8_nohier_s24", "r8_hier_s24")


def load_gen_case(name, dtype=torch.float32):
    g = np.load(os.path.join(GOLDEN, f"gen_{name}.npz"))
    kw = ast.literal_eval(str(g["kwargs_json"]))
    sd = O.synthetic_state_dict(O.generator_template(), seed=int(g["seed"]),
                                sigma_bias=float(g["sigma_bias"]), dtype=dtype)
    zs = dict(z_nerf=torch.from_numpy(g["z_nerf"]).to(dtype), z_inr=torch.from_numpy(g["z_inr"]).to(dtype))
    draws = {k[5:]: torch.from_numpy(g[k]).to(dtype) for k in g.files if k.startswith("draw_")}
    if "noise_c" not in draws:      # non-hierarchical: only 3 draws exist
        draws["noise_c"] = None
        draws["pdf_u"] = None
    meta = dict(B=int(g["B"]), img_size=int(g["img_size"]), nerf_noise=float(g["nerf_noise"]))
    ref = {k: torch.from_numpy(g[k]) for k in ("img", "pitch_yaw", "pixels_fea", "depth", "all_z", "coarse")}
    return sd, zs, draws, kw, meta, ref


def oracle_replay(name, dtype=torch.float32):
    sd, zs, draws, kw, meta, ref = load_gen_case(name, dtype)
    with torch.no_grad():
        img, py, r = O.generator_forward(sd, zs, draws, img_size=meta["img_size"],
                                         nerf_noise=meta["nerf_noise"], return_aux_img=True,
                                         return_all=True, **kw)
    return img, py, r, ref


def digest(t):
    """Bit-exact fingerprint of a tensor / array (dtype, shape and bytes): torch.equal against a stored value."""
    import hashlib
    a = t.detach().cpu().contiguous().numpy() if isinstance(t, torch.Tensor) else np.ascontiguousarray(t)
    return hashlib.sha256(f"{a.dtype.str}{a.shape}".encode() + a.tobytes()).hexdigest()[:16]


def digests(sd):
    return {k: digest(v) for k, v in sd.items()}


def digest_all(sd):
    """One digest of a whole state_dict: its keys in order and every tensor's digest."""
    return digest(np.array(json.dumps(list(digests(sd).items()))))


def sample(t, k=2048, seed=0):
    """A fixed, seeded sample of k elements of t (all of them when t is smaller): the stored part of a large output."""
    flat = t.detach().reshape(-1)
    if flat.numel() <= k:
        return flat.clone()
    idx = torch.randperm(flat.numel(), generator=torch.Generator().manual_seed(seed))[:k].sort().values
    return flat[idx]


N_PROJ = 32
# ||P d|| / sqrt(N_PROJ) lies within [0.47, 1.64] x ||d|| for a fixed d, but with probability 1e-6 at either end
# (chi-square with N_PROJ degrees of freedom): the slack of an L2 bound checked through projections()
JL_SLACK = 1.64


def projections(t, seed=0, m=N_PROJ):
    """m seeded Gaussian projections <r_i, t> of the whole of t (accumulated in float64).  ||P a - P b|| / sqrt(m) estimates
    ||a - b|| (Johnson-Lindenstrauss), so the stored projections of a reference tensor too large to store check an L2 bound
    over all of its elements."""
    flat = t.detach().reshape(-1).double()
    g = torch.Generator().manual_seed(seed)
    return torch.stack([torch.randn(flat.numel(), generator=g).double() @ flat for _ in range(m)])


def projected_l2(t, proj_ref, seed=0):
    """the estimate of ||t - ref|| from ref's stored projections (same seed)"""
    return ((projections(t, seed, proj_ref.numel()) - proj_ref.double()).norm() / proj_ref.numel() ** 0.5).item()


def rel_err(a, b):
    """max |a-b| / max|b|  and  L2-relative."""
    a, b = a.double(), b.double()
    return ((a - b).abs().max() / b.abs().max().clamp_min(1e-30)).item(), \
           ((a - b).norm() / b.norm().clamp_min(1e-30)).item()


# ------------------------------------------------------------------ GPU-side helpers
import contextlib


def draws_sequence(draws, hierarchical=True):
    """The draw tensors in the order GeneratorNerfINR.forward consumes them."""
    seq = [draws["jitter_u"][..., None], draws["yaw_n"], draws["pitch_n"]]
    if hierarchical:
        seq += [draws["noise_c"][..., None], draws["pdf_u"]]
    seq.append(draws["noise_f"][..., None])
    return seq


@contextlib.contextmanager
def replay_draws(seq, device):
    """Make torch.rand / torch.randn return the given tensors in order (so a module forward
    consumes exactly the draws the reference consumed)."""
    it = iter(seq)
    o_rand, o_randn = torch.rand, torch.randn

    def nxt(*a, **k):
        t = next(it)
        shape = a[0] if len(a) == 1 and isinstance(a[0], (tuple, list, torch.Size)) else a
        assert tuple(t.shape) == tuple(shape), (tuple(t.shape), tuple(shape))
        return t.to(device=device, dtype=torch.float32)

    torch.rand = torch.randn = nxt
    try:
        yield
    finally:
        torch.rand, torch.randn = o_rand, o_randn


def close_frac(a, b, tol):
    """fraction of rows (last dim reduced by max) whose abs error is within tol * max|b|"""
    a, b = a.double().cpu(), b.double().cpu()
    scale = b.abs().max().clamp_min(1e-30)
    err = (a - b).abs().reshape(-1, a.shape[-1]).amax(-1) / scale
    return (err <= tol).double().mean().item(), err.max().item()


def build_generator(device, sd=None, frozen=False):
    import cips3d_b200
    cls = cips3d_b200.GeneratorNerfINR_freeze_NeRF if frozen else cips3d_b200.GeneratorNerfINR
    cfg = {k: (dict(v) if isinstance(v, dict) else v) for k, v in O.G_CFG.items()}
    G = cls(**cfg, device=device).to(device).eval()
    if sd is not None:
        G.load_state_dict(sd)
    return G


# ------------------------------------------------------------------ pi-GAN surface goldens (tools/make_golden_pigan.py)
PIGAN_CASES = ("spatial_r8", "spatial_r8_noise_backs", "tall_r6_lockview", "spatial_r6_nohier_s24", "spatial_r6_staged_psi07")


def load_pigan_case(name, dtype=torch.float32):
    g = np.load(os.path.join(GOLDEN, f"pigan_{name}.npz"))
    kw = ast.literal_eval(str(g["kwargs_json"]))
    sd = O.synthetic_state_dict(O.pigan_template(), seed=int(g["seed"]), sigma_bias=float(g["sigma_bias"]), dtype=dtype)
    z = torch.from_numpy(g["z"]).to(dtype)
    draws = {k[5:]: torch.from_numpy(g[k]).to(dtype) for k in g.files if k.startswith("draw_")}
    draws.setdefault("noise_c", None)
    draws.setdefault("pdf_u", None)
    meta = dict(B=int(g["B"]), img_size=int(g["img_size"]), nerf_noise=float(g["nerf_noise"]), siren_cls=str(g["siren_cls"]),
                staged_psi=float(g["staged_psi"]))
    if meta["staged_psi"] >= 0:
        meta["avg"] = (torch.from_numpy(g["avg_frequencies"]).to(dtype), torch.from_numpy(g["avg_phase_shifts"]).to(dtype))
    ref = {k: torch.from_numpy(g[k]) for k in ("img", "pitch_yaw", "coarse", "all_z", "rgb", "depth")}
    return sd, z, draws, kw, meta, ref


def pigan_freq_phase(sd, z, meta):
    """mapping network output, truncated towards the stored averages for the staged_forward case (generators.py:121-126)"""
    fr, ph = O.pigan_mapping(sd, z)
    if meta["staged_psi"] >= 0:
        af, ap = meta["avg"]
        psi = meta["staged_psi"]
        fr, ph = af + psi * (fr - af), ap + psi * (ph - ap)
    return fr, ph
