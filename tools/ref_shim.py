"""Import shim that lets the UNMODIFIED reference (a checkout at $CIPS3D_REFERENCE) run on CPU.

TEST INFRASTRUCTURE ONLY.  Used by the tools/make_golden*.py scripts, which store what the
reference computes under tests/golden for the parity tests, and by bench.py's reference legs;
the tests take only its configuration constants.  Never imported by the product.

The reference depends on the author's un-vendored `tl2` package (README.md:62, no
version pin) plus `easydict` and `streamlit`; none of them contributes arithmetic to
the hot path (SURVEY.md §8c).  This module installs stand-ins into ``sys.modules``:

* ``tl2.launch.launch_utils.global_cfg``      – attribute bag, ``tl_debug`` False
* ``tl2.proj.fvcore.{MODEL_REGISTRY,build_model}``
* ``tl2.proj.pytorch.{torch_utils,init_func}``, ``...pytorch_hook.VerboseModel``
* ``tl2.tl2_utils.{dict2string,get_class_repr}``
* ``exp.comm.op``  – CPU stand-ins for the two JIT CUDA ops used by the
  discriminator (restating exp/comm/op/fused_bias_act_kernel.cu:19-50 and
  exp/comm/op/upfirdn2d_kernel.cu:52-139 with differentiable torch ops).
"""
import importlib
import math
import os
import sys
import types

REF_ROOT = os.environ.get("CIPS3D_REFERENCE", "/root/reference")


def reference_available() -> bool:
    return os.path.isdir(os.path.join(REF_ROOT, "exp", "cips3d", "models"))


class _Cfg(dict):
    def __getattr__(self, k):
        return self.get(k, False)

    def __setattr__(self, k, v):
        self[k] = v


class _Registry:
    def __init__(self):
        self._d = {}

    def register(self, name_prefix=None, **kw):
        def deco(cls):
            self._d[f"{name_prefix}.{cls.__name__}" if name_prefix else cls.__name__] = cls
            return cls
        return deco

    def get(self, name):
        return self._d[name]


def _mod(name, **attrs):
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    m.__path__ = []  # behave like a package so sub-imports resolve through sys.modules
    sys.modules[name] = m
    parent, _, child = name.rpartition(".")
    if parent and parent in sys.modules:
        setattr(sys.modules[parent], child, m)
    return m


def _install_tl2():
    import torch
    import torch.nn as nn

    registry = _Registry()

    def build_model(cfg, **kwargs):
        cfg = dict(cfg)
        for m in cfg.pop("register_modules", []):
            importlib.import_module(m)
        name = cfg.pop("name")
        cfg.pop("optim", None)
        cfg.update(kwargs)
        return registry.get(name)(**cfg)

    def kaiming_leaky_init(m):
        # tl2 source is absent; this mirrors exp/cips3d/models/multi_head_mapping.py:22-25
        # and piGAN_lib/siren/siren.py:43-46 (same author's in-tree twins).
        if m.__class__.__name__.find("Linear") != -1:
            torch.nn.init.kaiming_normal_(m.weight, a=0.2, mode="fan_in", nonlinearity="leaky_relu")

    class VerboseModel:
        @staticmethod
        def forward_verbose(*a, **k):
            return None

    class _AnyAttr(types.ModuleType):
        def __getattr__(self, k):
            if k.startswith("__"):
                raise AttributeError(k)
            return lambda *a, **kw: None

    _mod("tl2")
    _mod("tl2.launch")
    _mod("tl2.launch.launch_utils", global_cfg=_Cfg(tl_debug=False))
    _mod("tl2.proj")
    _mod("tl2.proj.fvcore", MODEL_REGISTRY=registry, build_model=build_model)
    _mod("tl2.proj.fvcore.checkpoint", Checkpointer=object)
    _mod("tl2.proj.pytorch")
    tu = _AnyAttr("tl2.proj.pytorch.torch_utils")
    tu.__path__ = []
    sys.modules[tu.__name__] = tu
    sys.modules["tl2.proj.pytorch"].torch_utils = tu
    _mod("tl2.proj.pytorch.init_func", kaiming_leaky_init=kaiming_leaky_init)
    _mod("tl2.proj.pytorch.pytorch_hook", VerboseModel=VerboseModel)
    _mod("tl2.proj.stylegan2_ada",
         persistence=types.SimpleNamespace(persistent_class=lambda c: c))
    for n in ("tl2.proj.cv2", "tl2.proj.pil", "tl2.proj.streamlit"):
        _mod(n)
    for n, a in (("tl2.proj.cv2", "cv2_utils"), ("tl2.proj.pil", "pil_utils"),
                 ("tl2.proj.streamlit", "st_utils")):
        sub = _AnyAttr(f"{n}.{a}")
        sys.modules[sub.__name__] = sub
        setattr(sys.modules[n], a, sub)
    _mod("tl2.tl2_utils",
         dict2string=lambda dict_obj=None, **k: str(dict_obj),
         get_class_repr=lambda self: f"{self.__class__.__name__}({getattr(self, 'repr_str', '')})")
    sys.modules["tl2"].tl2_utils = sys.modules["tl2.tl2_utils"]

    class EasyDict(dict):
        __getattr__ = dict.get
        __setattr__ = dict.__setitem__

    _mod("easydict", EasyDict=EasyDict)
    st = _AnyAttr("streamlit")
    sys.modules["streamlit"] = st


def _install_ops():
    """CPU stand-ins for exp/comm/op (fused_act.py:73-86, upfirdn2d.py:144-149)."""
    import torch
    import torch.nn as nn
    import torch.nn.functional as F

    def fused_leaky_relu(input, bias, negative_slope=0.2, scale=2 ** 0.5):
        # fused_bias_act_kernel.cu:26-46: x += b[(i/step_b)%size_b]; lrelu; *scale
        shape = [1, -1] + [1] * (input.dim() - 2)
        return F.leaky_relu(input + bias.view(*shape), negative_slope) * scale

    class FusedLeakyReLU(nn.Module):
        def __init__(self, channel, negative_slope=0.2, scale=2 ** 0.5):
            super().__init__()
            self.bias = nn.Parameter(torch.zeros(channel))
            self.negative_slope = negative_slope
            self.scale = scale

        def forward(self, input):
            return fused_leaky_relu(input, self.bias, self.negative_slope, self.scale)

    def upfirdn2d(input, kernel, up=1, down=1, pad=(0, 0)):
        # upfirdn2d_kernel.cu:52-139 for up=1: pad, correlate with the flipped
        # kernel, decimate.  (B,C,H,W) in, depthwise.
        assert up == 1
        b, c, h, w = input.shape
        x = F.pad(input, [pad[0], pad[1], pad[0], pad[1]])
        k = torch.flip(kernel, [0, 1])[None, None].repeat(c, 1, 1, 1).to(x.dtype)
        out = F.conv2d(x, k, groups=c)
        return out[:, :, ::down, ::down]

    pkg = "exp.comm.op"
    m = types.ModuleType(pkg)
    m.FusedLeakyReLU = FusedLeakyReLU
    m.fused_leaky_relu = fused_leaky_relu
    m.upfirdn2d = upfirdn2d
    m.__path__ = []
    sys.modules[pkg] = m


_INSTALLED = False


def install():
    """Make `import exp.cips3d.models.generator` (the real reference) work on CPU."""
    global _INSTALLED
    if _INSTALLED:
        return
    if not reference_available():
        raise RuntimeError(f"reference not found at {REF_ROOT}")
    _install_tl2()
    if REF_ROOT not in sys.path:
        sys.path.insert(0, REF_ROOT)
    import exp.comm  # noqa: F401  (real package; then override its `op` sub-package)
    _install_ops()
    sys.modules["exp.comm"].op = sys.modules["exp.comm.op"]
    _INSTALLED = True


# ffhq_exp.yaml:43-81 (G_cfg_3D2D) and :86-96 (D_cfg), minus registry keys
G_CFG = dict(
    z_dim=256,
    nerf_cfg=dict(in_dim=3, hidden_dim=128, hidden_layers=2, rgb_dim=32, style_dim=128),
    mapping_nerf_cfg=dict(z_dim=256, hidden_dim=128, base_layers=4, head_layers=0),
    inr_cfg=dict(input_dim=32, style_dim=512, hidden_dim=512, pre_rgb_dim=3),
    mapping_inr_cfg=dict(z_dim=512, hidden_dim=512, base_layers=8, head_layers=0,
                         add_norm=True, norm_out=True),
)
D_CFG = dict(diffaug=False, max_size=1024, channel_multiplier=2, first_downsample=False,
             stddev_group=0)
# ffhq_exp.yaml:117-126
G_KWARGS = dict(fov=12, ray_start=0.88, ray_end=1.12, num_steps=12, h_stddev=0.3,
                v_stddev=0.155, hierarchical_sample=True, psi=1., sample_dist="gaussian")


def build_reference_generator(device="cpu", frozen=False):
    install()
    from exp.cips3d.models import generator as ref_gen
    cls = ref_gen.GeneratorNerfINR_freeze_NeRF if frozen else ref_gen.GeneratorNerfINR
    import copy
    return cls(**copy.deepcopy(G_CFG), device=device)


def build_reference_discriminator(**over):
    install()
    from exp.cips3d.models import discriminator as ref_d
    cfg = dict(D_CFG)
    cfg.update(over)
    return ref_d.Discriminator_MultiScale_Aux(**cfg)
