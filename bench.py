#!/usr/bin/env python
"""bench.py -- generator-forward throughput of the CIPS-3D hot path on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

Metric (BASELINE.json): generator fwd images/sec @ FFHQ r256, 24 samples/ray.  A step is one
GeneratorNerfINR.forward over a batch of synthetic latents (per-GPU batch fixed -> weak scaling);
one rank per GPU, no data-path collective (SURVEY.md section 8e).  Prints ONE JSON line.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

R, BATCH_PER_GPU, NUM_STEPS = 256, 16, 12
NERF_FLOP_PER_RAY = 1302528.0      # BASELINE.md section 3 (24 points x 54 272)
CIPS_FLOP_PER_PIXEL = 8964096.0
METRIC = "generator fwd images/sec @ FFHQ r256, 24 samples/ray"
# exp/cips3d/configs/ffhq_exp.yaml:43-81 (G_cfg_3D2D) and :117-126 (G_kwargs)
G_CFG = dict(
    z_dim=256,
    nerf_cfg=dict(in_dim=3, hidden_dim=128, hidden_layers=2, rgb_dim=32, style_dim=128),
    mapping_nerf_cfg=dict(z_dim=256, hidden_dim=128, base_layers=4, head_layers=0),
    inr_cfg=dict(input_dim=32, style_dim=512, hidden_dim=512, pre_rgb_dim=3),
    mapping_inr_cfg=dict(z_dim=512, hidden_dim=512, base_layers=8, head_layers=0, add_norm=True, norm_out=True),
)
G_KWARGS = dict(fov=12, ray_start=0.88, ray_end=1.12, num_steps=12, h_stddev=0.3, v_stddev=0.155,
                hierarchical_sample=True, psi=1., sample_dist="gaussian")
WEIGHT_SEED = 1234          # ffhq_exp.yaml:146; both arms: the (reference-identical) constructor init under this seed
REF_ROOT = os.path.join(ROOT, "baseline", "_ref")
DRAW_SEED = 2000            # the forward's random draws (jitter, camera, noise) in the timed steps: the same on every run
DUMP_BYTES = 64 << 20       # --dump-outputs writes at most this much


def bench_config(res, B, world):
    """the `config` object, identical in both arms (the driver compares them)"""
    return {"workload": f"FFHQ r{res} generator forward (GeneratorNerfINR, ffhq_exp.yaml G_cfg_3D2D), "
                        f"{B} images/GPU/step, 12 coarse + 12 fine samples/ray, nerf_noise 0",
            "resolution": res, "batch_per_gpu": B, "global_batch": B * world, "samples_per_ray": 24,
            "parallelism": f"dp{world} (no data-path collective)",
            "l2": "per-step inputs (random draws ~%.0f MB) exceed the 126 MB L2" % (B * res * res * 48 * 4 / 1e6)}


def reference_generator(device):
    """The UNMODIFIED reference GeneratorNerfINR from baseline/_ref (tools/install_reference.py), tl2 satisfied by
    tools/ref_shim.py; None when the copy is absent."""
    if not os.path.isdir(os.path.join(REF_ROOT, "exp", "cips3d", "models")):
        return None
    os.environ["CIPS3D_REFERENCE"] = REF_ROOT
    tools = os.path.join(ROOT, "tools")
    if tools not in sys.path:
        sys.path.insert(0, tools)
    import ref_shim
    torch.manual_seed(WEIGHT_SEED)
    return ref_shim.build_reference_generator(device).to(device).eval()     # the constructor's `device` is only an attribute


def dump_outputs(out_dir, arrays):
    """Write each array as <out_dir>/<name>.npy in float32.  One larger than its share of DUMP_BYTES is replaced by a
    fixed seeded sample of its elements (the same positions for the same shape), so that two builds compare element
    for element."""
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_BYTES // len(arrays)
    for name, t in arrays.items():
        a = t.detach().float().cpu().numpy()
        if a.nbytes > share:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, share // a.itemsize, replace=False))]
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def peaks():
    """-> (peak TFLOP/s used for roofline.frac, HBM GB/s, source string, the other bf16 figure).  The timed region of the default run
    is a few tenths of a second, not a long sustained step, so `frac` is quoted against the BURST dense-bf16 figure (the stricter
    denominator; VERDICT r1 weak #11) and the sustained figure rides along as `frac_of_sustained`."""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d["bf16_tflops"], d["hbm_gbs"], "measured (MEASURED_PEAKS.json, burst bf16)", d.get("bf16_tflops_sustained")
    return 1590.0, 6650.0, "fallback (B200_PROFILING.md)", None


class ClockSampler(threading.Thread):
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, dev):
        super().__init__(daemon=True)
        self.dev, self.rows, self.stop_flag = dev, [], False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                      "-i", str(self.dev)], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        sm = [float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.rows)}


class CpuReference:
    """The reference's generator forward on the host cores: the UNMODIFIED reference modules from baseline/_ref
    (kind "reference") when tools/install_reference.py has put them there, else the oracle port (kind "port").
    One `step(b)` = one forward over b images at the bench resolution -- a bounded sample of the B-image bench step."""

    def __init__(self, res=R, threads=None):
        self.res = res
        self.G = reference_generator("cpu")
        if self.G is not None:
            self.kind = "reference"
            self.what = "UNMODIFIED reference GeneratorNerfINR.forward (baseline/_ref via tools/ref_shim.py), fp32 torch-CPU"
        else:
            from oracle import cips3d_oracle as O       # the one other place bench.py may execute oracle/: the CPU baseline
            self.O = O
            self.kind = "port"
            self.what = "oracle port of GeneratorNerfINR.forward (oracle/cips3d_oracle.py), fp32 torch-CPU"
            self.sd = O.synthetic_state_dict(O.generator_template(), seed=WEIGHT_SEED)
        self.gen = torch.Generator().manual_seed(0)
        self.threads = threads or self._calibrate()
        torch.set_num_threads(self.threads)

    def step(self, b, res=None):
        res = res or self.res
        zs = {"z_nerf": torch.randn(b, 256, generator=self.gen), "z_inr": torch.randn(b, 512, generator=self.gen)}
        t0 = time.perf_counter()
        with torch.no_grad():
            if self.G is not None:
                self.G(zs, img_size=res, **G_KWARGS)
            else:
                draws = self.O.draw_randoms(b, res, G_KWARGS["num_steps"], generator=self.gen)
                self.O.generator_forward(self.sd, zs, draws, img_size=res, nerf_noise=0.0, **self.O.G_KWARGS)
        return time.perf_counter() - t0

    def _calibrate(self):
        """torch-CPU scales badly past a few dozen threads: take the fastest of a few counts on a small forward"""
        best = (1e30, 1)
        self.step(1, 64)
        for th in sorted({min(os.cpu_count() or 1, t) for t in (8, 16, 32, 64, 128)}):
            torch.set_num_threads(th)
            t = min(self.step(1, 64) for _ in range(2))
            if t < best[0]:
                best = (t, th)
        return best[1]


def cpu_baseline_leg(seconds_budget=20.0):
    ref = CpuReference()
    t_one = ref.step(1)                      # warm-up (also sizes the sample)
    n = max(1, min(8, int(seconds_budget / max(t_one, 1e-3))))
    dt = sum(ref.step(1) for _ in range(n))
    return {"value": n / dt, "unit": "images/s", "cores": ref.threads, "kind": ref.kind,
            "sample": f"{n} x (1 image of the step's batch, r{R}, 12+12 samples/ray): {ref.what}"}


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation on this box's host cores, on our arm's config/metric.
    A step = the reference forward over ONE image of the B-image step (bounded sample: the full 16-image step takes
    ~1 min of CPU); value = images / time.  Rank 0 only."""
    if rank != 0:
        return
    t0 = time.perf_counter()
    ref = CpuReference(res=args.res)
    for _ in range(max(args.warmup, 0)):
        ref.step(1)
    ts = [ref.step(1) for _ in range(args.steps)]
    val = len(ts) / sum(ts)
    sample = f"each step = 1 image of the {args.batch}-image step, r{args.res}, 12+12 samples/ray: {ref.what}"
    line = {"metric": METRIC, "value": val, "unit": "images/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1000.0 * sum(ts) / len(ts), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "reference",
            "config": bench_config(args.res, args.batch, max(world, args.gpus)),
            "cpu_baseline": {"value": val, "unit": "images/s", "cores": ref.threads, "kind": ref.kind, "sample": sample},
            "e2e": {"value": val, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "wall_s": time.perf_counter() - t0}
    print(json.dumps(line), flush=True)


def reference_eager_gpu_leg(dev, res, B):
    """The unmodified reference GeneratorNerfINR as eager torch CUDA ops on this GPU (BASELINE.md section 4: "the
    implementation the new kernels have to beat"), TF32 off (torch default, the reference's setting) and on."""
    G = reference_generator(dev)
    if G is None:
        return {"unavailable": "baseline/_ref absent (tools/install_reference.py not run where /root/reference exists)"}
    out = {"impl": "UNMODIFIED reference modules (baseline/_ref), eager torch CUDA ops, fp32"}
    prev = torch.backends.cuda.matmul.allow_tf32
    try:
        for name, tf32 in (("tf32_off", False), ("tf32_on", True)):
            torch.backends.cuda.matmul.allow_tf32 = tf32
            for b in (B, 4, 1):
                try:
                    zs = G.get_zs(b)
                    with torch.no_grad():
                        G(zs, img_size=res, **G_KWARGS)
                        torch.cuda.synchronize()
                        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        n = 3
                        e0.record()
                        for _ in range(n):
                            G(zs, img_size=res, **G_KWARGS)
                        e1.record()
                        torch.cuda.synchronize()
                    out[name] = {"value": n * b / (e0.elapsed_time(e1) / 1e3), "unit": "images/s", "batch": b}
                    break
                except torch.OutOfMemoryError:
                    torch.cuda.empty_cache()
                    out[name] = {"unavailable": f"out of memory at batch {b}"}
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev
        del G
        torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH_PER_GPU, help="images per GPU per step")
    ap.add_argument("--res", type=int, default=R)
    ap.add_argument("--kernel-impl", default=os.environ.get("C3D_IMPL", "tc"), choices=["tc", "simt"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--u8", action="store_true", help="also time the uint8-delivery end-to-end leg (c3d_image_to_u8: opt-in until that "
                    "kernel has passed its GPU tests on hardware -- a fault there must not cost the contract line)")
    ap.add_argument("--no-eager", action="store_true", help="skip the eager-torch-on-the-same-GPU comparison")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned (the images and pitch/yaw "
                    "of GeneratorNerfINR.forward) as DIR/<name>.npy, float32")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return run_reference(args, rank, world)

    import torch.distributed as dist
    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    import __graft_entry__ as ge
    if rank == 0:
        ge.build()
    if world > 1:
        dist.barrier()
    os.environ["C3D_IMPL"] = args.kernel_impl
    import cips3d_b200
    from cips3d_b200 import _lib, ops
    lib = _lib.load()
    res, B = args.res, args.batch
    cfg = {k: (dict(v) if isinstance(v, dict) else v) for k, v in G_CFG.items()}
    torch.manual_seed(WEIGHT_SEED)          # the constructor reproduces the reference's init bit for bit (test_boundary_cpu)
    G = cips3d_b200.GeneratorNerfINR(**cfg, device=dev).to(dev).eval()     # parameters are initialised on the CPU, then moved
    kw = dict(G_KWARGS)
    torch.manual_seed(1000 + rank)
    zs_host = {"z_nerf": torch.randn(B, 256).pin_memory(), "z_inr": torch.randn(B, 512).pin_memory()}
    zs_dev = {k: v.to(dev) for k, v in zs_host.items()}
    out_host = torch.empty((B, 3, res, res), dtype=torch.float32).pin_memory()

    def step_resident():
        with torch.no_grad():
            return G(zs_dev, img_size=res, nerf_noise=0.0, **kw)

    def step_e2e():
        with torch.no_grad():
            z = {k: v.to(dev, non_blocking=True) for k, v in zs_host.items()}
            img, _ = G(z, img_size=res, nerf_noise=0.0, **kw)
            out_host.copy_(img.contiguous(), non_blocking=True)
        return img

    def timed(fn, steps, warmup, profile=False):
        t_ramp = time.perf_counter()          # SM clocks ramp from idle (120 MHz) over ~1 s of load: untimed pre-warm
        while time.perf_counter() - t_ramp < 1.5:
            fn()
            torch.cuda.synchronize()
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ops.PROFILE = {} if profile else None
        torch.manual_seed(DRAW_SEED + rank)    # the pre-warm runs for a time, not a count: reseed so every run draws alike
        l0 = lib.c3d_launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        out = None
        e0.record()
        for _ in range(steps):
            out = fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        launches = lib.c3d_launch_count() - l0
        prof, ops.PROFILE = ops.PROFILE, None
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dist.barrier()
            ms = t.item()
        return ms, launches, prof, out

    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    ms, launches, prof, last = timed(step_resident, args.steps, args.warmup, profile=True)
    ms_e2e, _, _, _ = timed(step_e2e, args.steps, max(1, args.warmup // 2))
    if sampler:
        sampler.stop_flag = True
        sampler.join(timeout=2)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"img": last[0], "pitch_yaw": last[1]})
    del last
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    imgs = B * world * args.steps
    value = imgs / (ms / 1e3)
    e2e = imgs / (ms_e2e / 1e3)
    peak_tf, peak_hbm, peak_src, peak_sustained = peaks()
    roof = {}
    for key, flop_unit, units in (("cips", CIPS_FLOP_PER_PIXEL, B * res * res), ("ray", NERF_FLOP_PER_RAY, B * res * res)):
        evs = (prof or {}).get(key, [])
        if evs:
            t_ms = float(np.median([a.elapsed_time(b) for a, b in evs]))
            ach = flop_unit * units / (t_ms * 1e-3) / 1e12
            roof[key] = {"bound": "tensor", "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach / peak_tf,
                         "traffic": None, "kernel_ms": t_ms, "launches_timed": len(evs),
                         "algorithmic_flop_per_launch": flop_unit * units, "peak_source": peak_src,
                         "peak_sustained": peak_sustained, "frac_of_sustained": (ach / peak_sustained) if peak_sustained else None}
    # DRAM traffic per launch from the committed ncu --set full capture of this workload (profiles/traffic.json)
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        tj = json.load(open(tpath))
        for key, kname in (("cips", "c3d_cips_fwd"), ("ray", "c3d_ray_siren_fwd")):
            ent = tj.get(kname)
            if key in roof and ent and ent.get("batch") == B and ent.get("resolution") == res:
                roof[key]["traffic"] = ent["dram_bytes_per_launch"]
                roof[key]["traffic_source"] = ent.get("source")
    dominant = max(roof, key=lambda k: roof[k]["kernel_ms"]) if roof else None
    line = {
        "metric": METRIC, "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f16-split (fp32-equivalent) ray MLP, f16 CIPS MLP, fp32 accumulate"
        if args.kernel_impl == "tc" else "f32",
        "data": "synthetic",
        "config": bench_config(res, B, world),
        # kernel selection in effect (all unset = the defaults of this build)
        "kernel": {"impl": args.kernel_impl,
                   "variants": {k: os.environ[k] for k in ("C3D_CIPS_PAIR", "C3D_CIPS_CLUSTER", "C3D_RAY_MATH", "C3D_BLUR_TMA", "C3D_STYLE_PREP")
                                if os.environ.get(k)}},
        "e2e": {"value": e2e, "unit": "images/s", "h2d_bytes_per_step": int(B * (256 + 512) * 4),
                "d2h_bytes_per_step": int(B * 3 * res * res * 4), "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": int(launches),
        "clocks": sampler.summary() if sampler else None,
    }
    if dominant:
        line["roofline"] = dict(roof[dominant], kernel=("c3d_cips_fwd" if dominant == "cips" else "c3d_ray_siren_fwd"))
        other = "ray" if dominant == "cips" else "cips"
        if other in roof:
            line["roofline_secondary"] = dict(roof[other], kernel=("c3d_cips_fwd" if other == "cips" else "c3d_ray_siren_fwd"))
    if world == 1 and not args.no_eager:
        # the same forward as eager torch CUDA ops (fp32, TF32 off = torch default) on this GPU: what the reference's
        # PyTorch path executes; chunk the batch if the per-sample tensors would not fit
        try:
            G.force_torch_path = True
            eb = min(B, 4)
            ze = {k: v[:eb] for k, v in zs_dev.items()}
            with torch.no_grad():
                G(ze, img_size=res, nerf_noise=0.0, **kw)
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(2):
                    G(ze, img_size=res, nerf_noise=0.0, **kw)
                e1.record()
                torch.cuda.synchronize()
            line["torch_eager_same_gpu"] = {"value": 2 * eb / (e0.elapsed_time(e1) / 1e3), "unit": "images/s", "batch": eb,
                                            "note": "identical math as eager torch CUDA ops (cuBLAS fp32, TF32 off) through the same "
                                                    "module surface; not the product path"}
        except Exception as ex:  # out of memory etc. -- report, do not fail the bench
            line["torch_eager_same_gpu"] = {"unavailable": str(ex)[:120]}
        finally:
            G.force_torch_path = False
            torch.cuda.empty_cache()
    if world == 1 and args.u8:
        # the evaluation-dump form of the same end-to-end step (inference.gen_images: SURVEY 8(f) rank 4): the images leave
        # the GPU as uint8, converted by c3d_image_to_u8 -- 1 byte per sample over PCIe instead of 4.  Extra information,
        # measured after every contract number above is already taken.
        try:
            u8_host = torch.empty((B, res, res, 3), dtype=torch.uint8).pin_memory()

            def step_u8():
                with torch.no_grad():
                    z = {k: v.to(dev, non_blocking=True) for k, v in zs_host.items()}
                    img, _ = G(z, img_size=res, nerf_noise=0.0, **kw)
                    u8_host.copy_(ops.image_to_u8(img), non_blocking=True)

            for _ in range(2):
                step_u8()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                step_u8()
            e1.record()
            torch.cuda.synchronize()
            line["e2e_uint8"] = {"value": B * args.steps / (e0.elapsed_time(e1) / 1e3), "unit": "images/s",
                                 "h2d_bytes_per_step": int(B * (256 + 512) * 4), "d2h_bytes_per_step": int(B * 3 * res * res),
                                 "note": "same step, result delivered as (B, H, W, 3) uint8 = save_image's bytes"}
        except Exception as ex:
            line["e2e_uint8"] = {"unavailable": str(ex)[:120]}
    if world == 1 and not args.no_cpu_baseline:
        try:          # extra information: a failure here must never cost the contract line
            line["vs_reference_gpu_eager"] = reference_eager_gpu_leg(dev, res, B) if not args.no_eager else None
        except Exception as ex:
            line["vs_reference_gpu_eager"] = {"unavailable": f"{type(ex).__name__}: {str(ex)[:160]}"}
        if isinstance(line["vs_reference_gpu_eager"], dict):
            for k in ("tf32_off", "tf32_on"):
                ent = line["vs_reference_gpu_eager"].get(k)
                if isinstance(ent, dict) and ent.get("value"):
                    ent["ours_over_reference"] = value / ent["value"]
        try:
            line["cpu_baseline"] = cpu_baseline_leg(20.0)
        except Exception as ex:
            line["cpu_baseline"] = {"unavailable": f"{type(ex).__name__}: {str(ex)[:160]}"}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
