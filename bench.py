#!/usr/bin/env python
"""bench.py -- edited images/sec at 512x512 / 50-step DDIM / CFG (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" = one complete CFG DDIM sampling run (``DDIMSampler.sample``: 50 UNet evaluations on the
CFG-doubled batch + 50 fused updates) over one batch of synthetic edit requests.  Headline workload at every
N = BASELINE configs[1] per GPU (512x512 "replace" edit -> 64x64 latent, 50 DDIM steps, CFG 7.5,
batch 8, SD-1.5/IP2P UNet geometry with 8 input channels and 77x768 text context); N GPUs run N
such batches (weak scaling), no collective inside the loop.

Prints ONE JSON line (rank 0).  ``value`` is device-resident throughput, ``e2e`` the same metric
through the public API with pinned-host inputs/outputs inside the timed region.  The same line carries

  roofline       tensor-core contraction kernels of one UNet evaluation, CUDA events per launch
  cpu_baseline   the reference's own UNetModel + DDIMSampler (oracle/_ref staged copy; the restatement when absent)
                 on a bounded sample, host cores stated
  parity_check   eps of request 0 in the LAST timed graph replay vs the CPU reference on the same weights / inputs
  extra_configs  measured after the headline:  C2 (configs[2]: 20 mixed edit types, task router + task embedding +
                 expert streams active, 64 requests over the N GPUs), C3 (configs[3]: 768x768, 100 steps, visual tokens,
                 2 requests per GPU), C4 (configs[4]: one training step of the adapters per GPU at batch 16 with the NCCL
                 gradient all-reduce), dpm20 (configs[1] with 20-step DPM-Solver++(2M) instead of 50-step DDIM)
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SD15 = dict(image_size=32, in_channels=8, model_channels=320, out_channels=4, num_res_blocks=2,
            attention_resolutions=[4, 2, 1], channel_mult=[1, 2, 4, 4], num_heads=8,
            use_spatial_transformer=True, transformer_depth=1, context_dim=768, legacy=False)
# algorithmic FLOPs of one UNet sample-forward (SURVEY.md Appendix A): latent side -> FLOP
F_UNET = {32: 180.13e9, 64: 803.37e9, 96: 2148.33e9}
F64 = F_UNET[64]
METRIC = "edited images/sec (512x512, 50-step DDIM, CFG)"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=8, help="edit requests per GPU")
    ap.add_argument("--latent", type=int, default=64)
    ap.add_argument("--ddim-steps", type=int, default=50)
    ap.add_argument("--scale", type=float, default=7.5)
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--skip-cpu", action="store_true", help="skip the cpu_baseline and parity_check legs (profiling runs)")
    ap.add_argument("--skip-roofline", action="store_true")
    ap.add_argument("--skip-extra", action="store_true", help="skip the C2 / C3 / C4 / dpm20 / pipeline legs")
    ap.add_argument("--extra", default="C2,C3,C4,dpm20,pipeline", help="comma list of extra legs to run")
    ap.add_argument("--c2-total", type=int, default=64, help="configs[2]: requests summed over all GPUs")
    ap.add_argument("--c2-chunk", type=int, default=16, help="configs[2]: requests per sampling call on one GPU")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed sampling call returned (rank 0) as DIR/<name>.npy, float32")
    args = ap.parse_args()
    if args.dump_outputs and args.steps < 1:
        ap.error("--dump-outputs needs --steps >= 1")
    return args


# ---- clocks sampler (nvidia-smi during the timed region) ------------------------------------------
class Clocks:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "200"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        # "under load": the upper half of the samples (the sampler also sees the idle edges)
        load = sm[len(sm) // 2:] if sm else []
        med = load[len(load) // 2] if load else None
        return {"sm_mhz": med, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# ---- CPU arm: the reference's own UNetModel + DDIMSampler (staged copy), else the restatement -------------------
_CPU = {}


def _cpu_state_dict():
    """859.5 M seeded weights, generated once per process (untimed)."""
    import torch
    from oracle import weights
    from anyedit_b200.unet import UNetModel
    if "sd" not in _CPU:
        with torch.device("meta"):
            shapes = {k: tuple(v.shape) for k, v in UNetModel(**SD15).state_dict().items()}
        _CPU["sd"] = weights.make_state_dict(shapes, 3)
    return _CPU["sd"]


def _cpu_reference_unet(sd):
    """The reference ``UNetModel`` (openaimodel.py:412-786) built from the staged sources, or None when absent."""
    import torch
    from oracle import ref_import
    if not ref_import.available():
        return None, None
    if "ref" not in _CPU or _CPU.get("ref_sd") is not sd:
        UNetModel, DDIMSamplerCPU, _ = ref_import.load()
        with torch.device("meta"):
            net = UNetModel(**SD15)
        net = net.to_empty(device="cpu").eval()
        net.load_state_dict(sd)
        _CPU["ref"], _CPU["ref_sampler"], _CPU["ref_sd"] = net, DDIMSamplerCPU, sd
    return _CPU["ref"], _CPU["ref_sampler"]


def cpu_arm(latent, ddim_steps, scale, n_steps_sample=3):
    """Times the reference's CPU implementation of the path (eager torch fp32, all usable host threads) on a bounded
    sample of the workload: ONE edit request, CFG (B_eff = 2), ``n_steps_sample`` DDIM steps after one warm-up step
    (a (1 + n)-step ``DDIMSampler.sample``; every UNet call timed); images/sec extrapolated linearly to ``ddim_steps``."""
    import torch
    from oracle import ddim_oracle, ref_import, unet_oracle
    from oracle.cpu import usable_cores
    cores = usable_cores()              # min(affinity, cgroup CPU quota): what the box lets us use
    torch.set_num_threads(cores)
    sd = _cpu_state_dict()
    gen = torch.Generator().manual_seed(1234)
    x_T, c_cat = torch.randn(1, 4, latent, latent, generator=gen), torch.randn(1, 4, latent, latent, generator=gen)
    c_txt, u_txt = torch.randn(1, 77, 768, generator=gen), torch.randn(1, 77, 768, generator=gen)
    cond = {"c_concat": [c_cat], "c_crossattn": [c_txt]}
    uncond = {"c_concat": [c_cat], "c_crossattn": [u_txt]}
    sched = ddim_oracle.register_schedule("linear", 1000, 0.00085, 0.012)
    times = []
    ref_net, ref_sampler = _cpu_reference_unet(sd)
    # S must divide 1000 for the reference's uniform schedule (util.py:46-60): 1 + n in {2, 4, 5, 8, 10}
    S = {1: 2, 3: 4}.get(n_steps_sample, n_steps_sample + 1)
    with torch.no_grad():
        if ref_net is not None:
            kind = "reference"
            shim = ref_import.RefModelShim(ref_net, sched, "hybrid")
            inner = shim.apply_model

            def timed_apply(x, t, c):
                t0 = time.perf_counter()
                out = inner(x, t, c)
                times.append(time.perf_counter() - t0)
                return out

            shim.apply_model = timed_apply
            import contextlib
            import io
            with contextlib.redirect_stdout(io.StringIO()):      # the reference prints its banner on stdout; ours carries ONE JSON line
                ref_sampler(shim).sample(S, 1, (4, latent, latent), cond, verbose=False, x_T=x_T, eta=0.0,
                                         unconditional_guidance_scale=scale, unconditional_conditioning=uncond)
            what = "the reference's own ldm UNetModel + DDIMSampler (oracle/_ref staged sources"
        else:
            kind = "port"
            unet = lambda x, t, context=None, y=None: unet_oracle.unet_forward(sd, x, t, context, y, num_heads=8)

            def model_fn(x, t, c):
                t0 = time.perf_counter()
                out = ddim_oracle.apply_model(unet, "hybrid", x, t, c)
                times.append(time.perf_counter() - t0)
                return out

            ddim_oracle.ddim_sample(model_fn, sched, S, x_T, cond, uncond, scale, eta=0.0)
            what = "oracle restatement of the reference ldm UNetModel + DDIMSampler (oracle/_ref absent"
    per_step = sum(times[1:]) / max(1, len(times) - 1)
    ips = 1.0 / (per_step * ddim_steps)
    return {"value": ips, "unit": "images/s", "cores": cores, "kind": kind,
            "sample": f"{what}; fp32 eager torch, {cores} threads): 1 request, CFG B_eff=2, {latent}x{latent} latent, "
                      f"{len(times) - 1} DDIM steps after 1 warm-up ({per_step:.2f} s/step), extrapolated linearly to "
                      f"{ddim_steps} steps",
            "sec_per_unet_step": per_step}


def run_reference(args, rank, world):
    if rank != 0:
        return
    t_steps = []
    last = None
    for i in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        last = cpu_arm(args.latent, args.ddim_steps, args.scale, n_steps_sample=1 if i < args.warmup else 3)
        if i >= args.warmup:
            t_steps.append(time.perf_counter() - t0)
    ips = last["value"]
    line = {"impl": "reference", "metric": METRIC, "value": ips, "unit": "images/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * sum(t_steps) / len(t_steps),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args, world), "cpu_baseline": {**last, "value": ips},
            "e2e": {"value": ips, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def workload_config(args, world):
    return {"workload": f"BASELINE configs[1] per GPU: {8 * args.latent}x{8 * args.latent} replace edit, "
                        f"{args.ddim_steps} DDIM steps + CFG {args.scale}, batch {args.batch}/GPU "
                        f"(SD-1.5/IP2P UNet geometry: in=8, 320ch, mult 1-2-4-4, 8 heads, ctx 77x768)",
            "global_batch": args.batch * world, "latent": args.latent, "ddim_steps": args.ddim_steps,
            "guidance_scale": args.scale, "parallelism": f"dp{world} (requests sharded, no in-loop collective)",
            "l2_policy": "working set > L2 every step (1.72 GB fp16 weights + >1 GB activations vs 126 MB L2)"}


def synth_requests(B, h, seed, n_vis=0, vis_zero=False, first_index=0):
    """Pinned-host synthetic edit requests (SURVEY.md 8d): x_T, source-image latent, text context, one shared null
    text, optional visual tokens and edit codes (arange % 20 over the GLOBAL request index)."""
    import torch
    gen = torch.Generator().manual_seed(seed)
    host = {"x_T": torch.randn(B, 4, h, h, generator=gen), "c_cat": torch.randn(B, 4, h, h, generator=gen),
            "c_txt": torch.randn(B, 77, 768, generator=gen),
            "u_txt": torch.randn(1, 77, 768, generator=torch.Generator().manual_seed(4321)).repeat(B, 1, 1)}
    if n_vis:
        host["vis"] = torch.zeros(B, n_vis, 768) if vis_zero else torch.randn(B, n_vis, 768, generator=gen)
        host["code"] = (torch.arange(B) + first_index) % 20
    return {k: v.pin_memory() for k, v in host.items()}


def conds(devt):
    cond = {"c_concat": [devt["c_cat"]], "c_crossattn": [devt["c_txt"]]}
    uncond = {"c_concat": [devt["c_cat"]], "c_crossattn": [devt["u_txt"]]}
    if "vis" in devt:        # AnySD keys (anyedit_b200.anysd.AnySDDenoiser): both CFG halves see the same task / reference image
        for c in (cond, uncond):
            c["c_visual"], c["c_task"] = [devt["vis"]], devt["code"]
    return cond, uncond


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, last):
    """Writes what ``DDIMSampler.sample`` returned in the final timed call: ``samples`` [B, 4, h, h] and the logged
    ``x_inter_<i>`` / ``pred_x0_<i>`` latents, float32 .npy.  Inputs are seeded, so two builds can be compared file by file.
    Should the arrays pass DUMP_BYTES in all, each is cut to the same seeded sample of its flattened elements."""
    import numpy as np
    import torch
    arrays = {"samples": last["samples"]}
    for key in ("x_inter", "pred_x0"):
        arrays.update({f"{key}_{i}": t for i, t in enumerate(last["intermediates"][key])})
    arrays = {k: v.detach().float().cpu() for k, v in arrays.items()}
    budget = DUMP_BYTES - 4096 * len(arrays)           # room for the .npy headers
    keep = min(1.0, budget / sum(4 * a.numel() for a in arrays.values()))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        if keep < 1.0:
            idx = torch.randperm(a.numel(), generator=torch.Generator().manual_seed(0))[:int(keep * a.numel())]
            a = a.reshape(-1)[idx.sort().values]
        np.save(os.path.join(out_dir, f"{name}.npy"), a.numpy())


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    from anyedit_b200 import distributed as D
    from anyedit_b200 import ops
    from anyedit_b200.ddim import DDIMSampler
    from anyedit_b200.diffusion import LatentDenoiser
    from anyedit_b200.unet import UNetModel

    rank, local, world = D.init_from_env()
    assert torch.cuda.is_available(), "bench.py needs a CUDA device: anyedit_b200 has no CPU fallback"
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)

    # ---- model: random-init weights of the named architecture, built on rank 0, broadcast once ----
    torch.manual_seed(0)
    with torch.device(dev):
        net = UNetModel(**SD15)
    with torch.no_grad():
        for name, p in net.named_parameters():      # re-randomise the zero-init tensors
            if float(p.abs().max()) == 0.0 and p.dim() > 1:
                fan_in = p[0].numel()
                p.uniform_(-(3.0 / fan_in) ** 0.5, (3.0 / fan_in) ** 0.5)
    model = LatentDenoiser(net, "hybrid").to(dev)
    D.broadcast_module_(model, src=0)                # the one collective of the inference path
    net.prepare()

    def timed(fn, n):
        D.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        D.barrier()
        return D.max_over_ranks(e0.elapsed_time(e1) / 1e3, dev)

    def sampling_leg(sampler_obj, hosts, S, h, scale, warmup, steps, method="ddim"):
        """Times `steps` passes over the list of request chunks `hosts` (each one sampler call), resident and e2e.
        Returns (t_resident, t_e2e, kernel launches per resident pass, h2d bytes, d2h bytes)."""
        outs = [torch.empty(hh["x_T"].shape).pin_memory() for hh in hosts]

        def run(devt):
            cond, uncond = conds(devt)
            out, _ = sampler_obj.sample(S, devt["x_T"].shape[0], (4, h, h), cond, verbose=False, x_T=devt["x_T"], eta=0.0,
                                        unconditional_guidance_scale=scale, unconditional_conditioning=uncond)
            return out

        devs = [{k: v.to(dev) for k, v in hh.items()} for hh in hosts]

        def resident():
            for d_ in devs:
                run(d_)

        def e2e():
            for hh, oh in zip(hosts, outs):
                oh.copy_(run({k: v.to(dev, non_blocking=True) for k, v in hh.items()}), non_blocking=True)

        for _ in range(warmup):
            resident()
        n0 = ops.launch_count
        t_res = timed(resident, steps)
        launches = (ops.launch_count - n0) // max(1, steps)
        t_e2e = timed(e2e, steps)
        h2d = sum(v.numel() * v.element_size() for hh in hosts for v in hh.values())
        d2h = sum(o.numel() * o.element_size() for o in outs)
        return t_res, t_e2e, launches, h2d, d2h

    B, h, S = args.batch, args.latent, args.ddim_steps
    host = synth_requests(B, h, 1234 + rank)
    sampler = DDIMSampler(model, use_cuda_graph=not args.no_graph)

    clocks = Clocks(local)
    # warm-up first (the clock sampler should see the timed region)
    devt = {k: v.to(dev) for k, v in host.items()}
    for _ in range(args.warmup):
        c_, u_ = conds(devt)
        sampler.sample(S, B, (4, h, h), c_, verbose=False, x_T=devt["x_T"], eta=0.0, unconditional_guidance_scale=args.scale,
                       unconditional_conditioning=u_)
    if rank == 0:
        clocks.start()
    last = {}
    if args.dump_outputs:                 # keep what each sampler call returns; without the flag the timed path is untouched
        sample = sampler.sample

        def recorded_sample(*a, **kw):
            last["samples"], last["intermediates"] = res = sample(*a, **kw)
            return res
        sampler.sample = recorded_sample
    if os.environ.get("ANYSD_NCU"):      # ncu --profile-from-start off: launch list of the timed region only
        torch.cuda.cudart().cudaProfilerStart()
    t_res, t_e2e, launches, h2d, d2h = sampling_leg(sampler, [host], S, h, args.scale, 0, args.steps)
    launches *= args.steps                # the headline reports the launches of the whole timed region
    if os.environ.get("ANYSD_NCU"):
        torch.cuda.cudart().cudaProfilerStop()
    clk = clocks.stop() if rank == 0 else None
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, last)

    imgs = B * world * args.steps
    value, e2e = imgs / t_res, imgs / t_e2e

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = peaks.get("bf16_tflops_sustained", 1400.0)
    peak_src = "MEASURED_PEAKS.json bf16_tflops_sustained (of measured)" if peaks else "fallback 1400 (B200_PROFILING.md)"

    # ---- parity of the timed path: eps of request 0 in the LAST graph replay vs the CPU reference ----
    parity = None
    if rank == 0 and not args.skip_cpu:
        parity = parity_check(sampler, net, devt, B, h)

    # ---- roofline of the dominant kernel (tensor-core contraction: conv3x3 + linear GEMMs) --------
    roof = None
    if not args.skip_roofline and rank == 0:
        ops.trace = []
        x_in = torch.cat([devt["x_T"]] * 2)
        cond2 = {"c_concat": [torch.cat([devt["c_cat"]] * 2)], "c_crossattn": [torch.cat([devt["u_txt"], devt["c_txt"]])]}
        tt = torch.full((2 * B,), 500, device=dev, dtype=torch.long)
        for _ in range(2):
            ops.trace.clear()
            torch.cuda.synchronize()
            # the host needs longer to issue an eager forward (~440 launches) than the GPU to run it: without a head start
            # the event intervals would include launch latency.  ~25 ms of spinning keeps the device behind the host.
            torch.cuda._sleep(int(5e7))
            model.apply_model(x_in, tt, cond2)       # eager (no graph): events around every contraction launch
        torch.cuda.synchronize()
        agg = {}
        for kind, fl, e0, e1, _tag in ops.trace:
            a = agg.setdefault(kind, [0.0, 0.0, 0])
            a[0] += fl
            a[1] += e0.elapsed_time(e1) * 1e-3
            a[2] += 1
        ops.trace = None
        gemm_f = agg.get("gemm", [0, 0, 0])[0] + agg.get("conv3x3", [0, 0, 0])[0]
        gemm_t = agg.get("gemm", [0, 1e-9, 0])[1] + agg.get("conv3x3", [0, 0, 0])[1]
        ach = gemm_f / gemm_t / 1e12
        traffic = None
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "dominant_kernel_traffic.json"))).get("bytes_per_launch")
        except Exception:
            pass
        roof = {"bound": "tensor", "kernel": "implicit-GEMM conv3x3 + linear contraction (anysd_gemm_f16)",
                "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak, "peak_source": peak_src,
                "traffic": traffic,
                "per_kind": {k: {"tflops": (v[0] / v[1] / 1e12) if v[0] else None, "ms": v[1] * 1e3, "launches": v[2], "gflop": v[0] / 1e9}
                             for k, v in agg.items()},
                "whole_step_tflops": 2 * S * F_UNET[h] * B * world * args.steps / t_res / 1e12 if h in F_UNET else None}
        if roof["whole_step_tflops"]:
            roof["whole_step_frac"] = roof["whole_step_tflops"] / (peak * world)

    # ---- extra configs (BASELINE configs[2..4] + the DPM-Solver++ variant of configs[1]) ---------------------------
    extra = None
    if not args.skip_extra:
        extra = {}
        legs = [s for s in args.extra.split(",") if s]
        for leg in legs:
            try:
                extra[leg] = extra_leg(leg, args, net, model, dev, rank, world, sampling_leg, timed, peak)
            except Exception as e:                      # an extra leg must never take the headline down
                extra[leg] = {"error": f"{type(e).__name__}: {str(e).splitlines()[0][:200]}"}
                try:
                    torch.cuda.synchronize()
                except Exception:
                    pass

    cpu = None
    if rank == 0 and world == 1 and not args.skip_cpu:
        cpu = cpu_arm(h, S, args.scale)

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": 1e3 * t_res / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
                "config": workload_config(args, world), "clocks": clk,
                "e2e": {"value": e2e, "unit": "images/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "ms_per_step": 1e3 * t_e2e / args.steps},
                "gpu_launches": launches, "roofline": roof, "cpu_baseline": cpu, "parity_check": parity,
                "extra_configs": extra}
        print(json.dumps(line), flush=True)
    if world > 1:
        torch.distributed.destroy_process_group()


def parity_check(sampler, net, devt, B, h, tol=4e-3):
    """The stepper keeps the model output of its latest step (``last_eps``) and that step's input latent (``x_buf``):
    request 0's uncond / cond rows of the LAST graph replay of the timed region are recomputed by the CPU reference on
    the same weights (state_dict copied to the host) and inputs."""
    import torch
    from oracle import ref_import, unet_oracle
    from oracle.cpu import usable_cores
    st = next(reversed(sampler._graphs.values()))
    eps = st.last_eps.detach().float().cpu()
    x0 = st.x_buf[:1].detach().cpu()
    t_val = int(st.t_buf[0])
    sd = {k: v.detach().float().cpu() for k, v in net.state_dict().items()}
    torch.set_num_threads(usable_cores())
    x8 = torch.cat([x0, devt["c_cat"][:1].cpu()], 1)
    t = torch.full((1,), t_val, dtype=torch.long)
    ctxs = (devt["u_txt"][:1].cpu(), devt["c_txt"][:1].cpu())
    with torch.no_grad():
        if ref_import.available():
            UNetModel, _, _ = ref_import.load()
            with torch.device("meta"):
                ref = UNetModel(**SD15)
            ref = ref.to_empty(device="cpu").eval()
            ref.load_state_dict(sd)
            outs = [ref(x8, t, context=c) for c in ctxs]
            against = "reference (oracle/_ref staged ldm UNetModel, CPU fp32)"
            del ref
        else:
            outs = [unet_oracle.unet_forward(sd, x8, t, c, None, num_heads=8) for c in ctxs]
            against = "port (oracle/unet_oracle.py, CPU fp32)"
    rel = lambda a, b: float((a.double() - b.double()).norm() / b.double().norm())
    e_u, e_c = rel(eps[0], outs[0][0]), rel(eps[B], outs[1][0])
    return {"what": f"eps of request 0 (uncond, cond rows of B_eff={2 * B}) from the last CUDA-graph replay of the timed region, t={t_val}",
            "against": against, "rel_l2_uncond": e_u, "rel_l2_cond": e_c, "tol": tol, "graph": st.graph is not None,
            "shared_cfg_halves": bool(st.shared), "ok": bool(e_u < tol and e_c < tol)}


def extra_leg(leg, args, net, model, dev, rank, world, sampling_leg, timed, peak):
    import torch
    from anyedit_b200 import distributed as D
    from anyedit_b200 import ops
    from anyedit_b200.anysd import AnySDDenoiser, MoE
    from anyedit_b200.ddim import DDIMSampler

    def make_moe():
        """11 experts, 20 task codes (train.py:420-421); adapter / router / task tensors random (none is zero), identical
        on every rank (seeded) and broadcast like the frozen weights."""
        if not hasattr(extra_leg, "_moe"):
            torch.manual_seed(77)
            with torch.device(dev):
                moe = MoE(net, None, expert_num=11, num_tasks=20)
            with torch.no_grad():
                moe.task_embs.weight.normal_(0.0, 0.5)
            D.broadcast_module_(moe, src=0)
            extra_leg._moe = moe
        return extra_leg._moe

    if leg == "C2":
        total, chunk = args.c2_total, args.c2_chunk
        lo, hi = D.shard_range(total, rank, world)
        moe = make_moe()
        den = AnySDDenoiser(moe).to(dev)
        hosts = [synth_requests(min(chunk, hi - s), 64, 5000 + s, n_vis=16, vis_zero=True, first_index=s) for s in range(lo, hi, chunk)]
        smp = DDIMSampler(den, use_cuda_graph=not args.no_graph)
        t_res, t_e2e, launches, h2d, d2h = sampling_leg(smp, hosts, 50, 64, args.scale, 1, 1)
        fl = 2 * 50 * F64 * total
        return {"metric": "edited images/sec (512x512, 50-step DDIM, CFG, 20 mixed edit types: task router + task embedding + 11 expert streams)",
                "value": total / t_res, "unit": "images/s", "scaling": "strong", "ms_per_step": 1e3 * t_res,
                "e2e": {"value": total / t_e2e, "unit": "images/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
                "gpu_launches": launches, "whole_step_tflops": fl / t_res / 1e12, "whole_step_frac": fl / t_res / 1e12 / (peak * world),
                "config": {"workload": f"BASELINE configs[2]: {total} requests over {world} GPU(s) ({hi - lo} on this one, sampled {chunk} at a "
                                       f"time), edit_code = arange % 20, 16 visual tokens (zeros, SURVEY.md 8d) through 11 experts x 16 layers",
                           "global_batch": total, "latent": 64, "ddim_steps": 50, "guidance_scale": args.scale}}
    if leg == "C3":
        moe = make_moe()
        den = AnySDDenoiser(moe).to(dev)
        Bc = 2
        hosts = [synth_requests(Bc, 96, 7000 + rank, n_vis=16, first_index=rank * Bc)]
        smp = DDIMSampler(den, use_cuda_graph=not args.no_graph)
        t_res, t_e2e, launches, h2d, d2h = sampling_leg(smp, hosts, 100, 96, args.scale, 1, 1)
        n = Bc * world
        fl = 2 * 100 * F_UNET[96] * n
        return {"metric": "edited images/sec (768x768, 100-step DDIM, CFG, visual-conditioning stream)", "value": n / t_res, "unit": "images/s",
                "scaling": "weak", "ms_per_step": 1e3 * t_res,
                "e2e": {"value": n / t_e2e, "unit": "images/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
                "gpu_launches": launches, "whole_step_tflops": fl / t_res / 1e12, "whole_step_frac": fl / t_res / 1e12 / (peak * world),
                "config": {"workload": f"BASELINE configs[3] geometry: 768x768 visual_material_transfer (96x96 latent, 9216-token self-attention), "
                                       f"100 DDIM steps + CFG, {Bc} requests per GPU, 16 visual tokens ~N(0,1) through the expert streams",
                           "global_batch": n, "latent": 96, "ddim_steps": 100, "guidance_scale": args.scale}}
    if leg == "C4":
        from anyedit_b200.training import AdapterTrainer
        moe = make_moe()
        Bt = 16
        g = torch.Generator(device=dev).manual_seed(100 + rank)
        rn = lambda *s: torch.randn(*s, device=dev, generator=g)
        host = {"lat": torch.randn(Bt, 4, 64, 64), "noise": torch.randn(Bt, 4, 64, 64), "img": torch.randn(Bt, 4, 64, 64),
                "text": torch.randn(Bt, 77, 768), "vis": torch.randn(Bt, 16, 768)}
        host = {k: v.pin_memory() for k, v in host.items()}
        t_idx = torch.randint(0, 1000, (Bt,), device=dev, generator=g)
        code = (torch.arange(Bt, device=dev) + rank * Bt) % 20
        tr = AdapterTrainer(moe, lr=1e-5)
        devt = {k: v.to(dev) for k, v in host.items()}
        loss_host = torch.zeros(1).pin_memory()

        def resident():
            tr.step(devt["lat"], devt["noise"], t_idx, devt["img"], devt["text"], devt["vis"], code)

        def e2e():
            d_ = {k: v.to(dev, non_blocking=True) for k, v in host.items()}
            loss, _ = tr.step(d_["lat"], d_["noise"], t_idx, d_["img"], d_["text"], d_["vis"], code)
            loss_host.copy_(loss, non_blocking=True)

        for _ in range(2):
            resident()
        n0 = ops.launch_count
        steps = 3
        t_res = timed(resident, steps)
        launches = (ops.launch_count - n0) // steps
        t_e2e = timed(e2e, steps)
        n = Bt * world * steps
        fl = 3 * F64 * n
        moe.invalidate()                               # the adapters moved: nothing cached may survive into a later leg
        return {"metric": "training samples/sec (train.py DDPM noise-prediction step, 512x512, adapters only, NCCL gradient all-reduce)",
                "value": n / t_res, "unit": "samples/s", "scaling": "weak", "ms_per_step": 1e3 * t_res / steps,
                "e2e": {"value": n / t_e2e, "unit": "samples/s", "h2d_bytes_per_step": sum(v.numel() * 4 for v in host.values()),
                        "d2h_bytes_per_step": 4},
                "gpu_launches": launches, "whole_step_tflops": fl / t_res / 1e12, "whole_step_frac": fl / t_res / 1e12 / (peak * world),
                "loss": float(loss_host[0]),
                "config": {"workload": f"BASELINE configs[4]: AdapterTrainer.step (q_sample, taped forward, explicit backward through the frozen "
                                       f"UNet, AdamW on 11 experts x 16 layers + router + task table), batch {Bt}/GPU @64x64 latent, 16 visual "
                                       f"tokens, gradient all-reduce over {world} rank(s)", "global_batch": Bt * world}}
    if leg == "dpm20":
        from anyedit_b200.dpm_solver import DPMSolverSampler
        B, h = args.batch, args.latent
        hosts = [synth_requests(B, h, 1234 + rank)]
        smp = DPMSolverSampler(model, use_cuda_graph=not args.no_graph)
        t_res, t_e2e, launches, h2d, d2h = sampling_leg(smp, hosts, 20, h, args.scale, 2, 2)
        n = B * world * 2
        return {"metric": "edited images/sec (512x512, 20-step DPM-Solver++(2M), CFG)", "value": n / t_res, "unit": "images/s",
                "scaling": "weak", "ms_per_step": 1e3 * t_res / 2,
                "e2e": {"value": n / t_e2e, "unit": "images/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
                "gpu_launches": launches,
                "config": {"workload": "BASELINE configs[1] requests, sampled with the reference's DPMSolverSampler settings "
                                       "(dpm_solver/sampler.py:14-87: multistep, order 2, time_uniform, 20 steps) instead of 50-step DDIM",
                           "global_batch": B * world, "latent": h, "steps": 20}}
    if leg == "pipeline":
        # The whole edit request, stage by stage as visual_reference_tool.py:190-225 / the IP2P loop (SURVEY.md 3.1, 3.4) run it:
        # CLIP-L text tower on the prompt and on the null prompt, first-stage encode of the source image (mode of the posterior,
        # ddpm.py encode_first_stage / get_first_stage_encoding), the CFG DDIM loop of the headline, first-stage decode.
        from anyedit_b200.autoencoder import AutoencoderKL
        from anyedit_b200.encoders import CLIPTextModel
        B, h = args.batch, args.latent
        px = 8 * h
        if not hasattr(extra_leg, "_stages"):
            torch.manual_seed(91)
            ddconfig = dict(double_z=True, z_channels=4, resolution=256, in_channels=3, out_ch=3, ch=128, ch_mult=[1, 2, 4, 4],
                            num_res_blocks=2, attn_resolutions=[], dropout=0.0)          # the SD-1.x kl-f8 first stage (anydoor.yaml)
            with torch.device(dev):
                vae = AutoencoderKL(ddconfig, embed_dim=4)
                txt = CLIPTextModel({})                                                     # CLIP ViT-L/14 text tower defaults
            D.broadcast_module_(vae, src=0)
            D.broadcast_module_(txt, src=0)
            extra_leg._stages = (vae, txt)
        vae, txt = extra_leg._stages
        gen = torch.Generator().manual_seed(3100 + rank)
        ids = torch.randint(1000, 40000, (B, 77), generator=gen)
        ids[:, 0], ids[:, 20:] = 49406, 49407                                               # <bos> 19 tokens <eos> padding
        null_ids = torch.full((1, 77), 49407, dtype=torch.int64)
        null_ids[0, 0] = 49406
        host = {"img": (torch.rand(B, 3, px, px, generator=gen) * 2 - 1), "ids": ids, "null_ids": null_ids,
                "x_T": torch.randn(B, 4, h, h, generator=gen)}
        host = {k: v.pin_memory() for k, v in host.items()}
        out_host = torch.empty(B, 3, px, px).pin_memory()
        smp = DDIMSampler(model, use_cuda_graph=not args.no_graph)
        scale_factor = 0.18215

        def run(d_):
            c_txt = txt(d_["ids"]).last_hidden_state
            u_txt = txt(d_["null_ids"]).last_hidden_state.expand(B, -1, -1).contiguous()
            c_cat = vae.encode(d_["img"]).mode()
            cond = {"c_concat": [c_cat], "c_crossattn": [c_txt]}
            uncond = {"c_concat": [c_cat], "c_crossattn": [u_txt]}
            z, _ = smp.sample(50, B, (4, h, h), cond, verbose=False, x_T=d_["x_T"], eta=0.0, unconditional_guidance_scale=args.scale,
                              unconditional_conditioning=uncond)
            return vae.decode(z, z_scale=1.0 / scale_factor)

        devt = {k: v.to(dev) for k, v in host.items()}
        resident = lambda: run(devt)
        e2e = lambda: out_host.copy_(run({k: v.to(dev, non_blocking=True) for k, v in host.items()}), non_blocking=True)
        resident()
        n0 = ops.launch_count
        steps = 2
        t_res = timed(resident, steps)
        launches = (ops.launch_count - n0) // steps
        t_e2e = timed(e2e, steps)
        n = B * world * steps
        finite = bool(torch.isfinite(out_host).all())
        return {"metric": "edited images/sec, whole request (CLIP-L text encode x2 + first-stage encode + 50-step CFG DDIM + first-stage decode, "
                          "512x512 pixels in, 512x512 pixels out)",
                "value": n / t_res, "unit": "images/s", "scaling": "weak", "ms_per_step": 1e3 * t_res / steps,
                "e2e": {"value": n / t_e2e, "unit": "images/s", "h2d_bytes_per_step": sum(v.numel() * v.element_size() for v in host.values()),
                        "d2h_bytes_per_step": out_host.numel() * 4},
                "gpu_launches": launches, "output_finite": finite,
                "config": {"workload": f"BASELINE configs[1] requests end to end: {B} RGB source images {px}x{px} + token ids per GPU -> edited RGB "
                                       f"images; kl-f8 AutoencoderKL (ch 128, mult 1-2-4-4) and CLIP ViT-L/14 text tower, random-init weights",
                           "global_batch": B * world, "latent": h, "ddim_steps": 50, "guidance_scale": args.scale}}
    raise ValueError(f"unknown extra leg {leg!r}")


if __name__ == "__main__":
    main()
