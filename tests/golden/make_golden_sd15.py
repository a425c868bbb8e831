#!/usr/bin/env python
"""Golden vectors at the shapes bench.py times, produced by the REAL reference (build container only).

    python tests/golden/make_golden_sd15.py [fwd64] [c1] [c3] [c1_s1] [c3_s1]

Runs the reference's own ``UNetModel`` (ldm/modules/diffusionmodules/openaimodel.py:412-786) and
``DDIMSampler`` (ldm/models/diffusion/ddim.py:55-251) on CPU fp32 at the full SD-1.5 / IP2P geometry:

  sd15_fwd64.npz  one UNet evaluation at a 64x64 latent for the 8 distinct rows (4 uncond + 4 cond) of a
                  CFG batch of 4 edit requests at t = 981 (the first of 50 DDIM steps)
  sd15_c1.npz     BASELINE configs[1] trajectory of ONE request: 64x64 latent, 50 DDIM steps, CFG 7.5, eta 0
                  (final latent + x_inter / pred_x0 every 10 steps)
  sd15_c3.npz     BASELINE configs[3] geometry: 96x96 latent, 100 DDIM steps, CFG 7.5 (plain UNet; the visual
                  expert stream has no reference source)
  sd15_c1_s1.npz, sd15_c3_s1.npz   the same two requests at guidance scale 1.0 (no CFG amplification)

Inputs are regenerated from seeds by ``sd15_inputs.inputs_requests`` (torch CPU generator; the fixtures store float64
checksums of every input so that drift is detected); weights come from ``oracle.weights`` (scheme "torch",
seed 3) -- so the files hold outputs only.  CPU time here (8 cores): fwd64 ~1 min, c1 ~8 min, c3 ~45 min.
"""
import os
import sys
import time

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.abspath(os.path.join(HERE, "..", "..")))
sys.path.insert(0, HERE)

from oracle import ddim_oracle, ref_import, weights  # noqa: E402

from sd15_inputs import SD15, WEIGHT_SCHEME, WEIGHT_SEED, checksum, inputs_requests  # noqa: E402


def build_ref():
    UNetModel, DDIMSamplerCPU, _ = ref_import.load()
    with torch.device("meta"):
        shapes = {k: tuple(v.shape) for k, v in UNetModel(**SD15).state_dict().items()}
    sd = weights.make_state_dict(shapes, WEIGHT_SEED, scheme=WEIGHT_SCHEME)
    net = UNetModel(**SD15).eval()
    net.load_state_dict(sd)
    return net, DDIMSamplerCPU, weights.checksum(sd)


def main():
    which = set(sys.argv[1:]) or {"fwd64", "c1", "c3"}
    torch.set_grad_enabled(False)
    torch.set_num_threads(int(os.environ.get("GOLDEN_THREADS", "6")))
    net, DDIMSamplerCPU, wsum = build_ref()
    sched = ddim_oracle.register_schedule("linear", 1000, 0.00085, 0.012)
    model = ref_import.RefModelShim(net, sched, "hybrid")

    if "fwd64" in which:
        t0 = time.time()
        x_T, c_cat, c_txt, u_txt = inputs_requests(4, 64, 2024)
        x8 = torch.cat([x_T, c_cat], 1)
        t = torch.full((1,), 981, dtype=torch.long)
        eps_u = torch.cat([net(x8[i:i + 1], t, context=u_txt) for i in range(4)])
        eps_c = torch.cat([net(x8[i:i + 1], t, context=c_txt[i:i + 1]) for i in range(4)])
        np.savez(os.path.join(HERE, "sd15_fwd64.npz"), eps_u=eps_u.numpy(), eps_c=eps_c.numpy(), t=981, seed=2024,
                 in_sum=checksum(x_T, c_cat, c_txt, u_txt), wsum=wsum)
        print(f"fwd64 done in {time.time() - t0:.0f} s", flush=True)

    def trajectory(name, h, S, seed, log_every_t, scale=7.5):
        t0 = time.time()
        x_T, c_cat, c_txt, u_txt = inputs_requests(1, h, seed)
        sampler = DDIMSamplerCPU(model)
        out, inter = sampler.sample(S, 1, (4, h, h), {"c_concat": [c_cat], "c_crossattn": [c_txt]}, verbose=False, x_T=x_T,
                                    eta=0.0, unconditional_guidance_scale=scale, log_every_t=log_every_t,
                                    unconditional_conditioning={"c_concat": [c_cat], "c_crossattn": [u_txt]})
        x_inter = torch.stack(inter["x_inter"]).numpy()
        # 96x96: keep the fixture under 1 MB -- no pred_x0, and x_inter (printed along the trajectory, never asserted on) in
        # fp16; the asserted final latent stays fp32
        extra = {"pred_x0": torch.stack(inter["pred_x0"]).numpy()} if h <= 64 else {}
        np.savez(os.path.join(HERE, f"{name}.npz"), final=out.numpy(), x_inter=x_inter if h <= 64 else x_inter.astype(np.float16),
                 S=S, seed=seed, scale=scale, log_every_t=log_every_t, in_sum=checksum(x_T, c_cat, c_txt, u_txt), wsum=wsum, **extra)
        print(f"{name} done in {time.time() - t0:.0f} s", flush=True)

    if "c1" in which:
        trajectory("sd15_c1", 64, 50, 2025, 10)
    if "c3" in which:
        trajectory("sd15_c3", 96, 100, 2026, 20)
    # the same two requests without guidance amplification (scale 1.0: the conditional branch alone, ddim.py:187-188)
    if "c1_s1" in which:
        trajectory("sd15_c1_s1", 64, 50, 2025, 10, scale=1.0)
    if "c3_s1" in which:
        trajectory("sd15_c3_s1", 96, 100, 2026, 20, scale=1.0)


if __name__ == "__main__":
    main()
