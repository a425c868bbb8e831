"""CPU-only tests: host logic of the reference-facing API, state-dict compatibility, the C-ABI
library (loads and exports every declared symbol; no compute without a GPU) and the rank-sharding
helper over a 2-process gloo group."""
import ctypes
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
G = os.path.join(ROOT, "tests", "golden")


def test_library_builds_and_exports_every_declared_symbol():
    from anyedit_b200 import _lib, build
    path = build.build()
    assert os.path.exists(path)
    header = open(os.path.join(ROOT, "include", "anysd_b200.h")).read()
    declared = set(re.findall(r"\b(anysd_[a-z0-9_]+)\s*\(", header))
    declared -= {"anysd_gemm_params", "anysd_attn_params", "anysd_attn_bwd_params", "anysd_expert_attn_params"}
    assert len(declared) >= 15
    lib = ctypes.CDLL(path)
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/anysd_b200.h but not exported"
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    handle = _lib.load()
    assert handle.anysd_version() >= 100


def test_groupnorm_path_choice_is_geometry_only():
    """anysd_groupnorm_resident (a host-side query, no launch): the register-resident GroupNorm kernel serves the maps of at most
    8 x RL pixels (RL = 64 row lanes, 32 when a span is wider than 8 vectors) -- a function of (channels, pixels, groups) only, so the
    kernel an image runs through never depends on the batch."""
    from anyedit_b200 import _lib
    q = _lib.load().anysd_groupnorm_resident
    assert q(1280, 0, 256, 32) == 1 and q(1280, 0, 64, 32) == 1          # 16x16, 8x8 levels
    assert q(2560, 0, 256, 32) == 1 and q(1280, 1280, 256, 32) == 1      # 80 channels per group, as one tensor or as a skip concat
    assert q(640, 320, 64, 32) == 1                                      # 30 channels per group: 15-vector spans, 32 row lanes
    assert q(640, 0, 512, 32) == 1 and q(640, 0, 576, 32) == 0           # 8 x 64 pixels is the limit
    assert q(320, 0, 4096, 32) == 0 and q(640, 0, 1024, 32) == 0         # large maps: statistics from the producer's epilogue
    assert q(1920, 0, 256, 32) == 1 and q(1920, 0, 512, 32) == 0         # 32 row lanes: 256 pixels is the limit
    assert q(324, 0, 64, 32) == 0                                        # channels not divisible into the groups


def test_ddim_hooks_host_logic_duck_typed_model():
    """``score_corrector`` / ``quantize_denoised`` (ddim.py:219-221, 239-240) are host-side hooks between the model call and the update:
    the step then runs the reference's own tensor ops (no kernel), so with a duck-typed model (SURVEY.md 8b1: ``apply_model``,
    ``betas``, ``alphas_cumprod`` ...) the whole loop is checkable on the CPU against a step-by-step restatement of ddim.py:194-251,
    for the eps and the v parameterisation."""
    from anyedit_b200.ddim import DDIMSampler, _cat_cond
    from anyedit_b200.diffusion import make_beta_schedule

    class Duck(torch.nn.Module):
        def __init__(self, parameterization):
            super().__init__()
            acp = np.cumprod(1 - make_beta_schedule("linear", 1000, 0.00085, 0.012))
            self.num_timesteps, self.parameterization, self.device = 1000, parameterization, torch.device("cpu")
            self.betas = torch.tensor(1 - acp / np.append(1., acp[:-1]), dtype=torch.float32)
            self.alphas_cumprod = torch.tensor(acp, dtype=torch.float32)
            self.alphas_cumprod_prev = torch.tensor(np.append(1., acp[:-1]), dtype=torch.float32)

        def apply_model(self, x, t, c):
            ctx = c["c_crossattn"][0].mean(dim=(1, 2)).view(-1, 1, 1, 1)
            return torch.tanh(0.5 * x + ctx) + 0.1 * c["c_concat"][0] * torch.cos(t.float()).view(-1, 1, 1, 1)

    class Bend:
        def modify_score(self, mdl, e_t, x, t, c, gain=1.0):
            return gain * e_t + 0.01 * x

    class FirstStage:
        def __init__(self, step):
            self.step = step

        def quantize(self, z):
            return torch.round(z / self.step) * self.step, None, (None, None, None)

    b, S, scale = 2, 6, 7.5
    g = torch.Generator().manual_seed(0)
    cond = {"c_concat": [torch.randn(b, 4, 8, 8, generator=g)], "c_crossattn": [torch.randn(b, 5, 16, generator=g)]}
    uncond = {"c_concat": [cond["c_concat"][0]], "c_crossattn": [torch.randn(b, 5, 16, generator=g)]}
    xT = torch.randn(b, 4, 8, 8, generator=g)
    c_in = _cat_cond(uncond, cond)
    kw = dict(verbose=False, x_T=xT, eta=0.0, unconditional_guidance_scale=scale, unconditional_conditioning=uncond)
    for par in ("eps", "v"):
        model = Duck(par)
        model.first_stage_model = FirstStage(0.05)
        smp = DDIMSampler(model, use_cuda_graph=False)
        corr = Bend() if par == "eps" else None                  # the reference asserts eps for a corrector (ddim.py:220)
        got, inter = smp.sample(S, b, (4, 8, 8), cond, score_corrector=corr, corrector_kwargs={"gain": 0.9}, quantize_x0=True,
                                log_every_t=1, **kw)
        T = len(smp.ddim_timesteps)
        x = xT.clone()
        for i, step in enumerate(np.flip(smp.ddim_timesteps)):
            index = T - i - 1
            out = model.apply_model(torch.cat([x, x]), torch.full((2 * b,), int(step), dtype=torch.long), c_in)
            out = out[:b] + scale * (out[b:] - out[:b])
            a_t, a_prev = float(smp.ddim_alphas[index]), float(smp.ddim_alphas_prev[index])
            if par == "v":
                sa, s1 = float(model.alphas_cumprod[int(step)]) ** 0.5, (1 - float(model.alphas_cumprod[int(step)])) ** 0.5
                e_t, pred = sa * out + s1 * x, sa * x - s1 * out
            else:
                e_t = 0.9 * out + 0.01 * x
                pred = (x - float(smp.ddim_sqrt_one_minus_alphas[index]) * e_t) / (a_t ** 0.5)
            pred = torch.round(pred / 0.05) * 0.05
            x = (a_prev ** 0.5) * pred + ((1. - a_prev) ** 0.5) * e_t
        assert float((got - x).norm() / x.norm()) < 1e-5, par
        for p0 in inter["pred_x0"][1:]:
            assert float((p0 / 0.05 - torch.round(p0 / 0.05)).abs().max()) < 1e-3
    with pytest.raises(AssertionError):                          # 'not implemented' in the reference too
        DDIMSampler(Duck("v"), use_cuda_graph=False).sample(S, b, (4, 8, 8), cond, score_corrector=Bend(), **kw)


def test_bench_reference_arm_contract(tmp_path):
    """``bench.py --impl reference`` (the driver's reference arm): rank 0 prints ONE JSON line with the contract's keys, timed on the
    reference's own CPU implementation (``oracle/_ref`` staged sources when present, the restatement otherwise); any other rank exits
    0 without output.  Run on a shrunken workload (8x8 latent, 4 DDIM steps) so that the CPU suite stays short."""
    import subprocess
    import sys
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--latent", "8", "--ddim-steps", "4",
           "--steps", "1", "--warmup", "1"]
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "LOCAL_RANK", "WORLD_SIZE")}
    other = subprocess.run(cmd, env={**env, "RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"}, capture_output=True, text=True, timeout=600)
    assert other.returncode == 0 and other.stdout.strip() == ""
    r0 = subprocess.run(cmd, env={**env, "RANK": "0", "LOCAL_RANK": "0", "WORLD_SIZE": "2"}, capture_output=True, text=True, timeout=900)
    assert r0.returncode == 0, r0.stderr[-2000:]
    lines = [ln for ln in r0.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["n_gpus"] == 2 and d["steps"] == 1 and d["warmup"] == 1
    assert d["unit"] == "images/s" and d["higher_is_better"] is True and d["value"] > 0 and d["ms_per_step"] > 0
    assert d["metric"].startswith("edited images/sec") and d["vs_baseline"] is None and d["data"] == "synthetic"
    assert d["config"]["workload"] and d["config"]["latent"] == 8 and d["config"]["ddim_steps"] == 4
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["sample"] and cb["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    from oracle import ref_import
    assert cb["kind"] == ("reference" if ref_import.available() else "port")


def test_bench_dump_outputs(tmp_path, monkeypatch):
    """``bench.py --dump-outputs``: the samples and every logged intermediate of the final sampler call as float32 .npy, whole
    while they fit the byte budget, else each cut to the same seeded sample of its elements, identically from call to call."""
    import bench
    gen = torch.Generator().manual_seed(0)
    lat = lambda: torch.randn(2, 4, 8, 8, generator=gen, dtype=torch.float64)
    last = {"samples": lat(), "intermediates": {"x_inter": [lat(), lat()], "pred_x0": [lat(), lat()]}}
    names = {"samples", "x_inter_0", "x_inter_1", "pred_x0_0", "pred_x0_1"}
    bench.dump_outputs(str(tmp_path / "full"), last)
    assert {f[:-4] for f in os.listdir(tmp_path / "full")} == names
    got = np.load(tmp_path / "full" / "samples.npy")
    assert got.dtype == np.float32 and np.array_equal(got, last["samples"].float().numpy())
    assert np.array_equal(np.load(tmp_path / "full" / "pred_x0_1.npy"), last["intermediates"]["pred_x0"][1].float().numpy())
    monkeypatch.setattr(bench, "DUMP_BYTES", 5 * 4096 + 5 * 4 * 256)   # room for half of each array
    for d in ("cut_a", "cut_b"):
        bench.dump_outputs(str(tmp_path / d), last)
    assert sum(os.path.getsize(tmp_path / "cut_a" / f) for f in os.listdir(tmp_path / "cut_a")) <= bench.DUMP_BYTES
    for n in names:
        a, b = np.load(tmp_path / "cut_a" / f"{n}.npy"), np.load(tmp_path / "cut_b" / f"{n}.npy")
        assert a.dtype == np.float32 and a.shape == (256,) and np.array_equal(a, b)
        assert np.isin(a, np.load(tmp_path / "full" / f"{n}.npy")).all()


def test_no_cpu_fallback():
    """Without a CUDA device the product path must fail loudly, never fall back."""
    from anyedit_b200 import ops
    from anyedit_b200.unet import UNetModel
    meta = json.load(open(os.path.join(G, "tiny_b_keys.json")))
    net = UNetModel(**meta["config"])
    with pytest.raises(RuntimeError):
        net(torch.zeros(1, 4, 8, 8), torch.zeros(1, dtype=torch.long), context=torch.zeros(1, 5, 96),
            y=torch.zeros(1, dtype=torch.long))
    with pytest.raises(Exception):
        ops.layernorm(torch.zeros(4, 64, dtype=torch.float16), torch.ones(64), torch.zeros(64),
                      torch.zeros(4, 64, dtype=torch.float16))
    # and the product never imports the oracle
    for root, _, files in os.walk(os.path.join(ROOT, "anyedit_b200")):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(root, f)).read()
                assert "import oracle" not in src and "from oracle" not in src, f


@pytest.mark.parametrize("name", ["tiny_a", "tiny_b", "sd15_meta", "anydoor_meta"])
def test_state_dict_layout_matches_reference(name):
    """Same keys and shapes as the reference UNetModel (686 tensors for SD-1.5; SURVEY.md 8b)."""
    from anyedit_b200.unet import UNetModel
    meta_dev = name.endswith("_meta")
    meta = json.load(open(os.path.join(G, f"{name.replace('_meta', '')}_keys.json")))
    if meta_dev:
        with torch.device("meta"):
            net = UNetModel(**meta["config"])
    else:
        net = UNetModel(**meta["config"])
    sd = net.state_dict()
    assert set(sd) == set(meta["keys"])
    assert all(list(sd[k].shape) == meta["keys"][k] for k in sd)
    assert sum(v.numel() for v in sd.values()) == meta["n_params"]
    if not meta_dev:
        # the reference's zero-init quirk is preserved (openaimodel.py:228-230, 729; attention.py:312-318)
        assert float(sd["out.2.weight"].abs().sum()) == 0.0
        assert float(sd["input_blocks.1.0.out_layers.3.weight"].abs().sum()) == 0.0
        assert float(sd["input_blocks.1.1.proj_out.weight"].abs().sum()) == 0.0


def test_constructor_contract():
    from anyedit_b200.unet import UNetModel
    base = dict(image_size=8, in_channels=4, model_channels=32, out_channels=4, num_res_blocks=1,
                attention_resolutions=[1], channel_mult=[1], num_heads=2, use_spatial_transformer=True, context_dim=32)
    UNetModel(**base)
    with pytest.raises(AssertionError):
        UNetModel(**{**base, "context_dim": None})
    with pytest.raises(AssertionError):
        UNetModel(**{**base, "num_heads": -1})
    with pytest.raises(ValueError):
        UNetModel(**{**base, "num_res_blocks": [1, 2]})
    with pytest.raises(TypeError):
        UNetModel(**base, not_a_kwarg=1)
    with pytest.raises(NotImplementedError):
        UNetModel(**{**base, "use_scale_shift_norm": True})
    net = UNetModel(**{**base, "num_classes": 3})
    with pytest.raises(AssertionError):   # y iff class-conditional (openaimodel.py:763-765)
        net(torch.zeros(1, 4, 8, 8), torch.zeros(1, dtype=torch.long), context=torch.zeros(1, 2, 32))


def test_schedule_bit_exact_through_product_api():
    from anyedit_b200 import ddim
    from anyedit_b200.diffusion import LatentDenoiser, make_beta_schedule
    g = np.load(os.path.join(G, "schedule.npz"))
    assert np.array_equal(make_beta_schedule("linear", 1000, 0.00085, 0.012), g["betas"])

    class Dummy(torch.nn.Module):
        def forward(self, x, t, context=None, y=None):
            return x[:, :4] * 0.5

    model = LatentDenoiser(Dummy(), "hybrid")
    assert np.array_equal(model.alphas_cumprod.numpy(), g["alphas_cumprod"].astype(np.float32))
    s = ddim.DDIMSampler(model)
    for S in (20, 50, 100):
        for eta in (0.0, 0.5):
            s.make_schedule(S, ddim_eta=eta, verbose=False)
            tag = f"{S}_{int(eta * 10)}"
            assert np.array_equal(s.ddim_timesteps, g[f"ts_{S}"])
            assert np.array_equal(np.asarray(s.ddim_alphas, dtype=np.float32), g[f"alphas_{tag}"])
            assert np.array_equal(np.asarray(s.ddim_alphas_prev, dtype=np.float64), g[f"alphas_prev_{tag}"])
            assert np.array_equal(np.asarray(s.ddim_sigmas, dtype=np.float64), g[f"sigmas_{tag}"])
            assert tuple(s.ddim_coef_host.shape) == (S, 7)        # 5 DDIM scalars + sqrt(acp[t]), sqrt(1 - acp[t]) for v-param
    assert np.array_equal(ddim.make_ddim_timesteps("quad", 20, 1000, verbose=False), g["ts_quad_20"])
    with pytest.raises(NotImplementedError):
        ddim.make_ddim_timesteps("nope", 20, 1000, verbose=False)


def test_conditioning_mux_matches_oracle():
    """DiffusionWrapper.forward key handling (ddpm.py:1332-1363) on CPU with a recording model."""
    from anyedit_b200.diffusion import LatentDenoiser
    from oracle import ddim_oracle

    class Rec(torch.nn.Module):
        def forward(self, x, t, context=None, y=None):
            self.seen = (x, context, y)
            return x[:, :4]

    x, cc, ca = torch.randn(2, 4, 8, 8), torch.randn(2, 4, 8, 8), torch.randn(2, 7, 16)
    t = torch.tensor([3, 4])
    adm = torch.tensor([1, 2])
    for key, cond in (("hybrid", {"c_concat": [cc], "c_crossattn": [ca]}),
                      ("crossattn", {"c_crossattn": [ca, ca]}), ("crossattn", ca), ("crossattn", [ca]),
                      ("concat", {"c_concat": [cc]}),
                      ("hybrid-adm", {"c_concat": [cc], "c_crossattn": [ca], "c_adm": adm}),
                      ("crossattn-adm", {"c_crossattn": [ca], "c_adm": adm})):
        rec = Rec()
        LatentDenoiser(rec, key).apply_model(x, t, cond)
        seen = {}
        ddim_oracle.apply_model(lambda a, b, context=None, y=None: seen.update(x=a, c=context, y=y) or a[:, :4],
                                key, x, t, cond)
        assert torch.equal(rec.seen[0], seen["x"])
        assert (rec.seen[1] is None) == (seen["c"] is None) and (seen["c"] is None or torch.equal(rec.seen[1], seen["c"]))
        assert (rec.seen[2] is None) == (seen["y"] is None)


def test_instantiate_from_config_aliases():
    from anyedit_b200.diffusion import instantiate_from_config
    cfg = {"target": "anyedit_b200.ldm.modules.diffusionmodules.openaimodel.UNetModel",
           "params": dict(image_size=8, in_channels=4, model_channels=32, out_channels=4, num_res_blocks=1,
                          attention_resolutions=[1], channel_mult=[1], num_heads=2, use_spatial_transformer=True,
                          context_dim=32)}
    net = instantiate_from_config(cfg)
    from anyedit_b200.unet import UNetModel
    assert isinstance(net, UNetModel)
    from anyedit_b200.ldm.models.diffusion.ddim import DDIMSampler  # noqa: F401
    from anyedit_b200.ldm.models.diffusion.ddpm import DiffusionWrapper, LatentDiffusion  # noqa: F401


def test_request_sharding_two_rank_gloo(tmp_path):
    """Edit requests shard over ranks with no data-path collective (SURVEY.md 8e): 2 gloo ranks on CPU
    each take their contiguous slice; the concatenation equals the unsharded batch; weights are
    broadcast once from rank 0."""
    script = tmp_path / "w.py"
    script.write_text(
        "import os, sys, torch, torch.distributed as dist\n"
        f"sys.path.insert(0, {ROOT!r})\n"
        "from anyedit_b200 import distributed as D\n"
        "dist.init_process_group('gloo')\n"
        "r, w = dist.get_rank(), dist.get_world_size()\n"
        "lo, hi = D.shard_range(7, r, w)\n"
        "m = torch.nn.Linear(4, 4)\n"
        "torch.manual_seed(r); torch.nn.init.normal_(m.weight)\n"
        "D.broadcast_module_(m, src=0)\n"
        "gathered = [None] * w\n"
        "dist.all_gather_object(gathered, (lo, hi, float(m.weight.sum())))\n"
        "if r == 0:\n"
        "    assert [g[:2] for g in gathered] == [(0, 4), (4, 7)], gathered\n"
        "    assert gathered[0][2] == gathered[1][2]\n"
        "    print('OK')\n"
        "dist.destroy_process_group()\n")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29533", str(script)],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "OK" in r.stdout, r.stdout + r.stderr


def test_gradient_allreduce_two_rank_gloo(tmp_path):
    """Training path (SURVEY.md 8e / a24): the only data-path collective is the all-reduce of the trainables' gradients;
    2 gloo ranks on CPU: every rank ends with the rank-sum, the helper reports the world size for the 1/world fold."""
    script = tmp_path / "g.py"
    script.write_text(
        "import os, sys, torch, torch.distributed as dist\n"
        f"sys.path.insert(0, {ROOT!r})\n"
        "from anyedit_b200 import distributed as D\n"
        "dist.init_process_group('gloo')\n"
        "r = dist.get_rank()\n"
        "g = [torch.full((5, 3), float(r + 1)), torch.arange(4.0) * (r + 1), None]\n"
        "w = D.allreduce_sum_(g)\n"
        "assert w == 2 and torch.equal(g[0], torch.full((5, 3), 3.0)) and torch.equal(g[1], torch.arange(4.0) * 3)\n"
        "# bucketed form used by AdapterTrainer.step: regions of ONE flat buffer reduced as they complete, waited at the end\n"
        "flat = torch.arange(10.0) * (r + 1)\n"
        "works = [D.allreduce_sum_async(flat[6:10]), D.allreduce_sum_async(flat[0:6])]\n"
        "assert D.world_size() == 2 and all(x is not None for x in works)\n"
        "for x in works: x.wait()\n"
        "assert torch.equal(flat, torch.arange(10.0) * 3)\n"
        "if r == 0: print('OK')\n"
        "dist.destroy_process_group()\n")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29534", str(script)],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "OK" in r.stdout, r.stdout + r.stderr


def test_training_host_logic():
    """a24 host side: conditioning dropout == the restated train.py:651-669; the dX weight packs are the rotated /
    transposed weights (checked against torch autograd on CPU, fp32); no CPU fallback for the step itself."""
    import torch.nn.functional as F
    from anyedit_b200 import training as T
    from oracle import train_oracle
    gen = torch.Generator().manual_seed(3)
    text, null, img = torch.randn(6, 7, 16, generator=gen), torch.randn(1, 7, 16, generator=gen), torch.randn(6, 4, 8, 8, generator=gen)
    p = torch.tensor([0.01, 0.06, 0.09, 0.12, 0.2, 0.9])
    a, b = T.conditioning_dropout(text, null, img, p, 0.05)
    ra, rb = train_oracle.conditioning_dropout(text, null, img, p, 0.05)
    assert torch.equal(a, ra) and torch.equal(b, rb)
    assert torch.equal(a[0], null[0]) and torch.equal(a[2], null[0]) and torch.equal(a[3], text[3])      # text dropped for p < 2P
    assert torch.equal(b[0], img[0]) and float(b[1].abs().max()) == 0.0 and float(b[3].abs().max()) == 0.0 and torch.equal(b[4], img[4])
    # conv: dX = conv3x3(dY, pack) with pack[ci, (a, b, co)] = w[co, ci, 2-a, 2-b]
    w = torch.randn(5, 3, 3, 3, generator=gen)
    x = torch.randn(2, 3, 6, 7, generator=gen, requires_grad=True)
    dy = torch.randn(2, 5, 6, 7, generator=gen)
    F.conv2d(x, w, padding=1).backward(dy)
    pack = T.pack_conv3_dx(w, "cpu").float().reshape(3, 3, 3, 5).permute(0, 3, 1, 2)       # -> OIHW of the dX conv
    assert torch.allclose(F.conv2d(dy, pack, padding=1), x.grad, atol=2e-2)                 # pack is fp16-rounded
    wl = torch.randn(9, 4, generator=gen)
    assert torch.allclose(T.pack_linear_dx(wl, "cpu").float(), wl.t().half().float())
    # the step needs CUDA tensors
    from anyedit_b200.anysd import MoE
    from anyedit_b200.unet import UNetModel
    meta = json.load(open(os.path.join(G, "tiny_a_keys.json")))
    tr = T.AdapterTrainer(MoE(UNetModel(**meta["config"]), None, expert_num=2, num_tasks=3))
    z = torch.zeros(1, 4, 16, 16)
    with pytest.raises(RuntimeError):
        tr.loss_and_grads(z, z, torch.zeros(1, dtype=torch.long), z, torch.zeros(1, 7, 64))


def test_cfg_halves_sharing_decision(monkeypatch):
    """Host logic of the shared-CFG-halves optimisation (ddim.py:190-210 batch construction): only when the two halves
    can differ in nothing but the cross-attention context."""
    from anyedit_b200.ddim import _halves_share_prefix
    monkeypatch.delenv("ANYSD_SHARE_CFG", raising=False)
    cc, txt, utxt = torch.randn(2, 4, 8, 8), torch.randn(2, 7, 16), torch.randn(2, 7, 16)
    c = {"c_concat": [cc], "c_crossattn": [txt]}
    assert _halves_share_prefix({"c_concat": [cc], "c_crossattn": [utxt]}, c)                      # same tensor object
    assert _halves_share_prefix({"c_concat": [cc.clone()], "c_crossattn": [utxt]}, c)              # equal values
    assert not _halves_share_prefix({"c_concat": [torch.zeros_like(cc)], "c_crossattn": [utxt]}, c)  # IP2P-style zero image
    assert not _halves_share_prefix({"c_concat": [cc], "c_crossattn": [utxt], "c_adm": torch.zeros(2)},
                                    {**c, "c_adm": torch.ones(2)})
    assert not _halves_share_prefix([utxt], [txt])                                                 # list conditioning: no claim
    assert _halves_share_prefix({"c_crossattn": [utxt]}, {"c_crossattn": [txt]})                   # pure cross-attention model
    monkeypatch.setenv("ANYSD_SHARE_CFG", "0")
    assert not _halves_share_prefix({"c_concat": [cc], "c_crossattn": [utxt]}, c)


def _toy_eps(x, t):
    return 0.3 * torch.sin(1.7 * x) + 0.05 * torch.cos(x * 0.5 + t.float().reshape(-1, 1, 1, 1) * 0.01)


def test_plms_plan_and_rows_match_oracle_on_cpu():
    """Host logic of anyedit_b200.plms (no GPU): the call plan + coefficient rows, pushed through a torch emulation of
    ``cfg_plms_kernel``'s arithmetic, reproduce oracle/plms_oracle.py (pinned to the reference PLMSSampler) bit for bit."""
    import numpy as np
    from anyedit_b200.ddim import make_ddim_sampling_parameters, make_ddim_timesteps, step_coefficients
    from anyedit_b200.plms import plms_plan
    from oracle import ddim_oracle, plms_oracle
    sched = ddim_oracle.register_schedule("linear", 1000, 0.00085, 0.012)
    x_T = torch.randn(2, 4, 8, 8, generator=torch.Generator().manual_seed(3))
    for S in (5, 10):
        ts = make_ddim_timesteps("uniform", S, 1000, verbose=False)
        sig, a, ap = make_ddim_sampling_parameters(sched["alphas_cumprod"], ts, 0.0, verbose=False)
        ddim = [step_coefficients(a, ap, sig, np.sqrt(1.0 - a), i)[:4] for i in range(S)]
        hist = [torch.zeros_like(x_T) for _ in range(3)]
        img, x_tmp = x_T, None
        f = lambda v: torch.tensor(v, dtype=torch.float32)
        for call in plms_plan(np.flip(ts)):
            xm = x_tmp if call["use_tmp"] else img
            e = _toy_eps(xm, torch.full((2,), call["t"]))
            c0, c1, c2, c3, den = (f(v) for v in call["comb"])
            ep = (((c0 * e - c1 * hist[0]) + c2 * hist[1]) - c3 * hist[2]) / den
            somat, sq_at, sq_ap, dr = (f(v) for v in ddim[call["index"]])
            pred = (img - somat * ep) / sq_at
            out = sq_ap * pred + dr * ep
            if call["push"]:
                hist = [e, hist[0], hist[1]]
            if call["final"]:
                img, x_tmp = out, None
            else:
                x_tmp = out
        ref, _ = plms_oracle.plms_sample(lambda x, t, c: _toy_eps(x, t), sched, S, x_T, None)
        assert torch.equal(img, ref), S


def test_dpmpp_tables_match_oracle_on_cpu():
    """Host logic of anyedit_b200.dpm_solver (no GPU): the schedule tables + a torch emulation of ``cfg_dpmpp_kernel``
    reproduce oracle/dpm_oracle.py (pinned to the reference DPMSolverSampler), S < 15 (order-1 final step) and S >= 15."""
    from anyedit_b200.dpm_solver import NoiseScheduleVP, dpmpp_2m_tables
    from oracle import ddim_oracle, dpm_oracle
    sched = ddim_oracle.register_schedule("linear", 1000, 0.00085, 0.012)
    x_T = torch.randn(2, 4, 8, 8, generator=torch.Generator().manual_seed(4))
    ns = NoiseScheduleVP("discrete", alphas_cumprod=sched["alphas_cumprod"])
    for S in (10, 20):
        t_model, coef = dpmpp_2m_tables(ns, S)
        x, mp = x_T, torch.zeros_like(x_T)
        for k in range(S):
            e = _toy_eps(x, torch.full((2,), t_model[k]))
            sig, alp, ratio, c, half_c, inv_r0 = coef[k]
            m = (x - sig * e) / alp
            x = (ratio * x - c * m) - half_c * (inv_r0 * (m - mp))
            mp = m
        ref = dpm_oracle.dpm_solver_pp_2m(lambda x_, t, c_: _toy_eps(x_, t), sched["alphas_cumprod"], S, x_T, None)
        err = float((x - ref).norm() / ref.norm())
        assert err < 2e-6, (S, err)
