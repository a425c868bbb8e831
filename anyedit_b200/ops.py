"""Torch-tensor wrappers over the C ABI (include/anysd_b200.h).

PyTorch is plumbing here: device memory, the current CUDA stream, nothing else.  Every function
launches hand-written sm_100a kernels from ``libanysd_b200.so`` on ``torch.cuda.current_stream()``
and raises on failure.  Tensors are NHWC / token-major fp16 unless stated.
"""
import os
import ctypes as C

import torch

from . import _lib
from ._lib import F16, F32, I64, AttnParams, GemmParams

_DT = {torch.float32: F32, torch.float16: F16, torch.int64: I64}

# Incremented by every kernel launch issued through this module (bench.py reports it).
launch_count = 0


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise _lib.AnysdError("anysd_b200 ops need CUDA tensors; there is no CPU fallback")


def _count(n=1):
    global launch_count
    launch_count += n


# Optional per-launch tracing for bench.py's roofline leg: when ``trace`` is a list, the tensor-core
# wrappers bracket their launch with CUDA events on the launching stream and append
# (kind, algorithmic_flops, start_event, end_event, tag).  None (default) adds no work.
trace = None


class _Traced:
    def __init__(self, kind, flops, tag=""):
        self.kind, self.flops, self.tag = kind, flops, tag

    def __enter__(self):
        if trace is not None:
            self.e0 = torch.cuda.Event(enable_timing=True)
            self.e1 = torch.cuda.Event(enable_timing=True)
            self.e0.record()
        return self

    def __exit__(self, *exc):
        if trace is not None:
            self.e1.record()
            trace.append((self.kind, self.flops, self.e0, self.e1, self.tag))
        return False


def device_info():
    lib = _lib.load()
    a, b, c = C.c_int(), C.c_int(), C.c_int()
    _lib.check(lib.anysd_device_info(C.byref(a), C.byref(b), C.byref(c)), "device_info")
    return a.value, b.value, c.value


def nchw_to_nhwc(src, dst, c_off=0):
    """src [N,C,H,W] f32|f16 contiguous -> dst[..., c_off:c_off+C] of NHWC fp16 [N,H,W,dstC]."""
    _cuda(src, dst)
    N, Cc, H, W = src.shape
    assert src.is_contiguous() and dst.is_contiguous() and dst.dtype == torch.float16
    _lib.check(_lib.load().anysd_nchw_to_nhwc_f16(_ptr(src), _DT[src.dtype], _ptr(dst), N, Cc, H, W,
                                                  dst.shape[-1], c_off, _stream()), "nchw_to_nhwc")
    _count()


def add_nchw_into_nhwc(src, dst):
    """dst NHWC fp16 [N,H,W,C] += src NCHW f32|f16 [N,C,H,W] (ControlNet residuals)."""
    _cuda(src, dst)
    N, Cc, H, W = src.shape
    assert tuple(dst.shape) == (N, H, W, Cc) and src.is_contiguous() and dst.is_contiguous()
    _lib.check(_lib.load().anysd_add_nchw_into_nhwc_f16(_ptr(src), _DT[src.dtype], _ptr(dst), N, Cc, H, W, _stream()),
               "add_nchw_into_nhwc")
    _count()


def nhwc_to_nchw(src, dst):
    """src NHWC f16|f32 [N,H,W,Cs] (first C channels used) -> dst NCHW f32|f16 [N,C,H,W]."""
    _cuda(src, dst)
    N, Cc, H, W = dst.shape
    assert src.is_contiguous() and dst.is_contiguous() and src.shape[-1] >= Cc
    _lib.check(_lib.load().anysd_nhwc_to_nchw(_ptr(src), _DT[src.dtype], src.shape[-1], _ptr(dst), _DT[dst.dtype], N, Cc,
                                              H, W, _stream()), "nhwc_to_nchw")
    _count()


def concat_channels(a, b, dst):
    _cuda(a, b, dst)
    rows = a.numel() // a.shape[-1]
    _lib.check(_lib.load().anysd_concat_channels_f16(_ptr(a), a.shape[-1], _ptr(b), b.shape[-1], _ptr(dst), rows,
                                                     _stream()), "concat_channels")
    _count()


def cast_f16(src, dst):
    _cuda(src, dst)
    assert src.dtype == torch.float32 and dst.dtype == torch.float16 and src.is_contiguous()
    _lib.check(_lib.load().anysd_cast_f32_to_f16(_ptr(src), _ptr(dst), src.numel(), _stream()), "cast")
    _count()


def timestep_embedding(t, out, max_period=10000.0):
    """t [N] int64|f32 -> out fp16 [N, dim] (util.py:154-174)."""
    _cuda(t, out)
    if t.dtype not in (torch.int64, torch.float32):
        t = t.float() if t.is_floating_point() else t.long()
    _lib.check(_lib.load().anysd_timestep_embedding_f16(_ptr(t), _DT[t.dtype], _ptr(out), out.shape[0], out.shape[1],
                                                        float(max_period), _stream()), "timestep_embedding")
    _count()


def emb_finalize(emb_lin, silu_out, table=None, idx=None, emb_out=None):
    _cuda(emb_lin, silu_out)
    N, D = emb_lin.shape
    rows = table.shape[0] if table is not None else 0
    _lib.check(_lib.load().anysd_emb_finalize(_ptr(emb_lin), _ptr(table), _ptr(idx), rows, _ptr(emb_out),
                                              _ptr(silu_out), N, D, _stream()), "emb_finalize")
    _count()


def router_gate(table, idx, W, bias, gate):
    """gate[b, l, :] = softmax(W[l] @ table[idx[b]] + bias[l]); W fp16 [L, E, D], gate fp32 [B, L, E]."""
    _cuda(table, idx, W, bias, gate)
    L, E, D = W.shape
    _lib.check(_lib.load().anysd_router_gate_f32(_ptr(table), _ptr(idx), table.shape[0], _ptr(W), _ptr(bias),
                                                 _ptr(gate), gate.shape[0], L, E, D, _stream()), "router_gate")
    _count()


_GN_FUSED = os.environ.get("ANYSD_GN_FUSED", "1")[:1] != "0"     # one cooperative launch (default) or stats + apply


def groupnorm_workspace(N, G=32, C=0, device="cuda"):
    nbytes = _lib.load().anysd_groupnorm_workspace_bytes(N, G, C)
    return torch.zeros(nbytes // 4, dtype=torch.float32, device=device)   # completion counters start at zero


def groupnorm(x1, gamma, beta, y, N, HW, eps, silu, ws, x2=None, G=32, stats=None):
    """GroupNorm(+SiLU).  ``stats`` (GnStats of x1, from the contraction(s) that produced it): only the streaming apply pass
    runs; otherwise the statistics are computed here."""
    _cuda(x1, y, ws)
    if stats is not None and x2 is None and stats.S * 32 == HW:
        Cc = x1.shape[-1]
        parts = stats.parts
        assert sum(c for _, c in parts) == Cc and len(parts) <= 2 and all(b.shape[0] >= N for b, _ in parts)
        s2 = parts[1][0] if len(parts) == 2 else None
        with _Traced("groupnorm", 0.0, f"N={N} HW={HW} C={Cc} epilogue-stats"):
            _lib.check(_lib.load().anysd_groupnorm_apply_nhwc_f16(_ptr(x1), Cc, _ptr(parts[0][0]), parts[0][1], _ptr(s2), stats.S, _ptr(gamma),
                                                              _ptr(beta), _ptr(y), N, HW, G, float(eps), int(bool(silu)), _ptr(ws),
                                                              ws.numel() * 4, _stream()), "groupnorm_apply")
        _count(2)
        return
    C1 = x1.shape[-1]
    C2 = x2.shape[-1] if x2 is not None else 0
    with _Traced("groupnorm", 0.0, f"N={N} HW={HW} C={C1}+{C2}"):
        _lib.check(_lib.load().anysd_groupnorm_nhwc_f16(_ptr(x1), C1, _ptr(x2), C2, _ptr(gamma), _ptr(beta), _ptr(y), N,
                                                        HW, G, float(eps), int(bool(silu)), _ptr(ws), ws.numel() * 4,
                                                        _stream()), "groupnorm")
    _count(1 if _GN_FUSED else 2)


def layernorm(x, gamma, beta, y, eps=1e-5):
    _cuda(x, y)
    Cc = x.shape[-1]
    M = x.numel() // Cc
    with _Traced("layernorm", 0.0, f"M={M} C={Cc}"):
        _lib.check(_lib.load().anysd_layernorm_f16(_ptr(x), _ptr(gamma), _ptr(beta), _ptr(y), M, Cc, float(eps),
                                                   _stream()), "layernorm")
    _count()


_GN_EPILOGUE = os.environ.get("ANYSD_GN_EPILOGUE", "1")[:1] != "0"      # GroupNorm statistics from the producer's epilogue


GN_EPILOGUE_MIN_ROWS = 1024          # pixels per image from which the producer's epilogue emits the statistics (see _want_stats)


class GnStats:
    """Epilogue statistics of one activation tensor: ``parts`` = [(fp32 [images, S, C_i, 2], C_i), ...] in channel order
    (two parts for a channel concat), ``S`` = slabs per image."""
    __slots__ = ("parts", "S")

    def __init__(self, parts, S):
        self.parts, self.S = parts, S


def _want_stats(p, images, dev, reuse=None):
    """Allocate the statistics buffer when the launch can fill it (anysd_gemm_stats_slabs); returns GnStats or None.
    ``reuse``: a GnStats of the same geometry whose buffer is refilled (persistent outputs read by a captured graph)."""
    # [measured, tests/diag_gn.py, batch 16] finalize + streaming apply vs the one-launch statistics + apply kernel:
    # 31 vs 42 us (64x64 map, 320 ch), 21 vs 29 us (32x32, 640 ch), 69 vs 103 us (64x64, 960 ch) -- but 23 vs 19 us at 16x16
    # and 15 vs 14 us at 8x8, where two launches cost more than the statistics pass they replace: maps of >= 1024 pixels only
    # (below that the register-resident kernel -- anysd_groupnorm_resident -- reads x once and needs no statistics)
    if not _GN_EPILOGUE or p.rows_per_batch < GN_EPILOGUE_MIN_ROWS:
        return None
    S = _lib.load().anysd_gemm_stats_slabs(C.byref(p))
    if S <= 0:
        return None
    slots = (images + 7) // 8 * 8            # >= the conv's images-per-tile rounding (at most 4 images share a 128-row tile)
    if isinstance(reuse, GnStats) and reuse.S == S and tuple(reuse.parts[0][0].shape) == (slots, S, p.N, 2):
        buf = reuse.parts[0][0]
    else:
        reuse = None
        buf = torch.empty(slots, S, p.N, 2, dtype=torch.float32, device=dev)
    p.stats, p.stats_images = buf.data_ptr(), slots
    return reuse if reuse is not None else GnStats([(buf, p.N)], S)


_SPLITK = os.environ.get("ANYSD_GEMM_SPLITK", "1")[:1] != "0"
_splitk_counters = {}


def _want_splitk(p, dev):
    """Scratch for split-K when the schedule wants it (few output tiles, long K): fp32 partial tiles + the per-device arrival
    counters (zeroed once; every launch re-arms them).  Returns the scratch tensor (kept alive by the caller's frame)."""
    if not _SPLITK:
        return None
    need = _lib.load().anysd_gemm_splitk_workspace_bytes(C.byref(p))
    if need == 0:
        return None
    cnt = _splitk_counters.get(dev)
    if cnt is None:
        cnt = _splitk_counters[dev] = torch.zeros(16384, dtype=torch.int32, device=dev)
    ws = torch.empty(need // 4, dtype=torch.float32, device=dev)
    p.splitk_workspace, p.splitk_workspace_bytes = ws.data_ptr(), need
    p.splitk_counters, p.splitk_counters_bytes = cnt.data_ptr(), cnt.numel() * 4
    return ws


SCHEDULE_KEYS = ("kernel", "ctas", "bn", "splits", "ext", "ln")


def _fill_schedule(p, schedule):
    """schedule.update(anysd_gemm_schedule(p)): the kernel (0 mma.sync, 1 tcgen05, 2 persistent tcgen05) and, for the
    persistent kernel, the CTAs per tile, the tile width, the K split and the epilogue variant these exact params launch."""
    vals = [C.c_int() for _ in SCHEDULE_KEYS]
    _lib.check(_lib.load().anysd_gemm_schedule(C.byref(p), *[C.byref(v) for v in vals]), "gemm_schedule")
    schedule.update(zip(SCHEDULE_KEYS, (v.value for v in vals)))


def row_stats_buffer(M, C, device):
    """fp32 [C / 64, M, 2]: the per-row moments a contraction's epilogue writes for the LayerNorm folded into its consumer."""
    assert C % 64 == 0
    return torch.empty(C // 64, M, 2, dtype=torch.float32, device=device)


def gemm(A, W, out, bias=None, rowadd=None, rows_per_batch=0, residual=None, act=0, M=None, K=None, lda=None,
         N=None, ldw=None, ld_rowadd=None, stats_images=0, row_stats=None, ln=None, schedule=None):
    """out[M, N'] = epilogue(A[M, K] @ W[N, K]^T); see anysd_gemm_params.
    ``stats_images`` > 0 (with ``rows_per_batch`` = rows of one image): also produce the GroupNorm statistics of ``out`` in the
    epilogue; returns a GnStats (None when the shape cannot).
    ``row_stats`` (row_stats_buffer(M, N)): per-row moments of ``out`` for a LayerNorm folded into the consumer.
    ``ln`` = (row statistics of A, column sums of the gamma-scaled W, eps): LayerNorm(A) @ W^T + b with A un-normalised.
    ``schedule`` (a dict): filled with what this launch runs (anysd_gemm_schedule, keys SCHEDULE_KEYS)."""
    _cuda(A, W, out)
    p = GemmParams()
    p.A, p.W, p.out = A.data_ptr(), W.data_ptr(), out.data_ptr()
    p.bias = bias.data_ptr() if bias is not None else None
    p.rowadd = rowadd.data_ptr() if rowadd is not None else None
    p.residual = residual.data_ptr() if residual is not None else None
    p.K = K if K is not None else A.shape[-1]
    p.M = M if M is not None else A.numel() // A.shape[-1]
    p.N = N if N is not None else W.shape[0]
    p.lda = lda if lda is not None else A.stride(-2) if A.dim() >= 2 else p.K
    p.ldw = ldw if ldw is not None else W.stride(0)
    p.ldo = out.stride(-2) if out.dim() >= 2 else out.shape[-1]
    p.ldr = residual.stride(-2) if residual is not None else 0
    p.ld_rowadd = ld_rowadd if ld_rowadd is not None else (rowadd.stride(0) if rowadd is not None else 0)
    p.rows_per_batch = rows_per_batch
    p.act = act
    p.out_dtype = _DT[out.dtype]
    p.conv = 0
    if row_stats is not None:
        assert row_stats.dtype == torch.float32 and row_stats.is_contiguous() and row_stats.numel() == (p.N // 64) * p.M * 2
        p.row_stats = row_stats.data_ptr()
    if ln is not None:
        lst, lcs, leps = ln
        assert lst.dtype == torch.float32 and lst.is_contiguous() and lst.numel() == (p.K // 64) * p.M * 2, "ln statistics shape"
        assert lcs.dtype == torch.float32 and lcs.is_contiguous() and lcs.numel() == p.N and bias is not None
        p.ln_stats, p.ln_colsum, p.ln_eps = lst.data_ptr(), lcs.data_ptr(), float(leps)
    st = _want_stats(p, stats_images, out.device) if stats_images > 0 else None
    _sk = _want_splitk(p, out.device) if (row_stats is None and ln is None) else None
    if schedule is not None:
        _fill_schedule(p, schedule)
    with _Traced("gemm", 2.0 * p.M * p.N * p.K, f"M={p.M} N={p.N} K={p.K} act={p.act} res={int(residual is not None)}"):
        _lib.check(_lib.load().anysd_gemm_f16(C.byref(p), _stream()), "gemm")
    _count()
    return st


def conv3x3(x, W, out, bias=None, rowadd=None, residual=None, stride=1, upsample=0, ld_rowadd=None,
            logical_cin=None, logical_cout=None, act=0, pad_rb=False, stats=False, schedule=None):
    """x NHWC fp16 [N,H,W,Cin]; W fp16 [Cout, 9*Cin] ((ky,kx,ci) K order); out [N*Ho*Wo, Cout].
    pad_rb (stride 2 only): zero padding on the right / bottom instead of all around (first-stage Downsample, model.py:83-85).
    ``schedule`` (a dict): filled with what this launch runs (see gemm)."""
    _cuda(x, W, out)
    Nimg, H, Wd, Cin = x.shape
    Hl, Wl = H << upsample, Wd << upsample
    if pad_rb:
        assert stride == 2 and not upsample
        Ho, Wo = (Hl - 2) // 2 + 1, (Wl - 2) // 2 + 1
    else:
        Ho, Wo = (Hl - 1) // stride + 1, (Wl - 1) // stride + 1
    p = GemmParams()
    p.A, p.W, p.out = x.data_ptr(), W.data_ptr(), out.data_ptr()
    p.bias = bias.data_ptr() if bias is not None else None
    p.rowadd = rowadd.data_ptr() if rowadd is not None else None
    p.residual = residual.data_ptr() if residual is not None else None
    p.M, p.N, p.K = Nimg * Ho * Wo, W.shape[0], 9 * Cin
    p.lda, p.ldw = Cin, W.stride(0)
    p.ldo = out.stride(-2)
    p.ldr = residual.stride(-2) if residual is not None else 0
    p.ld_rowadd = ld_rowadd if ld_rowadd is not None else (rowadd.stride(0) if rowadd is not None else 0)
    p.rows_per_batch = Ho * Wo
    p.act = act
    p.out_dtype = _DT[out.dtype]
    p.conv = 1
    p.conv_pad = int(bool(pad_rb))
    p.Nimg, p.H, p.Wd, p.Cin = Nimg, H, Wd, Cin
    p.stride, p.upsample = stride, upsample
    if upsample:   # scratch for the materialised nearest-x2 input of the tcgen05 path
        ws = torch.empty(Nimg * Hl * Wl * Cin, dtype=torch.float16, device=x.device)
        p.workspace, p.workspace_bytes = ws.data_ptr(), ws.numel() * 2
    # algorithmic FLOPs (trace only): zero-padded channels do not count
    fl = 2.0 * p.M * (logical_cout or p.N) * 9 * (logical_cin or Cin)
    st = _want_stats(p, Nimg, out.device, reuse=stats) if stats else None
    _sk = _want_splitk(p, out.device)
    if schedule is not None:
        _fill_schedule(p, schedule)
    with _Traced("conv3x3", fl, f"N={p.Nimg} {p.H}x{p.Wd} {p.Cin}->{p.N} s={p.stride} up={p.upsample} res={int(residual is not None)}"):
        _lib.check(_lib.load().anysd_gemm_f16(C.byref(p), _stream()), "conv3x3")
    _count()
    return st if stats else (Ho, Wo)


def attention(q, k, v, out, B, heads, n_q, n_kv, d, ld_q, ld_k, ld_v, ld_o, q_bs=None, k_bs=None, v_bs=None,
              o_bs=None, scale=None, gate=None, gate_stride=1, accumulate=False, head_stride=0, aux_cols=False, lse=None):
    """softmax(q k^T * scale) v per (batch, head); q/k/v may be column slices of fused projections.
    ``lse`` (fp32 [B, heads, n_q]): also store the base-2 log-sum-exp of every score row (for the backward)."""
    _cuda(q, k, v, out)
    p = AttnParams()
    p.q, p.k, p.v, p.out = q.data_ptr(), k.data_ptr(), v.data_ptr(), out.data_ptr()
    p.q_batch_stride = q_bs if q_bs is not None else n_q * ld_q
    p.k_batch_stride = k_bs if k_bs is not None else n_kv * ld_k
    p.v_batch_stride = v_bs if v_bs is not None else n_kv * ld_v
    p.o_batch_stride = o_bs if o_bs is not None else n_q * ld_o
    p.ld_q, p.ld_k, p.ld_v, p.ld_o = ld_q, ld_k, ld_v, ld_o
    p.B, p.heads, p.n_q, p.n_kv, p.d = B, heads, n_q, n_kv, d
    p.scale = float(scale if scale is not None else d ** -0.5)
    p.gate = gate.data_ptr() if gate is not None else None
    p.gate_stride = gate_stride
    p.accumulate = int(bool(accumulate))
    p.head_stride = head_stride
    p.aux_cols = int(bool(aux_cols))
    if lse is not None:
        assert lse.dtype == torch.float32 and lse.is_contiguous() and lse.numel() == B * heads * n_q
        p.lse = lse.data_ptr()
    with _Traced("attention", 4.0 * B * heads * n_q * n_kv * d, f"B={B} h={heads} nq={n_q} nkv={n_kv} d={d}"):
        _lib.check(_lib.load().anysd_attention_f16(C.byref(p), _stream()), "attention")
    _count()


def cfg_ddim_step(x, eps, coef, scale, cfg, x_prev, pred_x0=None, noise=None, v_param=False):
    """ddim.py:211-212, 228-250 in one kernel; all fp32 NCHW; coef is a device tensor of >= 5 floats (7 with v_param:
    the model output is v and coef[5:7] = sqrt(acp[t]), sqrt(1 - acp[t]))."""
    _cuda(x, eps, coef, x_prev)
    B = x.shape[0]
    n_per = x.numel() // B
    assert x.dtype == torch.float32 and eps.dtype == torch.float32 and x.is_contiguous() and eps.is_contiguous()
    _lib.check(_lib.load().anysd_cfg_ddim_step_f32(_ptr(x), _ptr(eps), _ptr(noise), _ptr(coef), float(scale),
                                                   int(bool(cfg)), int(bool(v_param)), _ptr(x_prev), _ptr(pred_x0), n_per, B, _stream()),
               "cfg_ddim_step")
    _count()


def cfg3_ddim_step(x, eps, coef, text_scale, image_scale, x_prev, pred_x0=None, noise=None):
    """InstructPix2Pix three-way guidance (eps = [text ; image ; uncond]) + DDIM update in one kernel."""
    _cuda(x, eps, coef, x_prev)
    B = x.shape[0]
    assert eps.shape[0] == 3 * B and x.dtype == torch.float32 and eps.dtype == torch.float32 and x.is_contiguous() and eps.is_contiguous()
    _lib.check(_lib.load().anysd_cfg3_ddim_step_f32(_ptr(x), _ptr(eps), _ptr(noise), _ptr(coef), float(text_scale), float(image_scale),
                                                    _ptr(x_prev), _ptr(pred_x0), x.numel() // B, B, _stream()), "cfg3_ddim_step")
    _count()


def cfg_plms_step(x, eps, coef, scale, cfg, hist, x_prev, pred_x0=None):
    """plms.py:178-244 in one kernel: CFG combine, multistep eps, DDIM update, history push; coef: 10 floats on the device,
    hist: fp32 [3, B, C, H, W] (zero-initialised)."""
    _cuda(x, eps, coef, hist, x_prev)
    B = x.shape[0]
    assert x.dtype == torch.float32 and eps.dtype == torch.float32 and hist.dtype == torch.float32
    assert x.is_contiguous() and eps.is_contiguous() and hist.is_contiguous() and hist.numel() == 3 * x.numel()
    _lib.check(_lib.load().anysd_cfg_plms_step_f32(_ptr(x), _ptr(eps), _ptr(coef), float(scale), int(bool(cfg)), _ptr(hist), _ptr(x_prev),
                                                   _ptr(pred_x0), x.numel() // B, B, _stream()), "cfg_plms_step")
    _count()


def cfg_dpmpp_step(x, eps, coef, scale, cfg, m_prev, x_next, x0_out=None):
    """One DPM-Solver++(2M) step (dpm_solver.py:352-365, 469-513, 723-778); coef: 6 floats on the device, m_prev: fp32 like x."""
    _cuda(x, eps, coef, m_prev, x_next)
    B = x.shape[0]
    assert x.dtype == torch.float32 and eps.dtype == torch.float32 and m_prev.dtype == torch.float32
    assert x.is_contiguous() and eps.is_contiguous() and m_prev.is_contiguous() and m_prev.numel() == x.numel()
    _lib.check(_lib.load().anysd_cfg_dpmpp_step_f32(_ptr(x), _ptr(eps), _ptr(coef), float(scale), int(bool(cfg)), _ptr(m_prev), _ptr(x_next),
                                                    _ptr(x0_out), x.numel() // B, B, _stream()), "cfg_dpmpp_step")
    _count()


def softmax_rows(S, P, scale):
    """P[r, :] = softmax(S[r, :] * scale); S fp32 [rows, n], P fp16 [rows, n] (row strides taken from the tensors)."""
    _cuda(S, P)
    assert S.dtype == torch.float32 and P.dtype == torch.float16 and S.stride(-1) == 1 and P.stride(-1) == 1
    rows, n = S.shape
    _lib.check(_lib.load().anysd_softmax_rows_f32(_ptr(S), S.stride(0), _ptr(P), P.stride(0), rows, n, float(scale), _stream()), "softmax_rows")
    _count()


def gaussian_posterior(moments, noise=None, sample=None, logvar=None, scale=1.0):
    """DiagonalGaussianDistribution pieces from fp32 NCHW moments [B, 2Z, H, W]; sample = scale * (mean + std * noise)."""
    _cuda(moments)
    assert moments.dtype == torch.float32 and moments.is_contiguous()
    B = moments.shape[0]
    zhw = moments.numel() // (2 * B)
    _lib.check(_lib.load().anysd_gaussian_posterior_f32(_ptr(moments), _ptr(noise), _ptr(sample), _ptr(logvar), float(scale), B, zhw, _stream()),
               "gaussian_posterior")
    _count()


def embed_tokens(ids, tok_table, pos_table, out):
    """out[b*n + i] = tok_table[ids[b, i]] + pos_table[i]; ids int64 [B, n], fp16 tables, out fp16 [B*n, D]."""
    _cuda(ids, tok_table, pos_table, out)
    B, n = ids.shape
    assert ids.dtype == torch.int64 and ids.is_contiguous() and tok_table.dtype == torch.float16 and pos_table.dtype == torch.float16
    assert tok_table.is_contiguous() and pos_table.is_contiguous() and pos_table.shape[0] >= n and out.is_contiguous()
    _lib.check(_lib.load().anysd_embed_tokens_f16(_ptr(ids), _ptr(tok_table), _ptr(pos_table), _ptr(out), B, n, tok_table.shape[1],
                                                  tok_table.shape[0], _stream()), "embed_tokens")
    _count()


def attention_small(q, k, v, out, B, heads, n_q, n_kv, d, ld_q, ld_k, ld_v, ld_o, scale=None, causal=False):
    """softmax(q k^T scale [+ causal mask]) v for short sequences (n_kv <= 256): the CLIP text tower."""
    _cuda(q, k, v, out)
    _lib.check(_lib.load().anysd_attention_small_f16(_ptr(q), _ptr(k), _ptr(v), _ptr(out), B, heads, n_q, n_kv, d, ld_q, ld_k, ld_v, ld_o,
                                                     float(scale if scale is not None else d ** -0.5), int(bool(causal)), _stream()),
               "attention_small")
    _count()


# ---- training step (SURVEY.md a24): thin wrappers, same conventions as above -------------------------------------
def q_sample(x0, noise, t, sqrt_acp, sqrt_1m_acp, out):
    _cuda(x0, noise, t, out)
    B = x0.shape[0]
    _lib.check(_lib.load().anysd_q_sample_f32(_ptr(x0), _ptr(noise), _ptr(t), _ptr(sqrt_acp), _ptr(sqrt_1m_acp), _ptr(out), B,
                                              x0.numel() // B, _stream()), "q_sample")
    _count()


def mse_loss(pred, target, d_pred, loss, grad_scale=1.0, grad_scale_dev=None):
    """pred/target fp32 NCHW; d_pred fp16 [N, HW, Cpad]; loss: 1-element fp32 tensor; grad_scale_dev: optional device
    scalar multiplied into the gradient (the dynamic loss scale)."""
    _cuda(pred, target, d_pred, loss)
    N, Cc = pred.shape[0], pred.shape[1]
    HW = pred.numel() // (N * Cc)
    ws = torch.empty(_lib.load().anysd_mse_workspace_bytes() // 4, dtype=torch.float32, device=pred.device)
    _lib.check(_lib.load().anysd_mse_loss_f32(_ptr(pred), _ptr(target), N, Cc, HW, d_pred.shape[-1], float(grad_scale), _ptr(grad_scale_dev),
                                              _ptr(d_pred), _ptr(loss), _ptr(ws), ws.numel() * 4, _stream()), "mse_loss")
    _count(2)


def geglu(pre, out):
    _cuda(pre, out)
    inner = out.shape[-1]
    _lib.check(_lib.load().anysd_geglu_f16(_ptr(pre), _ptr(out), out.numel() // inner, inner, _stream()), "geglu")
    _count()


def geglu_bwd(pre, d_out, d_pre):
    _cuda(pre, d_out, d_pre)
    inner = d_out.shape[-1]
    with _Traced("geglu_bwd", 0.0, f"inner={inner}"):
        _lib.check(_lib.load().anysd_geglu_bwd_f16(_ptr(pre), _ptr(d_out), _ptr(d_pre), d_out.numel() // inner, inner, _stream()), "geglu_bwd")
    _count()


def silu_bwd_f32(x, dy, dx):
    _cuda(x, dy, dx)
    _lib.check(_lib.load().anysd_silu_bwd_f32(_ptr(x), _ptr(dy), _ptr(dx), x.numel(), _stream()), "silu_bwd")
    _count()


def groupnorm_bwd(x1, gamma, beta, dy, dx, N, HW, eps, silu, x2=None, G=32):
    _cuda(x1, dy, dx)
    C1 = x1.shape[-1]
    C2 = x2.shape[-1] if x2 is not None else 0
    with _Traced("groupnorm_bwd", 0.0, f"N={N} HW={HW} C={C1}+{C2}"):
        _lib.check(_lib.load().anysd_groupnorm_bwd_nhwc_f16(_ptr(x1), C1, _ptr(x2), C2, _ptr(gamma), _ptr(beta), _ptr(dy), _ptr(dx), N, HW,
                                                            G, float(eps), int(bool(silu)), _stream()), "groupnorm_bwd")
    _count()


def layernorm_bwd(x, gamma, dy, dx, eps=1e-5):
    _cuda(x, dy, dx)
    Cc = x.shape[-1]
    with _Traced("layernorm_bwd", 0.0, f"C={Cc}"):
        _lib.check(_lib.load().anysd_layernorm_bwd_f16(_ptr(x), _ptr(gamma), _ptr(dy), _ptr(dx), x.numel() // Cc, Cc, float(eps), _stream()),
                   "layernorm_bwd")
    _count()


def attention_bwd(q, k, v, d_out, dq, dk, dv, B, heads, n_q, n_kv, d, ld_q, ld_k, ld_v, ld_do, ld_dq, ld_dk=0, ld_dv=0,
                  qk_scale=None, gate=None, gate_stride=1, d_gate=None, accumulate_dq=False, head_stride=0, out=None, ld_o=0, lse=None):
    """Backward of `attention` (recomputing the probabilities).  dk/dv None: frozen K/V.  out: this attention's own
    un-gated forward output (saves one sweep over K/V)."""
    _cuda(q, k, v, d_out, dq)
    p = _lib.AttnBwdParams()
    p.q, p.k, p.v, p.d_out, p.dq = q.data_ptr(), k.data_ptr(), v.data_ptr(), d_out.data_ptr(), dq.data_ptr()
    p.dk = dk.data_ptr() if dk is not None else None
    p.dv = dv.data_ptr() if dv is not None else None
    p.q_batch_stride, p.k_batch_stride, p.v_batch_stride = n_q * ld_q, n_kv * ld_k, n_kv * ld_v
    p.do_batch_stride, p.dq_batch_stride = n_q * ld_do, n_q * ld_dq
    p.dk_batch_stride, p.dv_batch_stride = n_kv * ld_dk, n_kv * ld_dv
    p.ld_q, p.ld_k, p.ld_v, p.ld_do, p.ld_dq, p.ld_dk, p.ld_dv = ld_q, ld_k, ld_v, ld_do, ld_dq, ld_dk, ld_dv
    p.B, p.heads, p.n_q, p.n_kv, p.d, p.head_stride = B, heads, n_q, n_kv, d, head_stride
    p.qk_scale = float(qk_scale if qk_scale is not None else d ** -0.5)
    p.gate = gate.data_ptr() if gate is not None else None
    p.gate_stride = gate_stride
    p.d_gate = d_gate.data_ptr() if d_gate is not None else None
    p.accumulate_dq = int(bool(accumulate_dq))
    p.out = out.data_ptr() if out is not None else None
    p.o_batch_stride, p.ld_o = n_q * ld_o, ld_o
    nbytes = _lib.load().anysd_attention_bwd_workspace_bytes(B, heads, n_q)
    ws = torch.empty(nbytes // 4, dtype=torch.float32, device=q.device)
    p.workspace, p.workspace_bytes = ws.data_ptr(), nbytes
    dpad = None
    if lse is not None and out is not None:        # the tcgen05 kernels (shape permitting; the library decides)
        assert lse.dtype == torch.float32 and lse.is_contiguous() and lse.numel() == B * heads * n_q
        hs = head_stride if head_stride > 0 else d
        dpad = torch.empty(B * n_q * heads * hs, dtype=torch.float16, device=q.device)
        p.lse, p.dout_padded = lse.data_ptr(), dpad.data_ptr()
    with _Traced("attention_bwd", 0.0, f"B={B} h={heads} nq={n_q} nkv={n_kv} d={d} dkv={int(dk is not None)}"):
        _lib.check(_lib.load().anysd_attention_bwd_f16(C.byref(p), _stream()), "attention_bwd")
    _count(2 if dk is not None else 1)


def _expert_params(q, ekv, gates, B, heads, n_q, n_kv, d, E, ld_q, ld_kv, ld_o, set_stride, v_offset, qk_scale, head_stride, out=None):
    p = _lib.ExpertAttnParams()
    p.q, p.kv = q.data_ptr(), ekv.data_ptr()
    p.out = out.data_ptr() if out is not None else None
    p.ld_q, p.ld_kv, p.ld_o = ld_q, ld_kv, ld_o
    p.B, p.heads, p.n_q, p.n_kv, p.d, p.head_stride, p.E = B, heads, n_q, n_kv, d, head_stride, E
    p.set_stride, p.v_offset = set_stride, v_offset
    p.qk_scale = float(qk_scale)
    p.gates, p.gate_b_stride = gates.data_ptr(), gates.stride(0)
    return p


def expert_attention(q, ekv, gates, out, B, heads, n_q, n_kv, d, E, ld_q, ld_kv, ld_o, set_stride, v_offset, qk_scale, head_stride=0):
    """out += sum_e gates[b, e] * softmax(qk_scale * q K_e^T) V_e for the E expert streams of one layer (one launch).
    gates: fp32 view [B, >= E] whose row stride selects the layer (gates[:, layer])."""
    _cuda(q, ekv, gates, out)
    p = _expert_params(q, ekv, gates, B, heads, n_q, n_kv, d, E, ld_q, ld_kv, ld_o, set_stride, v_offset, qk_scale, head_stride, out)
    with _Traced("expert_attention", 4.0 * B * heads * n_q * n_kv * d * E, f"B={B} h={heads} nq={n_q} nkv={n_kv} d={d} E={E}"):
        _lib.check(_lib.load().anysd_expert_attention_f16(C.byref(p), _stream()), "expert_attention")
    _count()


def expert_attention_bwd(q, ekv, gates, d_out, dq, dekv, d_gates, B, heads, n_q, n_kv, d, E, ld_q, ld_kv, ld_do, ld_dq, set_stride, v_offset,
                         qk_scale, head_stride=0):
    """Backward of `expert_attention`: dq += , dekv written in ekv's layout, d_gates (same view shape as gates) += ."""
    _cuda(q, ekv, gates, d_out, dq, dekv, d_gates)
    assert d_gates.stride(0) == gates.stride(0)
    p = _expert_params(q, ekv, gates, B, heads, n_q, n_kv, d, E, ld_q, ld_kv, ld_do, set_stride, v_offset, qk_scale, head_stride)
    nbytes = _lib.load().anysd_expert_attention_bwd_workspace_bytes(B, heads, E, n_q)
    ws = torch.empty(nbytes // 4, dtype=torch.float32, device=q.device)
    with _Traced("expert_attention_bwd", 0.0, f"B={B} h={heads} nq={n_q} nkv={n_kv} d={d} E={E}"):
        _lib.check(_lib.load().anysd_expert_attention_bwd_f16(C.byref(p), _ptr(d_out), ld_do, _ptr(dq), ld_dq, _ptr(dekv), _ptr(d_gates),
                                                              _ptr(ws), nbytes, _stream()), "expert_attention_bwd")
    _count(2)


def colsum(x, out, N, rows, accumulate=False):
    """x [N, rows, C] fp16 -> out[:N, :C] (fp32, row stride out.stride(0))."""
    _cuda(x, out)
    _lib.check(_lib.load().anysd_colsum_f16(_ptr(x), _ptr(out), N, rows, x.shape[-1], out.stride(0), int(bool(accumulate)), _stream()),
               "colsum")
    _count()


def add_(y, x):
    _cuda(y, x)
    assert y.numel() == x.numel() and y.is_contiguous() and x.is_contiguous()
    _lib.check(_lib.load().anysd_add_f16(_ptr(y), _ptr(x), y.numel(), _stream()), "add")
    _count()


def split_channels(src, a, b):
    _cuda(src, a, b)
    _lib.check(_lib.load().anysd_split_channels_f16(_ptr(src), _ptr(a), a.shape[-1], _ptr(b), b.shape[-1],
                                                    src.numel() // src.shape[-1], _stream()), "split_channels")
    _count()


def zero_insert2x(src, dst):
    _cuda(src, dst)
    N, H, W, Cc = src.shape
    _lib.check(_lib.load().anysd_zero_insert2x_f16(_ptr(src), _ptr(dst), N, H, W, Cc, _stream()), "zero_insert2x")
    _count()


def sumpool2x(src, dst):
    _cuda(src, dst)
    N, H, W, Cc = dst.shape
    _lib.check(_lib.load().anysd_sumpool2x_f16(_ptr(src), _ptr(dst), N, H, W, Cc, _stream()), "sumpool2x")
    _count()


def gemm_tn(A, B, out, M, Ka, Kb, lda=None, ldb=None, alpha=1.0, accumulate=False, head_d=0, head_stride=0, group_c=0,
            group_stride=0):
    """out[ka, kb] (+)= alpha * sum_m A[m, col(ka)] * B[m, kb]; A, B fp16, out fp32."""
    _cuda(A, B, out)
    with _Traced("gemm_tn", 0.0, f"M={M} Ka={Ka} Kb={Kb}"):
        _lib.check(_lib.load().anysd_gemm_tn_f32(_ptr(A), lda if lda is not None else A.stride(0), head_d, head_stride, group_c, group_stride,
                                                 _ptr(B),
                                                 ldb if ldb is not None else B.stride(0), _ptr(out), out.stride(0), M, Ka, Kb, float(alpha),
                                                 int(bool(accumulate)), _stream()), "gemm_tn")
    _count()


def gather_transpose(A, out, M, Ka, lda=None, head_d=0, head_stride=0, group_c=0, group_stride=0):
    """out[ka, m] = A[m, col(ka)]; out fp16 [Ka, ldo >= M] (columns >= M zero-filled)."""
    _cuda(A, out)
    _lib.check(_lib.load().anysd_gather_transpose_f16(_ptr(A), lda if lda is not None else A.stride(0), head_d, head_stride, group_c,
                                                      group_stride, _ptr(out), out.stride(0), M, Ka, _stream()), "gather_transpose")
    _count()


def router_bwd(gates, d_gates, te, W, dW, db, d_te, alpha=1.0):
    _cuda(gates, d_gates, te, W, dW, db, d_te)
    N, L, E = gates.shape
    _lib.check(_lib.load().anysd_router_bwd_f32(_ptr(gates), _ptr(d_gates), _ptr(te), _ptr(W), N, L, E, te.shape[-1], float(alpha),
                                                _ptr(dW), _ptr(db), _ptr(d_te), _stream()), "router_bwd")
    _count()


def scatter_add_rows(src, idx, table_grad, alpha=1.0):
    _cuda(src, idx, table_grad)
    _lib.check(_lib.load().anysd_scatter_add_rows_f32(_ptr(src), _ptr(idx), src.shape[0], src.shape[1], table_grad.shape[0], float(alpha),
                                                      _ptr(table_grad), _stream()), "scatter_add_rows")
    _count()


def _check_flat_f32(*ts):
    """The optimizer kernels take raw pointers and element counts: anything but dense fp32 on one device would be read and
    written out of bounds without an error."""
    dev = ts[0].device
    for t in ts:
        if t.dtype != torch.float32 or not t.is_contiguous() or t.device != dev or t.numel() != ts[0].numel():
            raise ValueError("anysd_b200 optimizer kernels need contiguous float32 tensors of equal size on one device "
                             f"(got {t.dtype}, contiguous={t.is_contiguous()}, {t.device}, {t.numel()} vs {ts[0].numel()} elements)")


def grad_check_(grad, scaler):
    """scaler[3] = 1 when any element of the flat fp32 gradient buffer is inf / nan."""
    _cuda(grad, scaler)
    _check_flat_f32(grad)
    _lib.check(_lib.load().anysd_grad_check_f32(_ptr(grad), grad.numel(), _ptr(scaler), _stream()), "grad_check")
    _count()


def adamw_scaled_(param, grad, exp_avg, exp_avg_sq, scaler, lr, beta1=0.9, beta2=0.999, eps=1e-8, weight_decay=1e-2, inv_world=1.0):
    """AdamW over flat fp32 buffers under the device-side loss scaler (skipped when scaler[3] != 0)."""
    _cuda(param, grad, exp_avg, exp_avg_sq, scaler)
    _check_flat_f32(param, grad, exp_avg, exp_avg_sq)
    _lib.check(_lib.load().anysd_adamw_scaled_f32(_ptr(param), _ptr(grad), _ptr(exp_avg), _ptr(exp_avg_sq), param.numel(), float(lr),
                                                  float(beta1), float(beta2), float(eps), float(weight_decay), float(inv_world), _ptr(scaler),
                                                  _stream()), "adamw_scaled")
    _count()


def loss_scale_update_(scaler, growth=2.0, backoff=0.5, interval=2000):
    _cuda(scaler)
    _lib.check(_lib.load().anysd_loss_scale_update_f32(_ptr(scaler), float(growth), float(backoff), int(interval), _stream()),
               "loss_scale_update")
    _count()


def adamw_(param, grad, exp_avg, exp_avg_sq, step, lr, beta1=0.9, beta2=0.999, eps=1e-8, weight_decay=1e-2, grad_scale=1.0):
    _cuda(param, grad, exp_avg, exp_avg_sq)
    _check_flat_f32(param, grad, exp_avg, exp_avg_sq)
    _lib.check(_lib.load().anysd_adamw_f32(_ptr(param), _ptr(grad), _ptr(exp_avg), _ptr(exp_avg_sq), param.numel(), float(lr),
                                           float(beta1), float(beta2), float(eps), float(weight_decay), int(step), float(grad_scale),
                                           _stream()), "adamw")
    _count()
