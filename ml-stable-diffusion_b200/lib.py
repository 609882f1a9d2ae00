"""ctypes binding of ``libb200sd.so`` (the C-ABI in ``include/b200sd.h``) + thin torch-tensor
wrappers.  PyTorch is plumbing here (device memory, streams); every compute call goes through
the C-ABI.  There is NO fallback: a missing library or a failing call raises."""
from __future__ import annotations

import ctypes as C
import os
import weakref

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libb200sd.so")
_lib = None


class B200SDError(RuntimeError):
    pass


class GemmArgs(C.Structure):
    _fields_ = [
        ("mode", C.c_int32), ("m", C.c_int32), ("n", C.c_int32), ("c0", C.c_int32), ("c1", C.c_int32),
        ("n_img", C.c_int32), ("h", C.c_int32), ("w", C.c_int32), ("stride", C.c_int32),
        ("geglu", C.c_int32), ("out_f32", C.c_int32), ("bias_rows", C.c_int32), ("bias_stride", C.c_int32),
        ("split_k", C.c_int32),
        ("block_n", C.c_int32), ("act", C.c_int32), ("wgt_tiled", C.c_int32), ("pad_after_only", C.c_int32),
        ("a0", C.c_void_p), ("a1", C.c_void_p), ("wgt", C.c_void_p), ("bias", C.c_void_p),
        ("residual", C.c_void_p), ("out", C.c_void_p), ("workspace", C.c_void_p),
        ("workspace_bytes", C.c_size_t),
        # fused normalisation (include/b200sd.h): halo convolution + GroupNorm operand transform, statistics outputs,
        # LayerNorm fold
        ("halo", C.c_int32), ("upsample2x", C.c_int32), ("gn_groups", C.c_int32), ("gn_silu", C.c_int32),
        ("gn_eps", C.c_float),
        ("gn_chan0", C.c_void_p), ("gn_chan1", C.c_void_p), ("gn_gamma", C.c_void_p), ("gn_beta", C.c_void_p),
        ("cs_partial", C.c_void_p), ("cs_chan", C.c_void_p), ("cs_tickets", C.c_void_p), ("cs_hw", C.c_int32),
        ("rs_out", C.c_void_p),
        ("ln_stat", C.c_void_p), ("ln_wg", C.c_void_p), ("ln_parts", C.c_int32), ("ln_eps", C.c_float),
        ("a2", C.c_void_p), ("a3", C.c_void_p), ("c2", C.c_int32), ("c3", C.c_int32),
    ]


class StepCoeffs(C.Structure):
    _fields_ = [
        ("guidance", C.c_float), ("cx", C.c_float), ("ce", C.c_float), ("ch", C.c_float * 4),
        ("x0_cx", C.c_float), ("x0_ce", C.c_float), ("x0_ch", C.c_float * 4), ("n_hist", C.c_int32),
        ("push_eps_slot", C.c_int32), ("push_x0_slot", C.c_int32), ("push_x_slot", C.c_int32),
        ("noise_pred_nhwc", C.c_int32),
    ]


class SamplerCoeffs(C.Structure):
    """b200sd_sampler_coeffs: the step coefficients + input scale, noise scale and Philox draw index."""
    _fields_ = [("step", StepCoeffs), ("in_scale", C.c_float), ("noise_scale", C.c_float), ("noise_draw", C.c_uint32)]


_SIGNATURES = {
    "b200sd_last_error": (C.c_char_p, []),
    "b200sd_version": (C.c_int, []),
    "b200sd_launch_count": (C.c_uint64, []),
    "b200sd_set_pdl": (None, [C.c_int]),
    "b200sd_set_launch_classes": (None, [C.c_uint32]),
    # model-level handles (capi.py holds the struct mirrors)
    "b200sd_unet_create": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]),
    "b200sd_unet_prepare_prompt": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "b200sd_unet_forward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_void_p, C.c_void_p]),
    "b200sd_unet_set_attention_impl": (C.c_int, [C.c_void_p, C.c_int32]),
    "b200sd_unet_device_bytes": (C.c_size_t, [C.c_void_p]),
    "b200sd_destroy": (None, [C.c_void_p]),
    "b200sd_gemm": (C.c_int, [C.POINTER(GemmArgs), C.c_void_p]),
    "b200sd_gemm_workspace_bytes": (C.c_size_t, [C.POINTER(GemmArgs)]),
    "b200sd_gemm_plan": (C.c_int, [C.POINTER(GemmArgs), C.POINTER(C.c_int32)]),
    "b200sd_gemm_plan_ex": (C.c_int, [C.POINTER(GemmArgs), C.POINTER(C.c_int32)]),
    "b200sd_gemm_describe_plan": (C.c_int, [C.POINTER(GemmArgs), C.c_char_p, C.c_size_t]),
    "b200sd_linear_small": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                      C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "b200sd_timestep_embedding": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_float,
                                            C.c_void_p]),
    "b200sd_group_norm": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                    C.c_float, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p,
                                    C.c_size_t, C.c_void_p]),
    "b200sd_group_norm_workspace_bytes": (C.c_size_t, [C.c_int32, C.c_int32, C.c_int32, C.c_int32]),
    "b200sd_group_norm_apply": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                          C.c_float, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p,
                                          C.c_void_p]),
    "b200sd_layer_norm": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                    C.c_float, C.c_void_p]),
    "b200sd_softmax_rows": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_float, C.c_void_p]),
    "b200sd_latent_prep": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_void_p, C.c_int32, C.c_int32,
                                     C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "b200sd_attention": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                   C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                   C.c_int32, C.c_float, C.c_int32, C.c_void_p]),
    "b200sd_attention_workspace_bytes": (C.c_size_t, []),
    "b200sd_attention_ws": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                      C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                      C.c_int32, C.c_float, C.c_int32, C.c_void_p, C.c_size_t, C.c_void_p]),
    "b200sd_nchw_to_nhwc": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                      C.c_int32, C.c_int32, C.c_void_p]),
    "b200sd_nhwc_to_nchw_f32": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                          C.c_int32, C.c_int32, C.c_void_p]),
    "b200sd_upsample2x": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                    C.c_void_p]),
    "b200sd_add": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "b200sd_ctx_to_tokens": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                       C.c_void_p]),
    "b200sd_embed_tokens": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                      C.c_int32, C.c_void_p]),
    "b200sd_cfg_scheduler_step": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                            C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.POINTER(StepCoeffs),
                                            C.c_void_p]),
    "b200sd_sampler_step": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                      C.c_int32, C.c_int32, C.c_int32, C.POINTER(SamplerCoeffs), C.c_void_p, C.c_void_p]),
    "b200sd_image_postprocess": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32,
                                           C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)


def lib_path() -> str:
    return _LIB_PATH


def load():
    """Load the CUDA library; raise loudly if it has not been built (no CPU fallback exists)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_LIB_PATH):
        raise B200SDError(
            f"{_LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). b200sd has no CPU or PyTorch fallback path.")
    lib = C.CDLL(_LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    if t is None:
        return None
    return C.c_void_p(t.data_ptr())


_DEBUG_SYNC = bool(os.environ.get("B200SD_DEBUG_SYNC"))


def _check(rc, what):
    if rc != 0:
        msg = load().b200sd_last_error().decode(errors="replace")
        raise B200SDError(f"{what} failed (rc={rc}): {msg}")
    if _DEBUG_SYNC:  # debugging aid: localise a faulting / hanging kernel
        print(f"[b200sd] {what} launched", flush=True)
        torch.cuda.synchronize()
        print(f"[b200sd] {what} done", flush=True)


def launch_count() -> int:
    return int(load().b200sd_launch_count())


# ------------------------------------------------------------------------------------------------
# op wrappers (torch tensors in, torch tensors out; all on the current CUDA stream)
# ------------------------------------------------------------------------------------------------
def _req(t, dtype, what):
    if t.dtype != dtype or not t.is_cuda or not t.is_contiguous():
        raise B200SDError(f"{what}: expected contiguous CUDA {dtype}, got {t.dtype} {t.device} "
                          f"contiguous={t.is_contiguous()}")


def gemm_args(mode, a0, wgt, out, *, a1=None, bias=None, residual=None, m=0, n=0, n_img=0, h=0, w=0, stride=1,
              geglu=False, bias_rows=0, bias_stride=0, split_k=0, block_n=0, workspace=None, act=0, pad_after_only=False):
    args = GemmArgs()
    args.mode = mode
    args.m = m
    args.n = n
    args.c0 = a0.shape[-1]
    args.c1 = 0 if a1 is None else a1.shape[-1]
    args.n_img, args.h, args.w, args.stride = n_img, h, w, stride
    args.geglu = int(geglu)
    args.out_f32 = int(out.dtype == torch.float32)
    args.bias_rows = bias_rows
    args.bias_stride = bias_stride
    args.split_k = split_k
    args.block_n = block_n
    args.act = act
    args.pad_after_only = int(pad_after_only)
    args.a0 = a0.data_ptr()
    args.a1 = None if a1 is None else a1.data_ptr()
    args.wgt = wgt.data_ptr()
    args.bias = None if bias is None else bias.data_ptr()
    args.residual = None if residual is None else residual.data_ptr()
    args.out = out.data_ptr()
    args.workspace = None if workspace is None else workspace.data_ptr()
    args.workspace_bytes = 0 if workspace is None else workspace.numel() * workspace.element_size()
    return args


def describe_plan(mode, m=0, n=0, c0=0, c1=0, n_img=0, h=0, w=0, stride=1, geglu=False, has_bias=True,
                  has_residual=False, bias_rows=0, split_k=0, block_n=0) -> str:
    """Host-only: the tiling the launcher would choose (no GPU needed)."""
    a = GemmArgs()
    a.mode, a.m, a.n, a.c0, a.c1, a.n_img, a.h, a.w, a.stride = mode, m, n, c0, c1, n_img, h, w, stride
    a.geglu, a.bias_rows, a.split_k, a.block_n = int(geglu), bias_rows, split_k, block_n
    a.bias = 1 if has_bias else None       # only tested for null-ness by the planner
    a.residual = 1 if has_residual else None
    buf = C.create_string_buffer(512)
    _check(load().b200sd_gemm_describe_plan(C.byref(a), buf, 512), "b200sd_gemm_describe_plan")
    return buf.value.decode()


TILED_WEIGHTS = os.environ.get("B200SD_TILED_W", "1") != "0"
_tiled_cache = {}


def pack_tiled(w2d, c0, c1, taps, bn, chunk_major=False, extra=(0, 0)):
    """[N, taps*(c0+c1) (+ c2 + c3)] -> [n_tiles, k_blocks, bn, 64] fp16 in the exact k-block order of the kernel's main
    loop (tap-major; per tap the 64-channel chunks of source 0, then of source 1; ragged chunks zero padded), so
    that each weight tile is one contiguous bn*128-byte burst in HBM.  chunk_major: k-block = chunk * taps + tap
    (the halo convolution walks all nine taps of one 64-channel chunk before the next chunk).  extra = (c2, c3): the
    folded shortcut's columns follow the convolution's: their chunks (source 2, then source 3) are the last k-blocks."""
    n, kpt = w2d.shape[0], c0 + c1
    kc0, kc1 = (c0 + 63) // 64, (c1 + 63) // 64
    kc = kc0 + kc1
    nt = (n + bn - 1) // bn
    c2, c3 = extra
    wp = torch.zeros(nt * bn, taps, kpt, dtype=w2d.dtype, device=w2d.device)
    wp[:n] = w2d[:, : taps * kpt].reshape(n, taps, kpt)
    out = torch.zeros(nt, taps, kc, bn, 64, dtype=w2d.dtype, device=w2d.device)
    for j in range(kc):
        lo = j * 64 if j < kc0 else c0 + (j - kc0) * 64
        hi = min(lo + 64, c0 if j < kc0 else kpt)
        out[:, :, j, :, : hi - lo] = wp[:, :, lo:hi].reshape(nt, bn, taps, hi - lo).permute(0, 2, 1, 3)
    if chunk_major:
        out = out.permute(0, 2, 1, 3, 4)
    out = out.reshape(nt, taps * kc, bn, 64)
    if c2 + c3:
        if chunk_major:
            raise B200SDError("pack_tiled: shortcut columns are not supported in the chunk-major (halo) layout")
        kc2, kc3 = (c2 + 63) // 64, (c3 + 63) // 64
        we = torch.zeros(nt * bn, c2 + c3, dtype=w2d.dtype, device=w2d.device)
        we[:n] = w2d[:, taps * kpt:]
        ext = torch.zeros(nt, kc2 + kc3, bn, 64, dtype=w2d.dtype, device=w2d.device)
        for j in range(kc2 + kc3):
            lo = j * 64 if j < kc2 else c2 + (j - kc2) * 64
            hi = min(lo + 64, c2 if j < kc2 else c2 + c3)
            ext[:, j, :, : hi - lo] = we[:, lo:hi].reshape(nt, bn, hi - lo)
        out = torch.cat([out, ext], 1)
    return out.contiguous()


def plan_ex(args):
    """(block_n, splits, kb_total, n_tiles, stat slots per image, staged, stages, m_tiles) of a call."""
    plan = (C.c_int32 * 8)()
    _check(load().b200sd_gemm_plan_ex(C.byref(args), plan), "b200sd_gemm_plan_ex")
    return tuple(int(v) for v in plan)


def _maybe_tile_weights(args, wgt, taps):
    """Static weight operands are re-laid out once per (weight, block_n) and cached."""
    bn = plan_ex(args)[0]
    key = (wgt.data_ptr(), bn, args.c0, args.c1, taps, bool(args.halo), args.c2, args.c3)
    hit = _tiled_cache.get(key)
    packed = None
    if hit is not None and hit[0]() is wgt and hit[1] == wgt._version:
        packed = hit[2]
    if packed is None:
        if torch.cuda.is_current_stream_capturing():
            return  # never pack during capture; the warm-up pass has populated the cache for these shapes
        packed = pack_tiled(wgt, args.c0, args.c1, taps, bn, chunk_major=bool(args.halo), extra=(args.c2, args.c3))
        if len(_tiled_cache) > 4096:  # drop entries whose source tensor is gone
            for k in [k for k, v in _tiled_cache.items() if v[0]() is None]:
                del _tiled_cache[k]
        _tiled_cache[key] = (weakref.ref(wgt), wgt._version, packed)
    args.wgt = packed.data_ptr()
    args.block_n = bn
    args.wgt_tiled = 1


def gemm_workspace_bytes(args) -> int:
    return int(load().b200sd_gemm_workspace_bytes(C.byref(args)))


def run_gemm(args):
    _check(load().b200sd_gemm(C.byref(args), _stream()), "b200sd_gemm")


_ws_cache = {}
_ws_retired = []   # superseded workspaces stay allocated: CUDA graphs captured earlier hold their addresses
_ticket_cache = {}


def _workspace(nbytes, device):
    """Process-wide scratch (split-K partials, GroupNorm / column-statistics partials).  Kernels that use it are
    stream-ordered on the single compute stream of the process.  It only ever grows (outside of CUDA-graph
    capture: the warm-up pass sizes it) and a superseded buffer is never freed, so pointers baked into
    previously captured graphs stay valid."""
    key = device.index
    ws = _ws_cache.get(key)
    if ws is None or ws.numel() * 4 < nbytes:
        if torch.cuda.is_current_stream_capturing():
            raise B200SDError("workspace would have to grow during CUDA-graph capture; run one eager "
                              "warm-up call with the same shapes first")
        if ws is not None:
            _ws_retired.append(ws)
        ws = torch.empty(max(nbytes // 4 + 1, 1 << 24), dtype=torch.float32, device=device)
        _ws_cache[key] = ws
    return ws


def _tickets(device):
    """Arrival counters of the statistics epilogue ([n_img][n_tiles] per call): zero once, self-resetting, shared by
    every call on the device (calls are stream ordered)."""
    t = _ticket_cache.get(device.index)
    if t is None:
        t = torch.zeros(1 << 16, dtype=torch.int32, device=device)
        _ticket_cache[device.index] = t
    return t


def _fused_args(args, x_dev, *, n_img, cout, gn=None, stats=None, cs_hw=0, ln=None, rowstats=None, m=0):
    """Fill the fused-normalisation fields of a GemmArgs.  gn: dict(chan0, chan1, gamma, beta, groups, eps, silu);
    stats: dict, receives 'chan' [n_img, cout, 2]; rowstats: dict, receives 'rows' [n_tiles, m, 2] and 'parts';
    ln: dict(stat, parts, wg, eps)."""
    keep = []
    if gn is not None:
        args.gn_groups, args.gn_silu, args.gn_eps = int(gn["groups"]), int(bool(gn["silu"])), float(gn["eps"])
        args.gn_chan0 = gn["chan0"].data_ptr()
        args.gn_chan1 = None if gn.get("chan1") is None else gn["chan1"].data_ptr()
        args.gn_gamma, args.gn_beta = gn["gamma"].data_ptr(), gn["beta"].data_ptr()
    if ln is not None:
        args.ln_stat, args.ln_wg = ln["stat"].data_ptr(), ln["wg"].data_ptr()
        args.ln_parts, args.ln_eps = int(ln["parts"]), float(ln.get("eps", 1e-5))
    if stats is not None or rowstats is not None:
        if stats is not None:
            args.cs_partial = 1  # planning query: non-null
            args.cs_hw = cs_hw
        if rowstats is not None:
            args.rs_out = 1
        try:
            pl = plan_ex(args)
        except B200SDError:
            if stats is None:
                raise
            # this geometry cannot emit column statistics (e.g. images smaller than 16 pixels): the caller sees no
            # 'chan' entry and its consumer falls back to the standalone GroupNorm kernel
            args.cs_partial, args.cs_hw, stats = None, 0, None
            if rowstats is None:
                return keep
            pl = plan_ex(args)
        n_tiles, slots = pl[3], pl[4]
        if stats is not None:
            if n_img * n_tiles > (1 << 16):
                raise B200SDError("statistics ticket table too small")
            chan = torch.empty(n_img, cout, 2, dtype=torch.float32, device=x_dev)
            part = _workspace(n_img * slots * cout * 2 * 4, x_dev)
            args.cs_partial, args.cs_chan, args.cs_tickets = part.data_ptr(), chan.data_ptr(), _tickets(x_dev).data_ptr()
            stats["chan"] = chan
            keep.append(chan)
        if rowstats is not None:
            parts = n_tiles if pl[5] else 2 * n_tiles  # register epilogue: one partial per column half of a tile
            rows = torch.empty(parts, m, 2, dtype=torch.float32, device=x_dev)
            args.rs_out = rows.data_ptr()
            rowstats["rows"], rowstats["parts"] = rows, parts
            keep.append(rows)
    return keep


def linear(x, wgt, bias=None, residual=None, *, x1=None, geglu=False, out_dtype=torch.float16, split_k=0,
           block_n=0, bias_rows=0, bias_stride=0, out=None, static_w=False, act=0, ln=None, stats=None, cs_hw=0,
           rowstats=None):
    """out[M, N] = epilogue([x | x1] @ wgt^T).  x [M, C0] fp16, wgt [N, C0(+C1)] fp16, bias fp32 [N].
    static_w: `wgt` is a model weight (constant address/content) and may be re-tiled + cached.
    ln: LayerNorm of x folded into this GEMM (wgt = gamma (.) W, bias = W beta + b; dict(stat, parts, wg, eps));
    stats / rowstats: dicts that receive the per-channel / per-row sums of the output (see _fused_args)."""
    _req(x, torch.float16, "linear x")
    _req(wgt, torch.float16, "linear wgt")
    m, n = x.shape[0], wgt.shape[0]
    n_out = n // 2 if geglu else n
    if out is None:
        out = torch.empty(m, n_out, dtype=out_dtype, device=x.device)
    args = gemm_args(0, x, wgt, out, a1=x1, bias=bias, residual=residual, m=m, n=n, geglu=geglu,
                     bias_rows=bias_rows, bias_stride=bias_stride, split_k=split_k, block_n=block_n, act=act)
    if ln is not None or stats is not None or rowstats is not None:
        args.split_k = 1
        _keep = _fused_args(args, x.device, n_img=(m // cs_hw if cs_hw else 0), cout=n, stats=stats, cs_hw=cs_hw, ln=ln,
                            rowstats=rowstats, m=m)
    if static_w and TILED_WEIGHTS:
        _maybe_tile_weights(args, wgt, 1)
    need = gemm_workspace_bytes(args)
    if need:
        ws = _workspace(need, x.device)
        args.workspace = ws.data_ptr()
        args.workspace_bytes = ws.numel() * 4
    run_gemm(args)
    return out


def conv3x3(x, wgt, bias=None, residual=None, *, x1=None, stride=1, out_dtype=torch.float16, split_k=0,
            block_n=0, bias_rows=0, bias_stride=0, out=None, act=0, static_w=True, pad_after_only=False,
            halo=False, gn=None, upsample=False, stats=None, rowstats=None, taps=9, shortcut=None):
    """3x3 pad-1 convolution.  x NHWC fp16 [N, H, W, C0]; wgt [Cout, 9*(C0+C1)] fp16 (OHWI);
    bias fp32 [Cout] or [N_img, Cout] with bias_rows = Hout*Wout.
    halo: the halo-reuse kernel (stride 1); gn: GroupNorm (+SiLU) of x ++ x1 applied while loading (dict(chan0, chan1,
    gamma, beta, groups, eps, silu), needs halo); upsample: x is read nearest-x2 upsampled (halo); stats: dict that
    receives 'chan', the per-channel (sum, sum of squares) of the output for the consumer's GroupNorm; taps=1 with
    halo: a 1x1 convolution (wgt [Cout, C0+C1]) that shares the halo kernel's GroupNorm operand path.
    shortcut = (s0, s1 or None): the ResNet shortcut folded in -- wgt is [Cout, 9*(C0+C1) + Cs0 + Cs1] (the 1x1
    shortcut matrix appended along K), bias the sum of both biases, s0 / s1 NHWC fp16 at the output resolution."""
    _req(x, torch.float16, "conv3x3 x")
    _req(wgt, torch.float16, "conv3x3 wgt")
    nimg, h, w, _ = x.shape
    if upsample:
        h, w = 2 * h, 2 * w
    cout = wgt.shape[0]
    ho, wo = h // stride, w // stride
    if out is None:
        out = torch.empty(nimg, ho, wo, cout, dtype=out_dtype, device=x.device)
    if (gn is not None or upsample or taps == 1) and not halo:
        raise B200SDError("conv3x3: gn / upsample / taps=1 need halo=True")
    args = gemm_args(1 if taps == 9 else 0, x, wgt, out, a1=x1, bias=bias, residual=residual, n=cout, n_img=nimg, h=h, w=w,
                     stride=stride, bias_rows=bias_rows, bias_stride=bias_stride, split_k=split_k, block_n=block_n, act=act,
                     pad_after_only=pad_after_only, m=(nimg * h * w if taps == 1 else 0))
    args.halo, args.upsample2x = int(halo), int(upsample)
    if shortcut is not None:
        s0, s1 = shortcut
        if stride != 1 or taps != 9 or halo or not (static_w and TILED_WEIGHTS):
            raise B200SDError("conv3x3: a folded shortcut needs the stride-1 9-tap kernel with static pre-tiled weights")
        _req(s0, torch.float16, "conv3x3 shortcut source")
        args.a2, args.c2 = s0.data_ptr(), s0.shape[-1]
        if s1 is not None:
            _req(s1, torch.float16, "conv3x3 shortcut source 1")
            args.a3, args.c3 = s1.data_ptr(), s1.shape[-1]
    _keep = None
    if gn is not None or stats is not None or rowstats is not None:
        args.split_k = 1
        _keep = _fused_args(args, x.device, n_img=nimg, cout=cout, gn=gn, stats=stats, cs_hw=ho * wo, rowstats=rowstats,
                            m=nimg * ho * wo)
    if halo and not (static_w and TILED_WEIGHTS):
        raise B200SDError("conv3x3: the halo kernel needs static pre-tiled weights")
    if static_w and TILED_WEIGHTS:
        _maybe_tile_weights(args, wgt, taps)
    need = gemm_workspace_bytes(args)
    if need:
        ws = _workspace(need, x.device)
        args.workspace = ws.data_ptr()
        args.workspace_bytes = ws.numel() * 4
    run_gemm(args)
    return out


def linear_small(x, wgt, bias=None, add=None, act_in=False, act_out=False):
    _req(x, torch.float32, "linear_small x")
    _req(wgt, torch.float16, "linear_small wgt")
    m, k = x.shape
    n = wgt.shape[0]
    out = torch.empty(m, n, dtype=torch.float32, device=x.device)
    _check(load().b200sd_linear_small(_ptr(x), _ptr(wgt), _ptr(bias), _ptr(add), _ptr(out), m, n, k,
                                      int(act_in), int(act_out), _stream()), "b200sd_linear_small")
    return out


def timestep_embedding(t, dim, flip_sin_to_cos=True, freq_shift=0.0):
    _req(t, torch.float32, "timestep_embedding t")
    out = torch.empty(t.shape[0], dim, dtype=torch.float32, device=t.device)
    _check(load().b200sd_timestep_embedding(_ptr(t), _ptr(out), t.shape[0], dim, int(flip_sin_to_cos),
                                            float(freq_shift), _stream()), "b200sd_timestep_embedding")
    return out


def group_norm(x, gamma, beta, groups, eps, silu=False, x1=None, out=None):
    """x NHWC fp16 [N, H, W, C0] (optionally ++ x1 [N, H, W, C1]) -> normalised [N, H, W, C0+C1]."""
    _req(x, torch.float16, "group_norm x")
    nimg, h, w, c0 = x.shape
    c1 = 0 if x1 is None else x1.shape[-1]
    if out is None:
        out = torch.empty(nimg, h, w, c0 + c1, dtype=torch.float16, device=x.device)
    need = int(load().b200sd_group_norm_workspace_bytes(nimg, h * w, c0 + c1, groups))
    ws = _workspace(need, x.device)
    _check(load().b200sd_group_norm(_ptr(x), _ptr(x1), c0, c1, nimg, h * w, groups, float(eps), _ptr(gamma),
                                    _ptr(beta), int(silu), _ptr(out), _ptr(ws), ws.numel() * 4, _stream()),
           "b200sd_group_norm")
    return out


def group_norm_apply(x, chan0, gamma, beta, groups, eps, silu=False, x1=None, chan1=None, out=None):
    """GroupNorm (+SiLU, + concat) from the producers' per-channel sums ``chan0`` / ``chan1`` [N, C, 2]: no statistics pass."""
    _req(x, torch.float16, "group_norm_apply x")
    nimg, h, w, c0 = x.shape
    c1 = 0 if x1 is None else x1.shape[-1]
    if out is None:
        out = torch.empty(nimg, h, w, c0 + c1, dtype=torch.float16, device=x.device)
    _check(load().b200sd_group_norm_apply(_ptr(x), _ptr(x1), c0, c1, nimg, h * w, groups, float(eps), _ptr(chan0), _ptr(chan1),
                                          _ptr(gamma), _ptr(beta), int(silu), _ptr(out), _stream()), "b200sd_group_norm_apply")
    return out


def layer_norm(x, gamma, beta, eps=1e-5, out=None):
    _req(x, torch.float16, "layer_norm x")
    rows, c = x.shape
    if out is None:
        out = torch.empty_like(x)
    _check(load().b200sd_layer_norm(_ptr(x), _ptr(gamma), _ptr(beta), _ptr(out), rows, c, float(eps), _stream()),
           "b200sd_layer_norm")
    return out


def attention(q, k, v, batch, heads, sq, sk, d=64, mask=None, impl=0, out=None, scale=None, causal=False):
    """q: view [batch*sq, >=heads*d] (row stride = q.stride(0)), k/v: [batch*sk, ...]; out [batch*sq, heads*d].
    causal: key j is visible to query i only if j <= i (CLIP text encoder)."""
    for t, nm in ((q, "q"), (k, "k"), (v, "v")):
        if t.dtype != torch.float16 or not t.is_cuda or t.stride(-1) != 1:
            raise B200SDError(f"attention {nm}: expected CUDA fp16 with unit inner stride")
    if out is None:
        out = torch.empty(batch * sq, heads * d, dtype=torch.float16, device=q.device)
    scale = float(d) ** -0.5 if scale is None else float(scale)
    ws = _attention_workspace(q.device)
    _check(load().b200sd_attention_ws(_ptr(q), _ptr(k), _ptr(v), _ptr(out), _ptr(mask), batch, heads, sq, sk, d,
                                      q.stride(0), k.stride(0), v.stride(0), out.stride(0), scale,
                                      int(impl) | (0x100 if causal else 0), _ptr(ws), ws.numel(),
                                      _stream()), "b200sd_attention_ws")
    return out


_attn_ws = {}


def _attention_workspace(device):
    """Zero-filled once per device: the stream-K pieces of split query tiles meet here; its counters return to zero at
    the end of every launch.  Launches on one stream are ordered, which is the only way this package launches."""
    key = device.index if device.index is not None else torch.cuda.current_device()
    ws = _attn_ws.get(key)
    if ws is None:
        ws = torch.zeros(int(load().b200sd_attention_workspace_bytes()), dtype=torch.uint8, device=device)
        _attn_ws[key] = ws
    return ws


def nchw_to_nhwc(x, c_pad=None, out=None):
    n, c, h, w = x.shape
    c_pad = c if c_pad is None else c_pad
    if x.dtype not in (torch.float16, torch.float32) or not x.is_contiguous():
        raise B200SDError("nchw_to_nhwc: expected contiguous fp16/fp32")
    if out is None:
        out = torch.empty(n, h, w, c_pad, dtype=torch.float16, device=x.device)
    elif out.dtype != torch.float16 or not out.is_contiguous() or tuple(out.shape) != (n, h, w, c_pad):
        raise B200SDError("nchw_to_nhwc: bad output buffer")
    _check(load().b200sd_nchw_to_nhwc(_ptr(x), int(x.dtype == torch.float32), _ptr(out), n, c, h, w, c_pad,
                                      _stream()), "b200sd_nchw_to_nhwc")
    return out


def nhwc_to_nchw_f32(x, c=None, out=None):
    n, h, w, c_pad = x.shape
    c = c_pad if c is None else c
    if out is None:
        out = torch.empty(n, c, h, w, dtype=torch.float32, device=x.device)
    _check(load().b200sd_nhwc_to_nchw_f32(_ptr(x), int(x.dtype == torch.float32), _ptr(out), n, c, h, w, c_pad,
                                          _stream()), "b200sd_nhwc_to_nchw_f32")
    return out


def upsample2x(x, out=None):
    _req(x, torch.float16, "upsample2x x")
    n, h, w, c = x.shape
    if out is None:
        out = torch.empty(n, 2 * h, 2 * w, c, dtype=torch.float16, device=x.device)
    _check(load().b200sd_upsample2x(_ptr(x), _ptr(out), n, h, w, c, _stream()), "b200sd_upsample2x")
    return out


def add(a, b, out=None):
    _req(a, torch.float16, "add a")
    _req(b, torch.float16, "add b")
    if out is None:
        out = torch.empty_like(a)
    _check(load().b200sd_add(_ptr(a), _ptr(b), _ptr(out), a.numel(), _stream()), "b200sd_add")
    return out


def embed_tokens(ids, token_embedding, position_embedding, out=None):
    """ids fp32 [B, S]; tables fp16 [V, D] / [S, D] -> fp16 [B*S, D] (token + position embedding)."""
    _req(ids, torch.float32, "embed_tokens ids")
    _req(token_embedding, torch.float16, "embed_tokens token_embedding")
    _req(position_embedding, torch.float16, "embed_tokens position_embedding")
    b, s = ids.shape
    v, d = token_embedding.shape
    if position_embedding.shape[0] < s or position_embedding.shape[1] != d:
        raise B200SDError("embed_tokens: position table does not cover the sequence")
    if out is None:
        out = torch.empty(b * s, d, dtype=torch.float16, device=ids.device)
    _check(load().b200sd_embed_tokens(_ptr(ids), _ptr(token_embedding), _ptr(position_embedding), _ptr(out), b, s, d, v,
                                      _stream()), "b200sd_embed_tokens")
    return out


def ctx_to_tokens(ctx, out=None):
    """(B, D, 1, S) fp16/fp32 -> [B*S, D] fp16."""
    b, d, _, s = ctx.shape
    if not ctx.is_contiguous():
        raise B200SDError("ctx_to_tokens: expected contiguous input")
    if out is None:
        out = torch.empty(b * s, d, dtype=torch.float16, device=ctx.device)
    _check(load().b200sd_ctx_to_tokens(_ptr(ctx), int(ctx.dtype == torch.float32), _ptr(out), b, d, s, _stream()),
           "b200sd_ctx_to_tokens")
    return out


def cfg_scheduler_step(noise_pred, latents, coeffs: StepCoeffs, hist=None, denoised=None, unet_in=None):
    _req(noise_pred, torch.float32, "cfg_scheduler_step noise_pred")
    _req(latents, torch.float32, "cfg_scheduler_step latents")
    n, c, h, w = latents.shape
    c_pad = 0 if unet_in is None else unet_in.shape[-1]
    _check(load().b200sd_cfg_scheduler_step(_ptr(noise_pred), _ptr(latents), _ptr(hist), _ptr(denoised),
                                            _ptr(unet_in), c_pad, n, c, h, w, C.byref(coeffs), _stream()),
           "b200sd_cfg_scheduler_step")
    return latents


def sampler_step(noise_pred, latents, coeffs: SamplerCoeffs, hist=None, denoised=None, unet_in=None, rng_key=None):
    """b200sd_sampler_step.  noise_pred None: input-only mode (unet_in = fp16(in_scale * latents)); rng_key: int32 CUDA
    tensor of 2 words (the Philox key), needed when coeffs.noise_scale != 0."""
    if noise_pred is not None:
        _req(noise_pred, torch.float32, "sampler_step noise_pred")
    _req(latents, torch.float32, "sampler_step latents")
    if rng_key is not None and (rng_key.dtype != torch.int32 or not rng_key.is_cuda or rng_key.numel() < 2):
        raise B200SDError("sampler_step: rng_key must be a CUDA int32 tensor of 2 words")
    n, c, h, w = latents.shape
    c_pad = 0 if unet_in is None else unet_in.shape[-1]
    _check(load().b200sd_sampler_step(_ptr(noise_pred), _ptr(latents), _ptr(hist), _ptr(denoised), _ptr(unet_in), c_pad,
                                      n, c, h, w, C.byref(coeffs), _ptr(rng_key), _stream()), "b200sd_sampler_step")
    return latents


def image_postprocess(x, c=3, want_u8=False):
    n, h, w, c_pad = x.shape
    of = torch.empty(n, h, w, c, dtype=torch.float32, device=x.device)
    ou = torch.empty(n, h, w, c, dtype=torch.uint8, device=x.device) if want_u8 else None
    _check(load().b200sd_image_postprocess(_ptr(x), int(x.dtype == torch.float32), c_pad, _ptr(of), _ptr(ou), n, h,
                                           w, c, _stream()), "b200sd_image_postprocess")
    return (of, ou) if want_u8 else of


def softmax_rows(scores, scale, out=None):
    _req(scores, torch.float32, "softmax_rows scores")
    rows, cols = scores.shape
    if out is None:
        out = torch.empty(rows, cols, dtype=torch.float16, device=scores.device)
    _check(load().b200sd_softmax_rows(_ptr(scores), _ptr(out), rows, cols, float(scale), _stream()),
           "b200sd_softmax_rows")
    return out


def latent_prep(z, w, b, inv_scale, c_pad=8):
    _req(z, torch.float32, "latent_prep z")
    n, c, h, wd = z.shape
    out = torch.empty(n, h, wd, c_pad, dtype=torch.float16, device=z.device)
    _check(load().b200sd_latent_prep(_ptr(z), _ptr(w), _ptr(b), float(inv_scale), _ptr(out), n, c, h, wd, c_pad,
                                     _stream()), "b200sd_latent_prep")
    return out
