"""ctypes binding of libmeshanything_b200.so (include/meshanything_b200.h).

The library is built in-tree by `meshanything_b200.build` (nvcc, sm_100a).  There is no CPU or
PyTorch fallback: if the shared object cannot be loaded every call raises.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import torch

from . import build as _build

MA_MAX_LAYERS = 32
EPI_NONE, EPI_RELU, EPI_GELU = 0, 1, 2
LIN_SEG64, LIN_SEG256 = 0x10, 0x20   # OR-ed into the epilogue: segmented order of the decoder's out_proj / fc2
GEN_NO_GRAPH, GEN_NO_FAST, GEN_NO_PDL, GEN_NO_EARLY_EXIT, GEN_NO_MEGA, GEN_TRACE, GEN_TC = 1, 2, 4, 8, 16, 32, 64

_vp = C.c_void_p


class DecoderWeights(C.Structure):
    _fields_ = (
        [("n_layers", C.c_int), ("vocab", C.c_int), ("codebook", C.c_int), ("npos", C.c_int)]
        + [(n, _vp * MA_MAX_LAYERS) for n in ("wqkv", "bqkv", "wo", "bo", "w1", "b1", "w2", "b2",
                                              "ln1g", "ln1b", "ln2g", "ln2b")]
        + [(n, _vp) for n in ("lm_head", "tok_table", "extra", "tok_pos", "cond", "pos")]
    )


class Sampling(C.Structure):
    _fields_ = [("do_sample", C.c_int), ("top_k", C.c_int), ("top_p", C.c_float), ("seed", C.c_uint64)]


_lib = None

EXPORTS = [
    "ma_abi_version", "ma_last_error", "ma_launch_count", "ma_linear_f16", "ma_layernorm",
    "ma_attention_scratch_bytes", "ma_attention_f16", "ma_attention_decode_f16", "ma_kv_cache_bytes", "ma_decoder_workspace_bytes",
    "ma_decode_generate", "ma_decoder_debug", "ma_encoder_workspace_bytes", "ma_encoder_forward",
    "ma_detokenize_workspace_bytes", "ma_detokenize", "ma_linear_tc_f16", "ma_set_tensor_cores", "ma_sample_tokens",
    "ma_attention_tc_f16", "ma_transpose_heads_f16",
    "ma_decode_slots_init", "ma_decode_slot_prefill", "ma_decode_slots_step", "ma_decode_slots_poll",
    "ma_mega_set_debug", "ma_linear_ws_set_mode", "ma_decode_slots_seek", "ma_decode_slot_stream", "ma_linear_ws_scratch_bytes", "ma_linear_ws_f16",
    "ma_sample_surface_workspace_bytes", "ma_sample_surface", "ma_tensor_core_linear_counts",
    "ma_mesh_udf", "ma_marching_cubes_workspace_bytes", "ma_marching_cubes_count", "ma_marching_cubes_emit",
]


def lib_path() -> str:
    return _build.LIB


def lib():
    """Load (building if stale and nvcc is available) the shared library."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.LIB
    # rebuild when the library is older than its sources -- in a development checkout only (.git present, nvcc
    # available): the GPU box gets the prebuilt file with a snapshot whose mtimes are those of the copy
    dev_tree = os.path.isdir(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), ".git"))
    stale = (os.path.exists(path) and dev_tree and _build.have_nvcc()
             and os.environ.get("MA_B200_NO_AUTOBUILD") != "1" and _build._stale())
    if not os.path.exists(path) or stale or (os.environ.get("MA_B200_REBUILD") == "1"):
        path = _build.build(force=True)
    L = C.CDLL(path)
    L.ma_abi_version.restype = C.c_int
    L.ma_last_error.restype = C.c_char_p
    L.ma_launch_count.restype = C.c_ulonglong
    L.ma_linear_f16.argtypes = [_vp, _vp, _vp, C.c_int, _vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _vp]
    L.ma_layernorm.argtypes = [_vp, _vp, _vp, _vp, C.c_float, C.c_int, C.c_int, _vp, _vp, _vp]
    L.ma_attention_scratch_bytes.argtypes = [C.c_int, C.c_int, C.c_int]
    L.ma_attention_scratch_bytes.restype = C.c_size_t
    L.ma_attention_f16.argtypes = [_vp, C.c_int, _vp, _vp, C.c_long, C.c_int, _vp, _vp, C.c_int, C.c_int,
                                   C.c_float, _vp, C.c_int, _vp, _vp]
    L.ma_kv_cache_bytes.argtypes = [C.c_int, C.c_int, C.c_int]
    L.ma_kv_cache_bytes.restype = C.c_size_t
    L.ma_decoder_workspace_bytes.argtypes = [C.c_int, C.c_int]
    L.ma_decoder_workspace_bytes.restype = C.c_size_t
    L.ma_decode_generate.argtypes = [C.POINTER(DecoderWeights), _vp, C.c_int, C.c_int, C.c_int, C.POINTER(Sampling),
                                     C.c_int, C.c_int, _vp, _vp, _vp, _vp, _vp, _vp, C.c_int, _vp]
    L.ma_sample_tokens.argtypes = [_vp, C.c_int, C.c_int, C.POINTER(Sampling), _vp, _vp, _vp]
    L.ma_attention_decode_f16.argtypes = [_vp, C.c_int, _vp, _vp, C.c_long, _vp, C.c_int, C.c_int, C.c_float, _vp, C.c_int,
                                          _vp, _vp]
    L.ma_attention_tc_f16.argtypes = [_vp, C.c_int, _vp, _vp, C.c_long, C.c_long, C.c_int, C.c_int, C.c_int, C.c_int,
                                      C.c_float, _vp, C.c_int, _vp]
    L.ma_transpose_heads_f16.argtypes = [_vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_long, C.c_int, _vp, _vp]
    L.ma_decode_slots_init.argtypes = [C.c_int, C.c_int, C.c_int, _vp, _vp]
    L.ma_linear_ws_set_mode.argtypes = [C.c_int]
    L.ma_linear_ws_set_mode.restype = None
    L.ma_decode_slot_stream.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, _vp, _vp]
    L.ma_decode_slots_seek.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _vp, _vp]
    L.ma_decode_slot_prefill.argtypes = [C.POINTER(DecoderWeights), _vp, C.c_int, C.c_int, C.c_int, C.c_int,
                                         C.POINTER(Sampling), C.c_int, C.c_int, _vp, _vp, _vp, _vp]
    L.ma_decode_slots_step.argtypes = [C.POINTER(DecoderWeights), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                       C.POINTER(Sampling), C.c_int, C.c_int, _vp, _vp, _vp, C.c_int, _vp]
    L.ma_decode_slots_poll.argtypes = [C.c_int, C.c_int, _vp, _vp, _vp, _vp]
    L.ma_decoder_debug.argtypes = [_vp, C.c_int, C.c_int, C.c_int, _vp, C.c_int]
    L.ma_mega_set_debug.argtypes = [C.c_ulonglong, C.c_int]
    L.ma_mega_set_debug.restype = None
    L.ma_encoder_workspace_bytes.argtypes = [C.c_int]
    L.ma_encoder_workspace_bytes.restype = C.c_size_t
    L.ma_encoder_forward.argtypes = [_vp, _vp, C.c_int, _vp, _vp, _vp, _vp]
    L.ma_detokenize_workspace_bytes.argtypes = [C.c_int, C.c_int]
    L.ma_detokenize_workspace_bytes.restype = C.c_size_t
    L.ma_detokenize.argtypes = [_vp, _vp, C.c_int, C.c_int, C.c_int, _vp, _vp, _vp, _vp, _vp]
    L.ma_linear_ws_scratch_bytes.restype = C.c_size_t
    L.ma_linear_ws_f16.argtypes = [_vp, _vp, _vp, C.c_int, _vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _vp, _vp]
    L.ma_sample_surface_workspace_bytes.argtypes = [C.c_int]
    L.ma_sample_surface_workspace_bytes.restype = C.c_size_t
    L.ma_sample_surface.argtypes = [_vp, _vp, C.c_int, C.c_int, C.c_ulonglong, _vp, _vp, _vp, _vp]
    L.ma_mesh_udf.argtypes = [_vp, _vp, C.c_int, C.c_int, _vp, _vp]
    L.ma_marching_cubes_workspace_bytes.argtypes = [C.c_int]
    L.ma_marching_cubes_workspace_bytes.restype = C.c_size_t
    L.ma_marching_cubes_count.argtypes = [_vp, C.c_int, C.c_float, _vp, _vp, _vp]
    L.ma_marching_cubes_emit.argtypes = [_vp, C.c_int, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, _vp, _vp,
                                         _vp, _vp]
    L.ma_linear_tc_f16.argtypes = [_vp, _vp, _vp, C.c_int, _vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _vp]
    L.ma_set_tensor_cores.argtypes = [C.c_int]
    L.ma_tensor_core_linear_counts.argtypes = [C.POINTER(C.c_ulonglong), C.POINTER(C.c_ulonglong)]
    L.ma_tensor_core_linear_counts.restype = None
    if L.ma_abi_version() != 1:
        raise RuntimeError("libmeshanything_b200.so: ABI version mismatch")
    _lib = L
    return L


def check(rc: int, what: str):
    if rc != 0:
        raise RuntimeError(f"{what} failed: {lib().ma_last_error().decode()}")


def ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


def stream_ptr() -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _need_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError("meshanything_b200: tensors must live on a CUDA device (no CPU fallback)")


# ---------------------------------------------------------------- canonical building blocks

def linear_f16(w: torch.Tensor, bias: Optional[torch.Tensor], x: torch.Tensor, epilogue: int = EPI_NONE,
               out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """fp16(x @ w.T + bias) with the canonical accumulation order.  w [N,K] fp16, x [M,K] fp16."""
    _need_cuda(w, bias, x)
    assert w.dtype == torch.float16 and x.dtype == torch.float16 and w.is_contiguous()
    assert x.dim() == 2 and x.stride(1) == 1
    M, K = x.shape
    N = w.shape[0]
    if out is None:
        out = torch.empty((M, N), dtype=torch.float16, device=x.device)
    check(lib().ma_linear_f16(ptr(w), ptr(bias), ptr(x), x.stride(0), ptr(out), out.stride(0), M, N, K, epilogue,
                              stream_ptr()), "ma_linear_f16")
    return out


def sample_surface(vertices: torch.Tensor, faces: torch.Tensor, n_samples: int, seed: int = 0,
                   want_index: bool = False):
    """Area-weighted surface samples + face normals on the GPU: fp16 [n_samples, 6] (and the face of every sample)."""
    _need_cuda(vertices, faces)
    v = vertices.to(torch.float32).contiguous()
    f = faces.to(torch.int32).contiguous()
    F = f.shape[0]
    ws = torch.empty(lib().ma_sample_surface_workspace_bytes(F), dtype=torch.uint8, device=v.device)
    out = torch.empty((n_samples, 6), dtype=torch.float16, device=v.device)
    idx = torch.empty((n_samples,), dtype=torch.int32, device=v.device) if want_index else None
    check(lib().ma_sample_surface(ptr(v), ptr(f), F, n_samples, int(seed), ptr(out), ptr(idx), ptr(ws), stream_ptr()),
          "ma_sample_surface")
    return (out, idx) if want_index else out


def mesh_udf(vertices: torch.Tensor, faces: torch.Tensor, size: int) -> torch.Tensor:
    """Unsigned distance field min(d, 2h) of a mesh normalised to +-0.9 on the size^3 grid of [-1, 1 - h]^3, h = 2/size:
    fp32 [size, size, size] indexed [i][j][k].  Face indices must lie in [0, V) (the caller checks)."""
    _need_cuda(vertices, faces)
    v = vertices.to(torch.float32).contiguous()
    f = faces.to(torch.int32).contiguous()
    field = torch.empty((size, size, size), dtype=torch.float32, device=v.device)
    check(lib().ma_mesh_udf(ptr(v), ptr(f), f.shape[0], size, ptr(field), stream_ptr()), "ma_mesh_udf")
    return field


def marching_cubes(field: torch.Tensor, level: float, inv_scale: float = 1.0, centre=(0.0, 0.0, 0.0)):
    """Closed, outward-oriented level set of a cubic fp32 field -> (vertices fp32 [V, 3], faces int32 [F, 3]) on the
    device; vertex = ((grid index * h) - 1) * inv_scale + centre.  Reads the two counts back (one synchronisation)."""
    _need_cuda(field)
    size = field.shape[0]
    if field.dim() != 3 or field.shape != (size, size, size):
        raise ValueError(f"marching_cubes: field must be a cube, got {tuple(field.shape)}")
    fd = field.to(torch.float32).contiguous()
    ws = torch.empty(max(lib().ma_marching_cubes_workspace_bytes(size), 1), dtype=torch.uint8, device=fd.device)
    counts = torch.empty(2, dtype=torch.int32, device=fd.device)
    check(lib().ma_marching_cubes_count(ptr(fd), size, C.c_float(level), ptr(counts), ptr(ws), stream_ptr()),
          "ma_marching_cubes_count")
    nv, nf = counts.tolist()
    verts = torch.empty((nv, 3), dtype=torch.float32, device=fd.device)
    faces = torch.empty((nf, 3), dtype=torch.int32, device=fd.device)
    if nf > 0:
        cx, cy, cz = (float(c) for c in centre)
        check(lib().ma_marching_cubes_emit(ptr(fd), size, C.c_float(level), C.c_float(inv_scale), C.c_float(cx),
                                           C.c_float(cy), C.c_float(cz), ptr(verts), ptr(faces), ptr(ws), stream_ptr()),
              "ma_marching_cubes_emit")
    return verts, faces


def tensor_core_linear_counts():
    """(Linear calls of the encoder / detokenizer that ran on tcgen05, calls that fell back to the canonical kernel)."""
    a, b = C.c_ulonglong(0), C.c_ulonglong(0)
    lib().ma_tensor_core_linear_counts(C.byref(a), C.byref(b))
    return a.value, b.value


_ws_scratch = {}


def linear_ws_f16(w: torch.Tensor, bias: Optional[torch.Tensor], x: torch.Tensor, epilogue: int = EPI_NONE) -> torch.Tensor:
    """fp16(x @ w.T + bias) for M <= 128 rows on the weight-streaming tcgen05 GEMM (hardware accumulation order)."""
    _need_cuda(w, bias, x)
    M, K = x.shape
    N = w.shape[0]
    scr = _ws_scratch.get(x.device)
    if scr is None:
        scr = _ws_scratch[x.device] = torch.zeros(lib().ma_linear_ws_scratch_bytes(), dtype=torch.uint8, device=x.device)
    out = torch.empty((M, N), dtype=torch.float16, device=x.device)
    check(lib().ma_linear_ws_f16(ptr(w), ptr(bias), ptr(x), x.stride(0), ptr(out), out.stride(0), M, N, K, epilogue,
                                 ptr(scr), stream_ptr()), "ma_linear_ws_f16")
    return out


def linear_tc_f16(w: torch.Tensor, bias: Optional[torch.Tensor], x: torch.Tensor, epilogue: int = EPI_NONE) -> torch.Tensor:
    """fp16(x @ w.T + bias) on the tcgen05 tensor cores (hardware accumulation order)."""
    _need_cuda(w, bias, x)
    M, K = x.shape
    N = w.shape[0]
    out = torch.empty((M, N), dtype=torch.float16, device=x.device)
    check(lib().ma_linear_tc_f16(ptr(w), ptr(bias), ptr(x), x.stride(0), ptr(out), out.stride(0), M, N, K, epilogue,
                                 stream_ptr()), "ma_linear_tc_f16")
    return out


def transpose_heads_f16(src: torch.Tensor, col0: int, head_stride: int, H: int, n: int, n_slots: int) -> torch.Tensor:
    """src fp16 [n_slots*n, ld] -> V^T fp16 [n_slots, H, 64, Tpad] (Tpad = n rounded up to 128, zero padded)."""
    _need_cuda(src)
    Tpad = (n + 127) // 128 * 128
    dst = torch.empty((n_slots, H, 64, Tpad), dtype=torch.float16, device=src.device)
    check(lib().ma_transpose_heads_f16(ptr(src), src.stride(0), col0, head_stride, H, n, Tpad, n_slots, ptr(dst),
                                       stream_ptr()), "ma_transpose_heads_f16")
    return dst


def attention_tc_f16(q: torch.Tensor, k: torch.Tensor, vt: torch.Tensor, nkeys: int, rows_per_slot: int,
                     scale: float = 0.125) -> torch.Tensor:
    """q [n_slots*rows_per_slot, H*64]; k [n_slots, H, T, 64]; vt [n_slots, H, 64, Tpad] (V transposed, zero beyond
    nkeys) -> [rows, H*64], on the tcgen05 tensor cores."""
    _need_cuda(q, k, vt)
    S, H, T, _ = k.shape
    Tpad = vt.shape[3]
    assert q.is_contiguous() and k.is_contiguous() and vt.is_contiguous() and q.shape[0] == S * rows_per_slot
    out = torch.empty_like(q)
    check(lib().ma_attention_tc_f16(ptr(q), q.stride(0), ptr(k), ptr(vt), T, Tpad, H, rows_per_slot, S, nkeys,
                                    C.c_float(scale), ptr(out), out.stride(0), stream_ptr()), "ma_attention_tc_f16")
    return out


def sample_tokens(logits: torch.Tensor, do_sample: bool = True, top_k: int = 50, top_p: float = 0.95, seed: int = 0,
                  want_support: bool = False):
    """One pick of the sampling chain (TopK -> TopP -> multinomial) over fp16 logits [B, vocab]."""
    _need_cuda(logits)
    assert logits.dtype == torch.float16 and logits.is_contiguous()
    B, vocab = logits.shape
    tok = torch.empty((B,), dtype=torch.int32, device=logits.device)
    sup = torch.empty((B, 256), dtype=torch.int32, device=logits.device) if want_support else None
    s = Sampling(int(do_sample), int(top_k), float(top_p), int(seed))
    check(lib().ma_sample_tokens(ptr(logits), B, vocab, C.byref(s), ptr(tok), ptr(sup), stream_ptr()),
          "ma_sample_tokens")
    return (tok, sup) if want_support else tok


def layernorm(x: Optional[torch.Tensor], res16: Optional[torch.Tensor], gamma: torch.Tensor, beta: torch.Tensor,
              eps: float = 1e-5, want32: bool = True, want16: bool = True):
    _need_cuda(x, res16, gamma, beta)
    src = x if x is not None else res16
    M, W = src.shape
    o32 = torch.empty((M, W), dtype=torch.float32, device=src.device) if want32 else None
    o16 = torch.empty((M, W), dtype=torch.float16, device=src.device) if want16 else None
    check(lib().ma_layernorm(ptr(x), ptr(res16), ptr(gamma), ptr(beta), eps, M, W, ptr(o32), ptr(o16), stream_ptr()),
          "ma_layernorm")
    return o32, o16


def attention_decode_f16(qkv: torch.Tensor, k: torch.Tensor, v: torch.Tensor, nkeys: torch.Tensor,
                         scale: float = 0.125) -> torch.Tensor:
    """qkv [M,3072] fp16 (q | k | v of the current token); k,v [M,16,T,64] fp16 caches (updated in place at nkeys-1);
    nkeys int32 [M] counts the current token.  Returns the attention output [M,1024] fp16."""
    _need_cuda(qkv, k, v, nkeys)
    M = qkv.shape[0]
    assert qkv.shape[1] == 3072 and qkv.is_contiguous() and k.is_contiguous() and v.is_contiguous()
    assert k.shape[0] == M and k.shape[1] == 16 and k.shape[3] == 64
    T = k.shape[2]
    max_keys = int(nkeys.max().item())
    scratch = torch.zeros(lib().ma_attention_scratch_bytes(M, 16, max_keys), dtype=torch.uint8, device=qkv.device)
    out = torch.empty((M, 1024), dtype=torch.float16, device=qkv.device)
    check(lib().ma_attention_decode_f16(ptr(qkv), 3072, ptr(k), ptr(v), T, ptr(nkeys), max_keys, M, scale, ptr(out),
                                        1024, ptr(scratch), stream_ptr()), "ma_attention_decode_f16")
    return out


def attention_f16(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, nkeys: torch.Tensor,
                  slots: Optional[torch.Tensor] = None, scale: float = 0.125) -> torch.Tensor:
    """q [M,H,64] fp16; k,v [S,H,T,64] fp16 (S cache slots); nkeys int32 [M]; slots int32 [M] or None (slot m)."""
    _need_cuda(q, k, v, nkeys, slots)
    M, H, D = q.shape
    assert D == 64 and k.is_contiguous() and v.is_contiguous() and q.is_contiguous()
    T = k.shape[2]
    max_keys = int(nkeys.max().item())
    scratch = torch.zeros(lib().ma_attention_scratch_bytes(M, H, max_keys), dtype=torch.uint8, device=q.device)
    out = torch.empty((M, H, D), dtype=torch.float16, device=q.device)
    check(lib().ma_attention_f16(ptr(q), H * D, ptr(k), ptr(v), T, H, ptr(slots), ptr(nkeys), max_keys, M, scale,
                                 ptr(out), H * D, ptr(scratch), stream_ptr()), "ma_attention_f16")
    return out
