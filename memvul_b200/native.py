"""ctypes binding of ``libmemvul_b200.so`` (C ABI in ``include/memvul_b200.h``).

PyTorch is plumbing here: it owns device memory and streams; every function below hands raw
device pointers and the current CUDA stream to the hand-written sm_100a kernels.  There is NO
CPU or library fallback: if the shared library is missing or the device is not a B200-class
GPU the call raises.
"""
from __future__ import annotations

import ctypes
import os
import subprocess
import threading
from typing import Dict, List, Optional

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
_REPO = os.path.dirname(_HERE)
LIB_PATH = os.environ.get("MEMVUL_LIB_PATH") or os.path.join(_HERE, "libmemvul_b200.so")   # override: experiment builds (tools/)
SOURCES = ["memvul_abi.cu", "ptx.cuh", "gemm_tcgen05.cuh", "gemm_tcgen05_2cta.cuh", "gemm_ln_tcgen05.cuh", "attention_tcgen05.cuh",
           "attention_tcgen05_v2.cuh", "attention_tcgen05_v3.cuh", "rowwise.cuh", "pool_match.cuh", "precise.cuh"]

ABI_VERSION = 3
EPI_BIAS_F16, EPI_BIAS_GELU_F16, EPI_BIAS_RESID_F32, EPI_BIAS_F32 = 0, 1, 2, 3
PM_POOL, PM_HEADER, PM_UTERM, PM_MATCH, PM_FINAL, PM_ALL = 1, 2, 4, 8, 16, 31

_lock = threading.Lock()
_lib: Optional[ctypes.CDLL] = None


class NativeError(RuntimeError):
    pass


def nvcc_command(out: str = LIB_PATH) -> List[str]:
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    return [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo",
            "-shared", "-Xcompiler", "-fPIC", "-o", out, os.path.join(_HERE, "csrc", "memvul_abi.cu")]


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile the CUDA library in-tree (cross-compiles without a GPU)."""
    srcs = [os.path.join(_HERE, "csrc", s) for s in SOURCES] + [os.path.join(_REPO, "include", "memvul_b200.h")]
    if not force and os.path.exists(LIB_PATH):
        if os.path.getmtime(LIB_PATH) >= max(os.path.getmtime(s) for s in srcs if os.path.exists(s)):
            return LIB_PATH
    cmd = nvcc_command()
    if verbose:
        print(" ".join(cmd))
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise NativeError("nvcc failed:\n" + r.stdout + r.stderr)
    return LIB_PATH


class BertLayerC(ctypes.Structure):
    _fields_ = [(n, ctypes.c_void_p) for n in (
        "w_qkv", "b_qkv", "w_ao", "b_ao", "ln1_g", "ln1_b", "w_ff1", "b_ff1", "w_ff2", "b_ff2", "ln2_g", "ln2_b")]


class BertWeightsC(ctypes.Structure):
    _fields_ = [("hidden", ctypes.c_int32), ("layers", ctypes.c_int32), ("heads", ctypes.c_int32),
                ("intermediate", ctypes.c_int32), ("vocab", ctypes.c_int32), ("max_pos", ctypes.c_int32),
                ("type_vocab", ctypes.c_int32), ("ln_eps", ctypes.c_float),
                ("word_emb", ctypes.c_void_p), ("pos_emb", ctypes.c_void_p), ("type_emb", ctypes.c_void_p),
                ("emb_ln_g", ctypes.c_void_p), ("emb_ln_b", ctypes.c_void_p),
                ("layer", ctypes.POINTER(BertLayerC))]


EXPORTS = ["memvul_abi_version", "memvul_last_error", "memvul_encoder_workspace_bytes", "memvul_encoder_forward",
           "memvul_mask_to_lens", "memvul_bank_prepare", "memvul_pool_match", "memvul_single_head",
           "memvul_gemm_f16", "memvul_gemm_ln_f16", "memvul_attention_f16", "memvul_attention_f32", "memvul_split3_f16",
           "memvul_layernorm", "memvul_embed_layernorm",
           "memvul_launch_count", "memvul_profile_enable", "memvul_profile_read"]
KERNEL_CLASSES = ["embed_ln", "gemm_qkv", "attention", "gemm_attn_out", "layernorm", "gemm_ffn_up", "gemm_ffn_down",
                  "pool_match", "other", "attention_cls", "cls_tail"]


def lib() -> ctypes.CDLL:
    global _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise NativeError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                                  "(memvul_b200 has no fallback path)")
            L = ctypes.CDLL(LIB_PATH)
            vp, i32, i64, f32 = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_float
            L.memvul_abi_version.restype = ctypes.c_int
            L.memvul_last_error.restype = ctypes.c_char_p
            L.memvul_encoder_workspace_bytes.restype = ctypes.c_size_t
            L.memvul_encoder_workspace_bytes.argtypes = [ctypes.POINTER(BertWeightsC), i32, i32, i32]
            L.memvul_encoder_forward.argtypes = [ctypes.POINTER(BertWeightsC), vp, vp, vp, vp, i32, i32, vp, vp,
                                                 ctypes.c_size_t, i32, vp, vp]
            L.memvul_mask_to_lens.argtypes = [vp, i32, i32, vp, vp, vp, vp]
            L.memvul_bank_prepare.argtypes = [vp, vp, i32, i32, vp, vp]
            L.memvul_pool_match.argtypes = [vp, i64, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32,
                                            vp, vp, vp, vp, vp, vp, vp, vp, i32, vp]
            L.memvul_single_head.argtypes = [vp, vp, i32, i32, vp, vp, vp]
            L.memvul_gemm_f16.argtypes = [vp, vp, vp, vp, vp, i32, i32, i32, i32, vp]
            L.memvul_gemm_ln_f16.argtypes = [vp, vp, vp, vp, vp, vp, f32, vp, vp, i32, i32, i32, vp]
            L.memvul_attention_f16.argtypes = [vp, vp, vp, vp, i32, i32, i32, vp]
            L.memvul_attention_f32.argtypes = [vp, vp, vp, vp, i32, i32, i32, vp]
            L.memvul_split3_f16.argtypes = [vp, vp, i32, i32, i32, vp]
            L.memvul_layernorm.argtypes = [vp, vp, vp, f32, vp, vp, i32, i32, vp]
            L.memvul_embed_layernorm.argtypes = [ctypes.POINTER(BertWeightsC), vp, vp, vp, vp, i32, i32, vp, vp, vp, vp]
            L.memvul_launch_count.restype = ctypes.c_longlong
            L.memvul_profile_enable.argtypes = [i32]
            L.memvul_profile_read.argtypes = [i32, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_longlong)]
            for name in EXPORTS:
                if name not in ("memvul_last_error", "memvul_encoder_workspace_bytes", "memvul_launch_count"):
                    getattr(L, name).restype = ctypes.c_int
            if L.memvul_abi_version() != ABI_VERSION:
                raise NativeError("libmemvul_b200.so ABI version mismatch")
            _lib = L
        return _lib


def _check(rc: int) -> None:
    if rc != 0:
        msg = lib().memvul_last_error().decode("utf-8", "replace")
        raise (ValueError if rc == -1 else NativeError)(f"memvul_b200 native call failed ({rc}): {msg}")


def _on(t: torch.Tensor):
    """Device guard: the kernels launch in the CURRENT CUDA context, so every native call runs with the device of its
    tensors current (a model moved with ``.cuda(1)`` in a process whose current device is 0 must still work)."""
    if not t.is_cuda:
        raise NativeError("memvul_b200 has no CPU path: tensors must live on a CUDA device")
    return torch.cuda.device(t.device)


def _stream(t: torch.Tensor) -> int:
    return torch.cuda.current_stream(t.device).cuda_stream


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _need(t: torch.Tensor, dtype, name: str) -> torch.Tensor:
    if not t.is_cuda:
        raise NativeError(f"{name} must be a CUDA tensor (memvul_b200 has no CPU path)")
    if t.dtype != dtype or not t.is_contiguous():
        raise ValueError(f"{name} must be contiguous {dtype}, got {t.dtype} contiguous={t.is_contiguous()}")
    return t


# ------------------------------------------------------------------------------- weights
def split3_weight(w: torch.Tensor) -> torch.Tensor:
    """fp32 [N,K] -> fp16 [N,3K] = [hi | hi | lo] with hi = fp16(w), lo = fp16(w - hi): the weight side of the
    split-fp16 accuracy mode (the activation side is [hi | lo | hi], so the K' = 3K product is
    a_hi w_hi + a_lo w_hi + a_hi w_lo)."""
    w = w.to(torch.float32)
    hi = w.to(torch.float16)
    lo = (w - hi.to(torch.float32)).to(torch.float16)
    return torch.cat([hi, hi, lo], dim=1).contiguous()


class PackedBert:
    """Device-resident BERT weights in the layout the kernels read: fp16 [out,in] GEMM kernels with
    query|key|value fused into one [3H,H] matrix, fp32 biases / LayerNorm / embedding tables.
    Built from a ``state_dict`` with HF ``BertModel`` names under ``prefix`` (SURVEY.md 8b)."""

    def __init__(self, sd: Dict[str, torch.Tensor], prefix: str, device: torch.device, ln_eps: float = 1e-12,
                 precise: bool = False):
        def f32(k):
            return sd[prefix + k].detach().to(device=device, dtype=torch.float32).contiguous()

        def f16(t):
            # accuracy mode (MEMVUL_ENC_PRECISE): [N, 3K] = [W_hi | W_hi | W_lo], the K-concatenated split operand that
            # pairs with the activations' [A_hi | A_lo | A_hi] (memvul_b200/csrc/precise.cuh)
            return split3_weight(t) if precise else t.to(torch.float16).contiguous()

        self.device = device
        self.precise = bool(precise)
        self.word = f32("embeddings.word_embeddings.weight")
        self.pos = f32("embeddings.position_embeddings.weight")
        self.type = f32("embeddings.token_type_embeddings.weight")
        self.emb_g = f32("embeddings.LayerNorm.weight")
        self.emb_b = f32("embeddings.LayerNorm.bias")
        self.hidden = self.word.shape[1]
        n_layers = 0
        while (prefix + f"encoder.layer.{n_layers}.attention.self.query.weight") in sd:
            n_layers += 1
        self.layers = n_layers
        self.heads = self.hidden // 64
        self.keep: List[torch.Tensor] = []
        self._layer_arr = (BertLayerC * n_layers)()
        for l in range(n_layers):
            p = f"encoder.layer.{l}."
            wqkv = f16(torch.cat([f32(p + "attention.self.query.weight"), f32(p + "attention.self.key.weight"),
                                  f32(p + "attention.self.value.weight")], 0))
            bqkv = torch.cat([f32(p + "attention.self.query.bias"), f32(p + "attention.self.key.bias"),
                              f32(p + "attention.self.value.bias")], 0).contiguous()
            ts = dict(w_qkv=wqkv, b_qkv=bqkv,
                      w_ao=f16(f32(p + "attention.output.dense.weight")), b_ao=f32(p + "attention.output.dense.bias"),
                      ln1_g=f32(p + "attention.output.LayerNorm.weight"), ln1_b=f32(p + "attention.output.LayerNorm.bias"),
                      w_ff1=f16(f32(p + "intermediate.dense.weight")), b_ff1=f32(p + "intermediate.dense.bias"),
                      w_ff2=f16(f32(p + "output.dense.weight")), b_ff2=f32(p + "output.dense.bias"),
                      ln2_g=f32(p + "output.LayerNorm.weight"), ln2_b=f32(p + "output.LayerNorm.bias"))
            for k, t in ts.items():
                setattr(self._layer_arr[l], k, t.data_ptr())
                self.keep.append(t)
            if l == 0:
                self.intermediate = ts["w_ff1"].shape[0]
        self.c = BertWeightsC(hidden=self.hidden, layers=n_layers, heads=self.heads, intermediate=self.intermediate,
                              vocab=self.word.shape[0], max_pos=self.pos.shape[0], type_vocab=self.type.shape[0],
                              ln_eps=ln_eps, word_emb=self.word.data_ptr(), pos_emb=self.pos.data_ptr(),
                              type_emb=self.type.data_ptr(), emb_ln_g=self.emb_g.data_ptr(),
                              emb_ln_b=self.emb_b.data_ptr(), layer=self._layer_arr)

    def workspace_bytes(self, B: int, S: int, flags: int = 0) -> int:
        return int(lib().memvul_encoder_workspace_bytes(ctypes.byref(self.c), B, S, flags))


# ------------------------------------------------------------------------------- calls
BAD_MASK, BAD_ID = 1, 2          # bits of the deferred error flag


def mask_to_lens(mask: torch.Tensor, with_row_start: bool = False):
    """bool [B,S] -> (lens int32 [B], bad int32 [1]) or, ``with_row_start``, (lens, row_start int32 [B+1], bad).
    ``bad`` bit 0: some mask is not a non-empty prefix mask (read it with the batch's results; no sync here)."""
    _need(mask, torch.bool, "mask")
    B, S = mask.shape
    lens = torch.empty(B, dtype=torch.int32, device=mask.device)
    row_start = torch.empty(B + 1, dtype=torch.int32, device=mask.device) if with_row_start else None
    bad = torch.zeros(1, dtype=torch.int32, device=mask.device)
    with _on(mask):
        _check(lib().memvul_mask_to_lens(mask.data_ptr(), B, S, lens.data_ptr(), _ptr(row_start), bad.data_ptr(),
                                         _stream(mask)))
    return (lens, row_start, bad) if with_row_start else (lens, bad)


def raise_for_flag(flag: int) -> None:
    """Turn the deferred device flag into the errors the reference raises."""
    if flag & BAD_MASK:
        raise ValueError("batch has a mask that is not a non-empty prefix mask (AllenNLP padding masks are)")
    if flag & BAD_ID:
        raise ValueError("token id or type id out of range for the embedding tables "
                         "(torch.embedding raises in the reference; custom_PTM_embedder.py:205 for type ids)")


ENC_CLS_ONLY, ENC_PACKED, ENC_PRECISE = 1, 2, 4


def encoder_flags(w: PackedBert, cls_only: bool, packed: bool) -> int:
    return (ENC_CLS_ONLY if cls_only else 0) | (ENC_PACKED if packed else 0) | (ENC_PRECISE if w.precise else 0)


def encoder_forward(w: PackedBert, token_ids: torch.Tensor, lens: torch.Tensor,
                    type_ids: Optional[torch.Tensor] = None, workspace: Optional[torch.Tensor] = None,
                    out: Optional[torch.Tensor] = None, cls_only: bool = False,
                    row_start: Optional[torch.Tensor] = None, bad: Optional[torch.Tensor] = None) -> torch.Tensor:
    """last_hidden_state fp32 [B,S,H] of HF BertModel for prefix-masked inputs.  ``cls_only``: only row 0 of each
    sequence is the last layer's output (what BertPooler consumes); the last layer skips the other rows.
    ``row_start`` (from ``mask_to_lens(..., with_row_start=True)``) selects the packed var-len execution: padded
    tokens are never computed.  ``bad``: device int32 flag that collects out-of-range ids."""
    _need(token_ids, torch.int64, "token_ids")
    _need(lens, torch.int32, "lens")
    if type_ids is not None:
        _need(type_ids, torch.int64, "type_ids")
    B, S = token_ids.shape
    flags = encoder_flags(w, cls_only, row_start is not None)   # a PackedBert(precise=True) selects the accuracy mode
    need = w.workspace_bytes(B, S, flags)
    if workspace is None or workspace.numel() < need:
        workspace = torch.empty(need, dtype=torch.uint8, device=token_ids.device)   # no initialisation needed (header)
    if out is None:
        out = torch.empty(B, S, w.hidden, dtype=torch.float32, device=token_ids.device)
    with _on(token_ids):
        _check(lib().memvul_encoder_forward(ctypes.byref(w.c), token_ids.data_ptr(), _ptr(type_ids), lens.data_ptr(),
                                            _ptr(row_start), B, S, out.data_ptr(), workspace.data_ptr(),
                                            workspace.numel(), flags, _ptr(bad), _stream(token_ids)))
    return out


def bank_prepare(bank: torch.Tensor, w_proj: torch.Tensor) -> torch.Tensor:
    _need(bank, torch.float32, "bank")
    _need(w_proj, torch.float32, "w_proj")
    G, D = bank.shape
    vterm = torch.empty(G, 2, dtype=torch.float32, device=bank.device)
    with _on(bank):
        _check(lib().memvul_bank_prepare(bank.data_ptr(), w_proj.data_ptr(), G, D, vterm.data_ptr(), _stream(bank)))
    return vterm


def match_flat_layout(cap: int, G: int):
    """Offsets (in 4-byte words) of the sections of the flat result buffer of one shard with room for ``cap`` issue
    reports: [probs cap*G*2 | best_probs cap*2 | best_idx cap (int32 bits)].  One contiguous buffer per shard means
    the sharded path's single all-gather (memvul_b200/dist.py) needs no pack / unpack kernels."""
    o_bp = cap * G * 2
    o_bi = o_bp + cap * 2
    return o_bp, o_bi, o_bi + cap


def pool_match(cls: torch.Tensor, cls_stride: int, B: int, w_pool, b_pool, w_head, b_head, w_proj=None, bank=None,
               vterm=None, same_idx: int = 0, phase_mask: int = PM_ALL, u: Optional[torch.Tensor] = None,
               pooled: Optional[torch.Tensor] = None, flat_capacity: Optional[int] = None, D: Optional[int] = None):
    """Fused pool + header + match.  Returns dict(u, pooled[, logits, probs, best_idx, best_probs]).
    ``flat_capacity``: allocate probs / best_probs / best_idx as views of ONE flat fp32 buffer (``out["_flat"]``) laid
    out by ``match_flat_layout(flat_capacity, G)`` -- what the multi-GPU gather sends as is."""
    dev = w_pool.device
    H = w_pool.shape[0]
    if D is None:
        D = w_head.shape[0] if w_head is not None else (u.shape[1] if u is not None else 4)
    G = 0 if bank is None else bank.shape[0]
    f = dict(dtype=torch.float32, device=dev)
    pooled = torch.empty(B, H, **f) if pooled is None else pooled
    u = torch.empty(B, D, **f) if u is None else u
    out = {"u": u, "pooled": pooled}
    uterm = best_key = logits = probs = best_idx = best_probs = None
    if phase_mask & (PM_UTERM | PM_MATCH | PM_FINAL):
        uterm = torch.empty(B, 2, **f)
        best_key = torch.empty(B, dtype=torch.int64, device=dev)
    if phase_mask & (PM_MATCH | PM_FINAL):
        logits = torch.empty(B, G, 2, **f)
        if flat_capacity is not None:
            cap = max(int(flat_capacity), B)
            o_bp, o_bi, n = match_flat_layout(cap, G)
            flat = torch.empty(n, **f)
            probs = flat[:B * G * 2].view(B, G, 2)
            best_probs = flat[o_bp:o_bp + B * 2].view(B, 2)
            best_idx = flat[o_bi:o_bi + B].view(torch.int32)
            out["_flat"], out["_flat_capacity"] = flat, cap
        else:
            probs = torch.empty(B, G, 2, **f)
            best_idx = torch.empty(B, dtype=torch.int32, device=dev)
            best_probs = torch.empty(B, 2, **f)
        out.update(logits=logits, probs=probs, best_idx=best_idx, best_probs=best_probs)
    with _on(w_pool):
        _check(lib().memvul_pool_match(_ptr(cls), cls_stride, _ptr(w_pool), _ptr(b_pool), _ptr(w_head), _ptr(b_head),
                                       _ptr(w_proj), _ptr(bank), _ptr(vterm), B, G, H, D, same_idx, _ptr(pooled),
                                       _ptr(u), _ptr(uterm), _ptr(best_key), _ptr(logits), _ptr(probs),
                                       _ptr(best_idx), _ptr(best_probs), phase_mask, _stream(w_pool)))
    out["_scratch"] = (uterm, best_key)
    return out


def single_head(feat: torch.Tensor, w_cls: torch.Tensor):
    _need(feat, torch.float32, "feat")
    _need(w_cls, torch.float32, "w_cls")
    B, D = feat.shape
    logits = torch.empty(B, 2, dtype=torch.float32, device=feat.device)
    probs = torch.empty_like(logits)
    with _on(feat):
        _check(lib().memvul_single_head(feat.data_ptr(), w_cls.data_ptr(), B, D, logits.data_ptr(), probs.data_ptr(),
                                        _stream(feat)))
    return logits, probs


# ---- building blocks (tests / profiling) ----
def gemm_f16(a: torch.Tensor, w: torch.Tensor, bias: torch.Tensor, epilogue: int,
             resid: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    _need(a, torch.float16, "a")
    _need(w, torch.float16, "w")
    _need(bias, torch.float32, "bias")
    M, K = a.shape
    N = w.shape[0]
    if out is None:
        out = torch.empty(M, N, dtype=torch.float32 if epilogue in (EPI_BIAS_RESID_F32, EPI_BIAS_F32) else torch.float16,
                          device=a.device)
    with _on(a):
        _check(lib().memvul_gemm_f16(a.data_ptr(), w.data_ptr(), bias.data_ptr(), _ptr(resid), out.data_ptr(), M, N, K,
                                     epilogue, _stream(a)))
    return out


def gemm_ln_f16(a: torch.Tensor, w: torch.Tensor, bias: torch.Tensor, resid: torch.Tensor, gamma: torch.Tensor,
                beta: torch.Tensor, eps: float = 1e-12, inplace: bool = False):
    """Fused LayerNorm(a @ w.T + bias + resid) -> (fp32, fp16); N must be 768."""
    _need(a, torch.float16, "a")
    _need(w, torch.float16, "w")
    _need(resid, torch.float32, "resid")
    M, K = a.shape
    N = w.shape[0]
    x32 = resid if inplace else torch.empty(M, N, dtype=torch.float32, device=a.device)
    x16 = torch.empty(M, N, dtype=torch.float16, device=a.device)
    with _on(a):
        _check(lib().memvul_gemm_ln_f16(a.data_ptr(), w.data_ptr(), bias.data_ptr(), resid.data_ptr(), gamma.data_ptr(),
                                        beta.data_ptr(), eps, x32.data_ptr(), x16.data_ptr(), M, N, K, _stream(a)))
    return x32, x16


def attention_f16(qkv: torch.Tensor, lens: torch.Tensor, B: int, S: int, H: int,
                  row_start: Optional[torch.Tensor] = None) -> torch.Tensor:
    """``row_start`` None: qkv rows are the padded [B*S] layout; else the packed layout (rows row_start[b]..)."""
    _need(qkv, torch.float16, "qkv")
    _need(lens, torch.int32, "lens")
    ctx = torch.zeros(qkv.shape[0], H, dtype=torch.float16, device=qkv.device)
    with _on(qkv):
        _check(lib().memvul_attention_f16(qkv.data_ptr(), lens.data_ptr(), _ptr(row_start), ctx.data_ptr(), B, S, H,
                                          _stream(qkv)))
    return ctx


def attention_f32(qkv: torch.Tensor, lens: torch.Tensor, B: int, S: int, H: int,
                  row_start: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Accuracy-mode attention: qkv fp32 [rows,3H] -> ctx fp32 [rows,H] (same layouts as ``attention_f16``)."""
    _need(qkv, torch.float32, "qkv")
    _need(lens, torch.int32, "lens")
    ctx = torch.zeros(qkv.shape[0], H, dtype=torch.float32, device=qkv.device)
    with _on(qkv):
        _check(lib().memvul_attention_f32(qkv.data_ptr(), lens.data_ptr(), _ptr(row_start), ctx.data_ptr(), B, S, H,
                                          _stream(qkv)))
    return ctx


def split3_f16(x: torch.Tensor, gelu: bool = False) -> torch.Tensor:
    """fp32 [M,K] -> fp16 [M,3K] = [hi | lo | hi] (of gelu_erf(x) when ``gelu``): the activation side of the accuracy mode."""
    _need(x, torch.float32, "x")
    M, K = x.shape
    out = torch.empty(M, 3 * K, dtype=torch.float16, device=x.device)
    with _on(x):
        _check(lib().memvul_split3_f16(x.data_ptr(), out.data_ptr(), M, K, 1 if gelu else 0, _stream(x)))
    return out


def layernorm(y: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, eps: float = 1e-12):
    _need(y, torch.float32, "y")
    M, H = y.shape
    x32 = torch.empty_like(y)
    x16 = torch.empty(M, H, dtype=torch.float16, device=y.device)
    with _on(y):
        _check(lib().memvul_layernorm(y.data_ptr(), gamma.data_ptr(), beta.data_ptr(), eps, x32.data_ptr(),
                                      x16.data_ptr(), M, H, _stream(y)))
    return x32, x16


def embed_layernorm(w: PackedBert, token_ids: torch.Tensor, type_ids: Optional[torch.Tensor] = None,
                    lens: Optional[torch.Tensor] = None, row_start: Optional[torch.Tensor] = None,
                    bad: Optional[torch.Tensor] = None):
    _need(token_ids, torch.int64, "token_ids")
    B, S = token_ids.shape
    x32 = torch.zeros(B * S, w.hidden, dtype=torch.float32, device=token_ids.device)
    x16 = torch.zeros(B * S, w.hidden, dtype=torch.float16, device=token_ids.device)
    with _on(token_ids):
        _check(lib().memvul_embed_layernorm(ctypes.byref(w.c), token_ids.data_ptr(), _ptr(type_ids), _ptr(lens),
                                            _ptr(row_start), B, S, x32.data_ptr(), x16.data_ptr(), _ptr(bad),
                                            _stream(token_ids)))
    return x32, x16


# ---- measurement hooks ----
def launch_count() -> int:
    return int(lib().memvul_launch_count())


def profile_enable(on: bool) -> None:
    _check(lib().memvul_profile_enable(1 if on else 0))


def profile_read() -> Dict[str, Dict[str, float]]:
    """Synchronises the device; {kernel class: {"ms": summed device ms, "launches": n}} since the last read."""
    n = len(KERNEL_CLASSES)
    ms = (ctypes.c_double * n)()
    cnt = (ctypes.c_longlong * n)()
    rc = lib().memvul_profile_read(n, ms, cnt)
    if rc < 0:
        _check(rc)
    return {k: {"ms": ms[i], "launches": int(cnt[i])} for i, k in enumerate(KERNEL_CLASSES)}
