"""Host-side mirror of the reference's vit.h interface on top of the C ABI (include/vitb200.h).

Names and argument meaning follow the reference (vit.h:118-122) so tests read like reference usage:

    model = vit_model_load(path)                      # reference vit.cpp:308  (here: parse + upload to the GPU)
    probs, idx, val = vit_predict(model, images)      # reference vit.cpp:1004 (here: batched, on the GPU)

There is NO CPU fallback: if libvitb200.so is missing or no B200 is present these functions raise.
"""
from __future__ import annotations

import ctypes as C
import os
import re
from typing import Optional

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libvitb200.so")
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "vitb200.h")
_lib = None


class VitB200Error(RuntimeError):
    pass


class Hparams(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("hidden_size", "num_hidden_layers", "num_attention_heads", "num_classes",
                                          "patch_size", "img_size", "ftype")] + [("eps", C.c_float)]


class Taps(C.Structure):
    _fields_ = [("layer", C.c_int32)] + [(n, C.c_void_p) for n in
                                         ("embed", "ln1", "qkv", "attn", "x1", "ln2", "h", "x2", "final_ln", "x_final")]


class Tensor(C.Structure):
    """vitb200_tensor (include/vitb200.h): one host tensor as found in vit_model::tensors (reference vit.h:88)."""
    _fields_ = [("name", C.c_char_p), ("data", C.c_void_p), ("type", C.c_int32), ("n_dims", C.c_int32), ("ne", C.c_int64 * 4)]


def declared_symbols() -> list:
    """Every function name include/vitb200.h declares (for the CPU-side ABI test)."""
    src = open(HEADER_PATH).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(vitb200_[a-z_0-9]+)\s*\(", src)))


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise VitB200Error(f"{LIB_PATH} is missing: build it with ./build.sh (python -c 'import __graft_entry__ as g; "
                               "g.build()'). The vit.cpp_b200 forward path has no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        vp, i32, f32p = C.c_void_p, C.c_int, C.c_void_p
        L.vitb200_last_error.restype = C.c_char_p
        L.vitb200_create_from_file.argtypes = [C.c_char_p, i32, i32, C.POINTER(vp)]
        L.vitb200_create_from_file_ex.argtypes = [C.c_char_p, i32, i32, i32, C.POINTER(vp)]
        L.vitb200_create_ex.argtypes = [vp, vp, i32, i32, i32, i32, C.POINTER(vp)]
        L.vitb200_in_chans.argtypes = [vp]
        L.vitb200_head_tokens.argtypes = [vp]
        L.vitb200_create.argtypes = [vp, vp, i32, i32, i32, C.POINTER(vp)]
        L.vitb200_destroy.argtypes = [vp]
        L.vitb200_destroy.restype = None
        L.vitb200_get_hparams.argtypes = [vp, C.POINTER(Hparams)]
        L.vitb200_label.argtypes = [vp, i32]
        L.vitb200_label.restype = C.c_char_p
        L.vitb200_forward.argtypes = [vp, f32p, i32, f32p, f32p, vp, f32p, i32]
        L.vitb200_forward_async.argtypes = [vp, f32p, i32, f32p, f32p, vp, f32p, i32]
        L.vitb200_sync.argtypes = [vp]
        L.vitb200_profile_enable.argtypes = [vp, i32]
        L.vitb200_profile_read.argtypes = [vp, i32, C.POINTER(C.c_double), C.POINTER(C.c_int), C.POINTER(C.c_double)]
        L.vitb200_forward_sharded.argtypes = [vp, i32, f32p, i32, f32p, f32p, vp, f32p, i32]
        L.vitb200_forward_u8.argtypes = [vp, vp, vp, vp, i32, i32, vp, vp, vp, vp, vp, i32]
        L.vitb200_forward_u8_async.argtypes = [vp, vp, vp, vp, i32, i32, vp, vp, vp, vp, i32]
        L.vitb200_forward_device.argtypes = [vp, vp, i32, vp, vp, vp, vp, i32, vp]
        L.vitb200_last_launch_count.argtypes = [vp]
        L.vitb200_stream.argtypes = [vp]
        L.vitb200_stream.restype = vp
        L.vitb200_forward_debug.argtypes = [vp, f32p, i32, f32p, f32p, C.POINTER(Taps)]
        L.vitb200_test_gemm.argtypes = [i32, i32, i32, i32, i32, vp, vp, vp, vp, vp]
        L.vitb200_test_dequant.argtypes = [i32, vp, C.c_int64, vp]
        L.vitb200_test_gemm_q8.argtypes = [i32, i32, i32, i32, vp, vp, vp, vp, vp, vp, i32, vp]
        L.vitb200_test_layernorm.argtypes = [i32, i32, i32, vp, vp, vp, C.c_float, vp]
        L.vitb200_test_softmax_topk.argtypes = [i32, i32, i32, i32, vp, i32, vp, vp, vp]
        L.vitb200_test_attention.argtypes = [i32, i32, i32, i32, i32, vp, vp]
        L.vitb200_test_attention_hilo.argtypes = [i32, i32, i32, i32, vp, vp, vp]
        _lib = L
    return _lib


def _check(rc: int, what: str):
    if rc != 0:
        raise VitB200Error(f"{what}: {lib().vitb200_last_error().decode()}")


class VitModel:
    """vit_model + vit_state of the reference (vit.h:72-89), living on one GPU."""

    def __init__(self, handle, device: int, max_batch: int):
        self._h = handle
        self.device = device
        self.max_batch = max_batch
        hp = Hparams()
        _check(lib().vitb200_get_hparams(self._h, C.byref(hp)), "vitb200_get_hparams")
        self.hparams = hp
        self.hidden_size, self.num_classes, self.img_size = hp.hidden_size, hp.num_classes, hp.img_size
        self.n_tokens = (hp.img_size // hp.patch_size) ** 2 + 1
        self.in_chans = lib().vitb200_in_chans(self._h)        # 3, or 1 for a ViTSTR model (vitstr.cpp:713)
        self.head_tokens = lib().vitb200_head_tokens(self._h)  # classifier rows per image (1, or 25 for ViTSTR)

    def label(self, i: int) -> Optional[str]:
        s = lib().vitb200_label(self._h, i)
        return s.decode() if s else None

    @property
    def handle(self):
        return self._h

    def last_launch_count(self) -> int:
        return lib().vitb200_last_launch_count(self._h)

    def close(self):
        if self._h:
            lib().vitb200_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def vit_model_load(fname: str, device: int = 0, max_batch: int = 256, head_tokens: int = 1) -> VitModel:
    """reference: bool vit_model_load(const std::string &fname, vit_model &model)  (vit.cpp:308).  head_tokens = 25 loads a
    ViTSTR model (reference extensions/vitstr.cpp: 1-channel input, classifier over the first 25 tokens)."""
    h = C.c_void_p()
    _check(lib().vitb200_create_from_file_ex(fname.encode(), device, max_batch, head_tokens, C.byref(h)), "vit_model_load")
    return VitModel(h, device, max_batch)


def vit_model_from_tensors(vf, device: int = 0, max_batch: int = 8, head_tokens: int = 1, edit=None) -> VitModel:
    """vitb200_create_ex with a caller-built tensor list -- what the vit.h-side shim does with vit_model::tensors.  `vf` is a parsed
    model file (ggml_file.VitFile: numpy-shaped f32 / f16 arrays); `edit(entries)` may reorder / duplicate / reshape the list of
    [name, array, ggml_type, ne] entries first (tests of the loader's shape and name checks)."""
    entries = []
    for name, arr in vf.tensors.items():
        if name.endswith(".q8_0_raw"):
            continue
        ft = vf.tensor_ftype[name]
        if ft not in (0, 1):
            raise VitB200Error("vit_model_from_tensors: f32 / f16 tensors only")
        a = np.ascontiguousarray(arr, np.float16 if ft == 1 else np.float32)
        if name == "patch_embed.proj.bias":
            a = a.reshape(1, a.size, 1, 1)  # convert-pth-to-ggml.py:150-151
        entries.append([name, a, ft, list(reversed(a.shape))])
    if edit is not None:
        entries = edit(entries) or entries
    ts = (Tensor * len(entries))()
    keep = []
    for t, (name, a, ft, ne) in zip(ts, entries):
        nm = name.encode()
        keep.append((nm, a))
        t.name, t.data, t.type, t.n_dims = nm, a.ctypes.data, ft, len(ne)
        for i in range(4):
            t.ne[i] = ne[i] if i < len(ne) else 1
    hp = Hparams(vf.hidden_size, vf.num_hidden_layers, vf.num_attention_heads, vf.num_classes, vf.patch_size, vf.img_size, vf.ftype, 1e-6)
    h = C.c_void_p()
    _check(lib().vitb200_create_ex(C.byref(hp), ts, len(entries), device, max_batch, head_tokens, C.byref(h)), "vitb200_create")
    return VitModel(h, device, max_batch)


def vit_predict(model: VitModel, images: np.ndarray, topk: int = 5, want_logits: bool = False):
    """Batched reference vit_predict (vit.cpp:1004): images float32[B,S,S,3] (image_f32 layout) on the HOST.
    Returns (probs[B,C], topk_idx[B,k], topk_prob[B,k]) (+ logits[B,C] if want_logits).  For a ViTSTR model (head_tokens = n,
    images float32[B,S,S] or [B,S,S,1]) every output gains a token axis: probs[B,n,C], topk[B,n,k]."""
    imgs = np.ascontiguousarray(images, dtype=np.float32)
    ch = model.in_chans
    if imgs.ndim == (3 if ch == 3 else 2):
        imgs = imgs[None]
    B = imgs.shape[0]
    assert imgs.size == B * model.img_size * model.img_size * ch, imgs.shape
    lead = (B,) if model.head_tokens == 1 else (B, model.head_tokens)
    probs = np.empty(lead + (model.num_classes,), np.float32)
    logits = np.empty(lead + (model.num_classes,), np.float32) if want_logits else None
    idx = np.empty(lead + (topk,), np.int32)
    val = np.empty(lead + (topk,), np.float32)
    _check(lib().vitb200_forward(model.handle, imgs.ctypes.data, B, probs.ctypes.data,
                                 logits.ctypes.data if want_logits else None, idx.ctypes.data, val.ctypes.data, topk),
           "vit_predict")
    return (probs, idx, val, logits) if want_logits else (probs, idx, val)


def vit_predict_sharded(models, images: np.ndarray, topk: int = 5):
    """Data-parallel batched vit_predict over several VitModel engines (one per GPU) from one host thread.  Output shapes follow
    vit_predict: a ViTSTR model (head_tokens = n) returns probs[B,n,C], topk[B,n,k]; all engines must hold the same model."""
    imgs = np.ascontiguousarray(images, dtype=np.float32)
    B = imgs.shape[0]
    nc, ht = models[0].num_classes, models[0].head_tokens
    if any(m.head_tokens != ht or m.num_classes != nc or m.in_chans != models[0].in_chans for m in models):
        raise VitB200Error("vit_predict_sharded: the engines hold different models")
    assert imgs.size == B * models[0].img_size * models[0].img_size * models[0].in_chans, imgs.shape
    lead = (B,) if ht == 1 else (B, ht)
    probs = np.empty(lead + (nc,), np.float32)
    idx = np.empty(lead + (topk,), np.int32)
    val = np.empty(lead + (topk,), np.float32)
    hs = (C.c_void_p * len(models))(*[m.handle for m in models])
    _check(lib().vitb200_forward_sharded(hs, len(models), imgs.ctypes.data, B, probs.ctypes.data, None, idx.ctypes.data,
                                         val.ctypes.data, topk), "vit_predict_sharded")
    return probs, idx, val


def vit_predict_sharded_async(models, images: np.ndarray, probs: np.ndarray, idx: np.ndarray, val: np.ndarray):
    """Pipelined vit_predict_sharded (vitb200_forward_sharded_async): enqueues the global batch over the engines and returns; the
    caller-owned `images` / output arrays (C-contiguous, shapes as vit_predict_sharded returns them) must stay alive and untouched
    until sync_all(models).  Lets one host thread keep several global batches in flight (two pipeline slots per engine)."""
    B = images.shape[0]
    if images.dtype != np.float32 or not images.flags.c_contiguous:
        raise ValueError("images must be a C-contiguous float32 array")
    for a, dt in ((probs, np.float32), (idx, np.int32), (val, np.float32)):
        if a.dtype != dt or not a.flags.c_contiguous or a.shape[0] != B:
            raise ValueError("output arrays must be C-contiguous, one leading row per image")
    hs = (C.c_void_p * len(models))(*[m.handle for m in models])
    L = lib()
    L.vitb200_forward_sharded_async.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
    _check(L.vitb200_forward_sharded_async(hs, len(models), images.ctypes.data, B, probs.ctypes.data, None, idx.ctypes.data,
                                           val.ctypes.data, idx.shape[-1]), "vit_predict_sharded_async")


def sync_all(models):
    hs = (C.c_void_p * len(models))(*[m.handle for m in models])
    L = lib()
    L.vitb200_sync_all.argtypes = [C.c_void_p, C.c_int]
    _check(L.vitb200_sync_all(hs, len(models)), "vitb200_sync_all")


def vit_image_preprocess_predict(model: VitModel, images_u8, bilinear: bool = False, topk: int = 5, predict: bool = True):
    """reference vit_image_preprocess (vit.cpp:289) + vit_predict on the GPU for a list of HxWx3 uint8 RGB arrays of any size.
    Returns (image_f32 batch [B,S,S,3], probs, topk_idx, topk_prob, logits); the last four are None if predict is False."""
    imgs = [np.ascontiguousarray(a, dtype=np.uint8) for a in images_u8]
    B = len(imgs)
    ptrs = (C.c_void_p * B)(*[a.ctypes.data for a in imgs])
    nx = (C.c_int * B)(*[a.shape[1] for a in imgs])
    ny = (C.c_int * B)(*[a.shape[0] for a in imgs])
    S = model.img_size
    f32 = np.empty((B, S, S, 3), np.float32)
    probs = np.empty((B, model.num_classes), np.float32) if predict else None
    logits = np.empty((B, model.num_classes), np.float32) if predict else None
    idx = np.empty((B, topk), np.int32) if predict else None
    val = np.empty((B, topk), np.float32) if predict else None
    _check(lib().vitb200_forward_u8(model.handle, ptrs, nx, ny, B, int(bilinear), f32.ctypes.data,
                                    probs.ctypes.data if predict else None, logits.ctypes.data if predict else None,
                                    idx.ctypes.data if predict else None, val.ctypes.data if predict else None, topk if predict else 0),
           "vit_image_preprocess")
    return f32, probs, idx, val, logits


TAP_SHAPES = {
    "embed": lambda B, N, D: (B, N, D), "ln1": lambda B, N, D: (B, N, D), "qkv": lambda B, N, D: (B, N, 3 * D),
    "attn": lambda B, N, D: (B, N, D), "x1": lambda B, N, D: (B, N, D), "ln2": lambda B, N, D: (B, N, D),
    "h": lambda B, N, D: (B, N, 4 * D), "x2": lambda B, N, D: (B, N, D), "final_ln": lambda B, N, D: (B, D),
    "x_final": lambda B, N, D: (B, N, D),
}


def vit_predict_debug(model: VitModel, images: np.ndarray, tap_layer: int, taps=tuple(TAP_SHAPES)):
    """Forward with intermediates copied back (tests only)."""
    imgs = np.ascontiguousarray(images, dtype=np.float32)
    B = imgs.shape[0]
    probs = np.empty((B, model.num_classes), np.float32)
    logits = np.empty((B, model.num_classes), np.float32)
    tp = Taps()
    tp.layer = tap_layer
    out = {}
    for n in taps:
        out[n] = np.zeros(TAP_SHAPES[n](B, model.n_tokens, model.hidden_size), np.float32)
        setattr(tp, n, out[n].ctypes.data)
    _check(lib().vitb200_forward_debug(model.handle, imgs.ctypes.data, B, probs.ctypes.data, logits.ctypes.data,
                                       C.byref(tp)), "vit_predict_debug")
    return probs, logits, out


ATTN_AUTO, ATTN_MMA, ATTN_TC, ATTN_TC_LONG = 0, 1, 2, 3


def test_attention(qkv16: np.ndarray, B: int, N: int, H: int, kernel: int = ATTN_AUTO, device: int = 0) -> np.ndarray:
    """Stand-alone attention kernel: qkv16 float16 [B*N, 3*H*64] -> float32 [B*N, H*64]."""
    q = np.ascontiguousarray(qkv16, np.float16).reshape(B * N, 3 * H * 64)
    out = np.empty((B * N, H * 64), np.float32)
    _check(lib().vitb200_test_attention(device, kernel, B, N, H, q.ctypes.data, out.ctypes.data), "vitb200_test_attention")
    return out


def split_hi_lo(x: np.ndarray):
    """x (float32) -> (hi, lo) float16 with hi = f16(x), lo = f16(x - hi): what the qkv GEMM's split-precision epilogue stores."""
    x = np.ascontiguousarray(x, np.float32)
    hi = x.astype(np.float16)
    lo = (x - hi.astype(np.float32)).astype(np.float16)
    return hi, lo


def test_attention_hilo(qkv32: np.ndarray, B: int, N: int, H: int, device: int = 0) -> np.ndarray:
    """The tcgen05 attention kernel (N <= 224) on split-precision operands: qkv32 float32 [B*N, 3*H*64] is passed as hi + lo."""
    hi, lo = split_hi_lo(np.asarray(qkv32, np.float32).reshape(B * N, 3 * H * 64))
    out = np.empty((B * N, H * 64), np.float32)
    _check(lib().vitb200_test_attention_hilo(device, B, N, H, hi.ctypes.data, lo.ctypes.data, out.ctypes.data),
           "vitb200_test_attention_hilo")
    return out


def test_dequant(ggml_type: int, blocks: np.ndarray) -> np.ndarray:
    """Host-only: the engine's upload-time conversion of quantised blocks -> float16[n_blocks*32]."""
    from .ggml_file import QUANT_BLOCK_BYTES
    raw = np.ascontiguousarray(blocks, np.uint8).reshape(-1)
    nb = raw.size // QUANT_BLOCK_BYTES[ggml_type]
    out = np.empty(nb * 32, np.uint16)
    _check(lib().vitb200_test_dequant(ggml_type, raw.ctypes.data, nb, out.ctypes.data), "vitb200_test_dequant")
    return out.view(np.float16)


def test_gemm(M: int, N: int, K: int, epilogue: int, A16: np.ndarray, W16: np.ndarray, bias: np.ndarray,
              resid: Optional[np.ndarray] = None, device: int = 0) -> np.ndarray:
    A = np.ascontiguousarray(A16, np.float16)
    W = np.ascontiguousarray(W16, np.float16)
    b = np.ascontiguousarray(bias, np.float32)
    r = np.ascontiguousarray(resid, np.float32) if resid is not None else None
    out = np.empty((M, N), np.float32)
    _check(lib().vitb200_test_gemm(device, M, N, K, epilogue, A.ctypes.data, W.ctypes.data, b.ctypes.data,
                                   r.ctypes.data if r is not None else None, out.ctypes.data), "vitb200_test_gemm")
    return out


def test_gemm_q8(x, w_blocks, bias, device: int = 0, iters: int = 0):
    """The q8_0 linear layer on the integer tensor cores (vitb200_test_gemm_q8): x float32 [M][K], w_blocks = uint8 bytes of a q8_0
    tensor [N][K/32] blocks (model-file layout), bias [N].  Returns (y [M][N] f32, xq [M][K] int8, xd [M][K/32] f32, ms per launch or None)."""
    x = np.ascontiguousarray(x, np.float32)
    w = np.ascontiguousarray(w_blocks, np.uint8)
    b = np.ascontiguousarray(bias, np.float32)
    M, K = x.shape
    N = b.shape[0]
    if w.size != N * (K // 32) * 34:
        raise ValueError("w_blocks does not hold N * K / 32 q8_0 blocks")
    y = np.empty((M, N), np.float32)
    xq = np.empty((M, K), np.int8)
    xd = np.empty((M, K // 32), np.float32)
    ms = C.c_float(0.0)
    _check(lib().vitb200_test_gemm_q8(device, M, N, K, x.ctypes.data, w.ctypes.data, b.ctypes.data, y.ctypes.data, xq.ctypes.data,
                                      xd.ctypes.data, iters, C.cast(C.pointer(ms), C.c_void_p)), "vitb200_test_gemm_q8")
    return y, xq, xd, (ms.value if iters > 0 else None)


def test_layernorm(x, w, b, eps: float = 1e-6, device: int = 0):
    """The block LayerNorm kernel alone (vitb200_test_layernorm): x float32 [rows][D] -> float32 [rows][D] (f16 values widened)."""
    x = np.ascontiguousarray(x, np.float32)
    w = np.ascontiguousarray(w, np.float32)
    b = np.ascontiguousarray(b, np.float32)
    y = np.empty_like(x)
    _check(lib().vitb200_test_layernorm(device, x.shape[0], x.shape[1], x.ctypes.data, w.ctypes.data, b.ctypes.data, eps, y.ctypes.data),
           "vitb200_test_layernorm")
    return y


def test_softmax_topk(logits, C: int, k: int, device: int = 0):
    """The final soft-max + top-k kernel alone (vitb200_test_softmax_topk): logits float32 [R][ldl] with ldl >= C (only the first C
    columns are read).  Returns (probs [R][C] f32, idx [R][k] int32, val [R][k] f32)."""
    lg = np.ascontiguousarray(logits, np.float32)
    R, ldl = lg.shape
    probs = np.empty((R, C), np.float32)
    idx = np.empty((R, k), np.int32)
    val = np.empty((R, k), np.float32)
    _check(lib().vitb200_test_softmax_topk(device, R, C, ldl, lg.ctypes.data, k, probs.ctypes.data, idx.ctypes.data, val.ctypes.data),
           "vitb200_test_softmax_topk")
    return probs, idx, val
