"""ctypes wrapper around oracle/libvitoracle.so (oracle/vit_oracle.c, our plain-C restatement of the
reference forward path).  TEST INFRASTRUCTURE: only tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline leg may import this."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libvitoracle.so")
_lib = None


def build(force: bool = False) -> None:
    src = os.path.join(_HERE, "vit_oracle.c")
    if force or not os.path.exists(LIB_PATH) or os.path.getmtime(LIB_PATH) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", _HERE, "restatement"], stdout=subprocess.DEVNULL)


class _Taps(C.Structure):
    _fields_ = [("layer", C.c_int)] + [(n, C.c_void_p) for n in
                                       ("embed", "ln1", "qkv", "attn", "x1", "ln2", "h", "x2", "final_ln", "x_final")]


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(LIB_PATH)
        L.vo_create.restype = C.c_void_p
        L.vo_create.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.vo_create_ex.restype = C.c_void_p
        L.vo_create_ex.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int]
        L.vo_destroy.argtypes = [C.c_void_p]
        L.vo_forward.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.vo_round_f16.argtypes = [C.c_void_p, C.c_void_p, C.c_int64]
        L.vo_gelu_table.argtypes = [C.c_void_p, C.c_void_p, C.c_int64]
        L.vo_exp_table.argtypes = [C.c_void_p, C.c_void_p, C.c_int64]
        L.vo_softmax_rows.argtypes = [C.c_void_p, C.c_int, C.c_int]
        L.vo_layernorm.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_float, C.c_void_p]
        L.vo_set_threads.argtypes = [C.c_int]
        L.vo_linear_q8_0.argtypes = [C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        _lib = L
    return _lib


class OracleModel:
    """The restatement's model, built from a parsed legacy-ggml file (ggml_file.VitFile)."""

    TAP_NAMES = ("embed", "ln1", "qkv", "attn", "x1", "ln2", "h", "x2", "final_ln", "x_final")

    def __init__(self, vf, tensor_specs, head_tokens: int = 1):
        """head_tokens = 25 restates the ViTSTR extension (its channel count comes from the patch kernel's shape)."""
        self.vf = vf
        self.in_chans = int(vf.tensors["patch_embed.proj.weight"].shape[1])
        self.head_tokens = head_tokens
        specs = tensor_specs(vf.hidden_size, vf.num_hidden_layers, vf.num_classes, vf.patch_size, vf.img_size, self.in_chans)
        self._keep = []
        ptrs = (C.c_void_p * len(specs))()
        types = (C.c_int32 * len(specs))()
        for i, (name, _shape, _is_mat) in enumerate(specs):
            ft = vf.tensor_ftype[name]
            arr = vf.tensors[name + ".q8_0_raw"] if ft == 8 else vf.tensors[name]
            arr = np.ascontiguousarray(arr)
            self._keep.append(arr)
            ptrs[i] = arr.ctypes.data
            types[i] = ft
        hp = (C.c_int32 * 6)(vf.hidden_size, vf.num_hidden_layers, vf.num_attention_heads, vf.num_classes,
                             vf.patch_size, vf.img_size)
        self._h = lib().vo_create_ex(hp, ptrs, types, self.in_chans, head_tokens)
        self.classes = vf.num_classes
        self.D = vf.hidden_size
        self.N = vf.n_tokens

    def forward(self, img_hwc: np.ndarray, tap_layer: int | None = None, taps=()):
        """Returns (probs, logits[, {tap: array}])."""
        img = np.ascontiguousarray(img_hwc, np.float32)
        shape = (self.classes,) if self.head_tokens == 1 else (self.head_tokens, self.classes)
        logits = np.empty(shape, np.float32)
        probs = np.empty(shape, np.float32)
        tp = None
        out = {}
        if taps:
            tp = _Taps()
            tp.layer = -1 if tap_layer is None else tap_layer
            shapes = {"embed": (self.N, self.D), "ln1": (self.N, self.D), "qkv": (self.N, 3 * self.D),
                      "attn": (self.N, self.D), "x1": (self.N, self.D), "ln2": (self.N, self.D),
                      "h": (self.N, 4 * self.D), "x2": (self.N, self.D), "final_ln": (self.D,),
                      "x_final": (self.N, self.D)}
            for n in taps:
                out[n] = np.zeros(shapes[n], np.float32)
                setattr(tp, n, out[n].ctypes.data)
        rc = lib().vo_forward(self._h, img.ctypes.data, logits.ctypes.data, probs.ctypes.data,
                              C.byref(tp) if tp is not None else None)
        assert rc == 0
        return (probs, logits, out) if taps else (probs, logits)

    def forward_batch(self, imgs: np.ndarray):
        ps, ls = zip(*(self.forward(imgs[i]) for i in range(imgs.shape[0])))
        return np.stack(ps), np.stack(ls)

    def close(self):
        if self._h:
            lib().vo_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def set_threads(n: int) -> None:
    lib().vo_set_threads(n)


def _unary(fn, x):
    x = np.ascontiguousarray(x, np.float32)
    y = np.empty_like(x)
    fn(x.ctypes.data, y.ctypes.data, x.size)
    return y


def round_f16(x):
    return _unary(lib().vo_round_f16, x)


def gelu_table(x):
    return _unary(lib().vo_gelu_table, x)


def exp_table(x):
    return _unary(lib().vo_exp_table, x)


def softmax_rows(x):
    y = np.ascontiguousarray(x, np.float32).copy()
    lib().vo_softmax_rows(y.ctypes.data, y.shape[0], y.shape[1])
    return y


def layernorm(x, w, b, eps=1e-6):
    x = np.ascontiguousarray(x, np.float32)
    w = np.ascontiguousarray(w, np.float32)
    b = np.ascontiguousarray(b, np.float32)
    y = np.empty_like(x)
    lib().vo_layernorm(x.ctypes.data, x.shape[0], x.shape[1], w.ctypes.data, b.ctypes.data, eps, y.ctypes.data)
    return y


def linear_q8_0(x, w_blocks, bias):
    """One q8_0 linear layer with the reference's arithmetic: x [T][K] f32, w_blocks = uint8 [N][K/32][34] (block_q8_0 as stored
    in a model file), bias [N].  Returns (y [T][N] f32, xq [T][K] int8, xd [T][K/32] f32 -- the quantised activation rows)."""
    x = np.ascontiguousarray(x, np.float32)
    w_blocks = np.ascontiguousarray(w_blocks, np.uint8)
    bias = np.ascontiguousarray(bias, np.float32)
    T, K = x.shape
    N = bias.shape[0]
    assert w_blocks.size == N * (K // 32) * 34
    y = np.empty((T, N), np.float32)
    xq = np.empty((T, K), np.int8)
    xd = np.empty((T, K // 32), np.float32)
    lib().vo_linear_q8_0(T, N, K, w_blocks.ctypes.data, bias.ctypes.data, x.ctypes.data, y.ctypes.data, xd.ctypes.data, xq.ctypes.data)
    return y, xq, xd


def preprocess_levels(rgb_u8, S: int, bilinear: bool = False):
    """numpy restatement of vit_image_preprocess's resize (reference vit.cpp:130-287) up to the u8 levels it rounds to before
    normalising: HxWx3 uint8 -> SxSx3 uint8.  Same sampling positions, taps and float32 roundings as the reference, but without the
    fused multiply-adds its compiled build contains, so an occasional level differs by one: the preprocess fixture stores the
    reference's levels as a residual against this prediction, which keeps it small (tests/golden/make_golden_ref.py)."""
    img = np.asarray(rgb_u8, np.uint8).astype(np.float32)
    ny, nx = img.shape[:2]
    f32 = np.float32
    j = np.arange(S, dtype=np.float32)
    if bilinear:
        xs_, ys_ = f32(nx) / f32(S), f32(ny) / f32(S)
        sx, sy = (j + f32(0.5)) * xs_ - f32(0.5), (j + f32(0.5)) * ys_ - f32(0.5)
        x0, y0 = np.maximum(0, np.floor(sx).astype(np.int64)), np.maximum(0, np.floor(sy).astype(np.int64))
        x1, y1 = np.minimum(x0 + 1, nx - 1), np.minimum(y0 + 1, ny - 1)
        dx, dy = (sx - x0.astype(np.float32))[None, :, None], (sy - y0.astype(np.float32))[:, None, None]
        v0 = img[y0][:, x0] * (f32(1) - dx) + img[y0][:, x1] * dx
        v1 = img[y1][:, x0] * (f32(1) - dx) + img[y1][:, x1] * dx
        v = v0 * (f32(1) - dy) + v1 * dy
    else:
        def cubic(p0, p1, p2, p3, t):
            d0, d2, d3 = (p0 - p1).astype(np.float64), (p2 - p1).astype(np.float64), (p3 - p1).astype(np.float64)
            a1 = (-1.0 / 3 * d0 + d2 - 1.0 / 6 * d3).astype(np.float32)
            a2 = (1.0 / 2 * d0 + 1.0 / 2 * d2).astype(np.float32)
            a3 = (-1.0 / 6 * d0 - 1.0 / 2 * d2 + 1.0 / 6 * d3).astype(np.float32)
            return p1 + a1 * t + a2 * t * t + a3 * t * t * t
        tx, ty = f32(nx) / f32(S), f32(ny) / f32(S)
        fx, fy = tx * j, ty * j
        x, y = fx.astype(np.int64), fy.astype(np.int64)
        dx, dy = (fx - x.astype(np.float32))[None, :, None], (fy - y.astype(np.float32))[:, None, None]
        cols = [np.clip(x + o, 0, nx - 1) for o in (-1, 0, 1, 2)]
        rows = [img[np.clip(y + o, 0, ny - 1)] for o in (-1, 0, 1, 2)]          # [S][nx][3] each
        C = [cubic(*(r[:, c] for c in cols), dx) for r in rows]
        v = cubic(*C, dy)
    r = np.sign(v) * np.floor(np.abs(v) + f32(0.5))                            # roundf: half away from zero
    return np.clip(r, 0, 255).astype(np.uint8)
