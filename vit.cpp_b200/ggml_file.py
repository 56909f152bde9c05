"""Legacy-ggml ViT model files (the reference's ".gguf" files are NOT GGUF).

Writer + reader for the container that reference ``convert-pth-to-ggml.py:105-158`` emits and
reference ``vit.cpp:308-712`` (``vit_model_load``) parses:

    int32 magic 0x67676d6c ("ggml", ggml.h:211)
    int32 hidden_size, num_hidden_layers, num_attention_heads, num_classes, patch_size, img_size, ftype
    int32 n_labels ; n_labels x { int32 id, int32 len, bytes }
    per tensor: int32 n_dims, int32 name_len, int32 ftype(0=f32,1=f16,2=q4_0,3=q4_1,6=q5_0,7=q5_1,8=q8_0) ;
                n_dims x int32 ne (reversed numpy shape) ; name ; raw data

There are no real timm weights in this environment (no network, no timm), so ``write_synthetic``
generates a seeded random model with the tensor names / shapes / dtypes of a timm
``VisionTransformer.state_dict()`` (recipe from SURVEY.md 8c: well separated top-5 logits).
The product loader is the C++ one in csrc/model_file.cpp; this module is host-side tooling for
tests and bench.py only.
"""
from __future__ import annotations

import struct
from dataclasses import dataclass, field
from typing import Dict, Tuple

import numpy as np

GGML_FILE_MAGIC = 0x67676D6C
QK8_0 = 32  # ggml-quants.h:42-46 block_q8_0 { f16 d; int8 qs[32]; }

CONFIGS = {
    # name: (hidden, layers, heads, patch, img)
    "tiny": (192, 12, 3, 16, 224),
    "small": (384, 12, 6, 16, 224),
    "base": (768, 12, 12, 16, 224),
    "large384": (1024, 24, 16, 16, 384),
    # small shapes for fast unit tests (not reference configs)
    "micro": (128, 2, 2, 16, 64),
    "micro14": (128, 2, 2, 14, 56),
    # ViT-L/16-384 geometry (hidden 1024, 16 heads, 577 tokens) cut to 2 layers so CPU-side checks stay fast
    "large384x2": (1024, 2, 16, 16, 384),
    # ViTSTR extension (reference extensions/vitstr.cpp): 1-channel 224x224 input, 96 classes, classifier over 25 tokens
    "vitstr_micro": (128, 2, 2, 16, 96),
    "vitstr_tiny": (192, 12, 3, 16, 224),
}
IN_CHANS = {"vitstr_micro": 1, "vitstr_tiny": 1}      # default 3
NUM_CLASSES = {"vitstr_micro": 96, "vitstr_tiny": 96}  # default 1000


@dataclass
class VitFile:
    hidden_size: int
    num_hidden_layers: int
    num_attention_heads: int
    num_classes: int
    patch_size: int
    img_size: int
    ftype: int
    id2label: Dict[int, str] = field(default_factory=dict)
    tensors: Dict[str, np.ndarray] = field(default_factory=dict)  # numpy-shaped (timm order)
    tensor_ftype: Dict[str, int] = field(default_factory=dict)

    @property
    def n_tokens(self) -> int:
        g = self.img_size // self.patch_size
        return g * g + 1


def tensor_specs(hidden: int, layers: int, classes: int, patch: int, img: int, in_chans: int = 3):
    """(name, numpy shape, is_matrix) in timm state_dict order (convert-pth-to-ggml.py:126-139)."""
    n_tok = (img // patch) ** 2 + 1
    specs = [
        ("cls_token", (1, 1, hidden), False),
        ("pos_embed", (1, n_tok, hidden), False),
        ("patch_embed.proj.weight", (hidden, in_chans, patch, patch), True),
        ("patch_embed.proj.bias", (hidden,), False),
    ]
    for i in range(layers):
        p = f"blocks.{i}."
        specs += [
            (p + "norm1.weight", (hidden,), False),
            (p + "norm1.bias", (hidden,), False),
            (p + "attn.qkv.weight", (3 * hidden, hidden), True),
            (p + "attn.qkv.bias", (3 * hidden,), False),
            (p + "attn.proj.weight", (hidden, hidden), True),
            (p + "attn.proj.bias", (hidden,), False),
            (p + "norm2.weight", (hidden,), False),
            (p + "norm2.bias", (hidden,), False),
            (p + "mlp.fc1.weight", (4 * hidden, hidden), True),
            (p + "mlp.fc1.bias", (4 * hidden,), False),
            (p + "mlp.fc2.weight", (hidden, 4 * hidden), True),
            (p + "mlp.fc2.bias", (hidden,), False),
        ]
    specs += [
        ("norm.weight", (hidden,), False),
        ("norm.bias", (hidden,), False),
        ("head.weight", (classes, hidden), True),
        ("head.bias", (classes,), False),
    ]
    return specs


def synth_tensors(hidden, layers, classes, patch, img, seed=0, round_bf16=False, in_chans=3):
    """Seeded synthetic weights (SURVEY.md 8c recipe)."""
    rng = np.random.default_rng(seed)
    out = {}
    for name, shape, is_mat in tensor_specs(hidden, layers, classes, patch, img, in_chans):
        if name == "head.weight":
            w = rng.normal(0.0, 0.2, shape)
        elif name.endswith("norm1.weight") or name.endswith("norm2.weight") or name == "norm.weight":
            w = 1.0 + rng.normal(0.0, 0.02, shape)
        elif is_mat and name.startswith("blocks."):
            w = rng.normal(0.0, 0.05, shape)
        else:
            w = rng.normal(0.0, 0.02, shape)
        w = w.astype(np.float32)
        if round_bf16 and is_mat and name != "patch_embed.proj.weight":
            u = w.view(np.uint32).astype(np.uint64)
            u = ((u + 0x7FFF + ((u >> 16) & 1)) >> 16) << 16  # RNE to bf16
            w = u.astype(np.uint32).view(np.float32)
        out[name] = w
    return out


def _write_header(f, hp: Tuple[int, ...], ftype: int, classes: int):
    hidden, layers, heads, patch, img = hp
    f.write(struct.pack("i", GGML_FILE_MAGIC))
    for v in (hidden, layers, heads, classes, patch, img):
        f.write(struct.pack("i", v))
    f.write(struct.pack("i", ftype))
    f.write(struct.pack("i", classes))
    for i in range(classes):
        s = f"LABEL_{i}".encode()
        f.write(struct.pack("i", i))
        f.write(struct.pack("i", len(s)))
        f.write(s)


def write_synthetic(path: str, config="tiny", ftype: int = 1, classes: int = 0, seed: int = 0,
                    round_bf16: bool = False, in_chans: int = 0) -> None:
    """Write a synthetic model.  ftype 1: 2-D(+4-D) weights f16, rest f32 (convert-pth-to-ggml.py:143-147).
    ftype 0: everything f32 EXCEPT the patch kernel, which the loader hard-codes as F16 (vit.cpp:515).
    `config` is a CONFIGS name or an explicit (hidden, layers, heads, patch, img) tuple; in_chans = 0 takes the config's default."""
    name = config if isinstance(config, str) else None
    hidden, layers, heads, patch, img = CONFIGS[name] if name else tuple(config)
    in_chans = in_chans or IN_CHANS.get(name, 3)
    classes = classes or NUM_CLASSES.get(name, 1000)
    assert ftype in (0, 1)
    tens = synth_tensors(hidden, layers, classes, patch, img, seed, round_bf16, in_chans)
    with open(path, "wb") as f:
        _write_header(f, (hidden, layers, heads, patch, img), ftype, classes)
        for name, shape, is_mat in tensor_specs(hidden, layers, classes, patch, img, in_chans):
            data = tens[name]
            ft = 1 if (is_mat and (ftype == 1 or name == "patch_embed.proj.weight")) else 0
            data = data.astype(np.float16) if ft == 1 else data.astype(np.float32)
            if name == "patch_embed.proj.bias":
                data = data.reshape(1, data.shape[0], 1, 1)  # convert-pth-to-ggml.py:150-151
            nm = name.encode()
            f.write(struct.pack("iii", data.ndim, len(nm), ft))
            for d in reversed(data.shape):
                f.write(struct.pack("i", d))
            f.write(nm)
            data.tofile(f)


def dequant_q8_0(raw: np.ndarray, n_elem: int) -> np.ndarray:
    """block_q8_0 stream -> f32 (ggml-quants.c dequantize_row_q8_0): x = d * q."""
    nb = n_elem // QK8_0
    blk = raw.reshape(nb, 34)
    d = blk[:, :2].copy().view(np.float16).astype(np.float32)  # [nb,1]
    q = blk[:, 2:].copy().view(np.int8).astype(np.float32)
    return (d * q).reshape(-1)


QUANT_BLOCK_BYTES = {2: 18, 3: 20, 6: 22, 7: 24, 8: 34}  # ggml-quants.h:11-47, 32 weights per block
QUANT_NAMES = {"q4_0": 2, "q4_1": 3, "q5_0": 6, "q5_1": 7, "q8_0": 8}


def dequant_blocks(ft: int, raw: np.ndarray, n_elem: int) -> np.ndarray:
    """q4_0 / q4_1 / q5_0 / q5_1 / q8_0 block stream -> f32, the arithmetic of ggml-quants.c dequantize_row_q* (:1074-1185)."""
    if ft == 8:
        return dequant_q8_0(raw, n_elem)
    nb = n_elem // 32
    blk = raw.reshape(nb, QUANT_BLOCK_BYTES[ft])
    has_min, five = ft in (3, 7), ft in (6, 7)
    d = blk[:, 0:2].copy().view(np.float16).astype(np.float32)
    off = 2
    m = np.zeros_like(d)
    if has_min:
        m = blk[:, 2:4].copy().view(np.float16).astype(np.float32)
        off = 4
    lo_hi = np.zeros((nb, 32), np.int32)
    if five:
        qh = blk[:, off:off + 4].copy().view(np.uint32).astype(np.int64)  # [nb,1]
        off += 4
        j = np.arange(16)
        lo_hi[:, :16] = ((qh >> j) << 4) & 0x10
        lo_hi[:, 16:] = (qh >> (j + 12)) & 0x10
    qs = blk[:, off:off + 16].astype(np.int32)
    x = np.concatenate([qs & 0x0F, qs >> 4], axis=1) | lo_hi
    if has_min:
        y = x.astype(np.float32) * d + m
    else:
        y = (x - (16 if five else 8)).astype(np.float32) * d
    return y.astype(np.float32).reshape(-1)


def read(path: str) -> VitFile:
    """Parse a legacy-ggml ViT file (f32 / f16 / q4_0 / q4_1 / q5_0 / q5_1 / q8_0 tensors)."""
    with open(path, "rb") as f:
        buf = f.read()
    off = 0

    def i32():
        nonlocal off
        v = struct.unpack_from("i", buf, off)[0]
        off += 4
        return v

    magic = i32()
    if magic != GGML_FILE_MAGIC:
        raise ValueError("bad magic")
    hidden, layers, heads, classes, patch, img, ftype = (i32() for _ in range(7))
    vf = VitFile(hidden, layers, heads, classes, patch, img, ftype % 1000)
    for _ in range(i32()):
        k = i32()
        ln = i32()
        vf.id2label[k] = buf[off:off + ln].decode()
        off += ln
    while off < len(buf):
        n_dims, ln, ft = i32(), i32(), i32()
        ne = [i32() for _ in range(n_dims)]
        name = buf[off:off + ln].decode()
        off += ln
        shape = tuple(reversed(ne))
        n = int(np.prod(shape))
        if ft == 0:
            arr = np.frombuffer(buf, np.float32, n, off).reshape(shape)
            off += 4 * n
        elif ft == 1:
            arr = np.frombuffer(buf, np.float16, n, off).reshape(shape)
            off += 2 * n
        elif ft in QUANT_BLOCK_BYTES:
            nbytes = n // 32 * QUANT_BLOCK_BYTES[ft]
            arr = np.frombuffer(buf, np.uint8, nbytes, off).copy()
            off += nbytes
            if ft == 8:
                vf.tensors[name + ".q8_0_raw"] = arr
            arr = dequant_blocks(ft, arr, n).reshape(shape)
        else:
            raise ValueError(f"unsupported tensor ftype {ft}")
        vf.tensors[name] = arr
        vf.tensor_ftype[name] = ft
    return vf


def synthetic_gray_images(batch: int, img_size: int, seed: int = 1234) -> np.ndarray:
    """float32[B,S,S], values = what the ViTSTR preprocess can emit: (u8/255 - 0.5)*2 (vitstr.cpp:174-175)."""
    rng = np.random.default_rng(seed)
    u8 = rng.integers(0, 256, size=(batch, img_size, img_size), dtype=np.uint8)
    return ((u8.astype(np.float32) / np.float32(255.0) - np.float32(0.5)) * np.float32(2.0)).astype(np.float32)


def synthetic_images(batch: int, img_size: int, seed: int = 1234) -> np.ndarray:
    """float32[B,S,S,3] HWC, values = what vit_image_preprocess can emit (vit.cpp:233-234,279-280):
    (u8 - mean_c)/std_c with u8 ~ U{0..255}.  SURVEY.md 8d."""
    rng = np.random.default_rng(seed)
    u8 = rng.integers(0, 256, size=(batch, img_size, img_size, 3), dtype=np.uint8)
    mean = np.array([123.675, 116.280, 103.530], np.float32)
    std = np.array([58.395, 57.120, 57.375], np.float32)
    return ((u8.astype(np.float32) - mean) / std).astype(np.float32)


# (ny, nx) of the random RGB inputs of preprocess_test_images: down-, identity- and up-scaling, odd aspect ratios, single rows and
# columns, a single pixel, extreme upscaling
PREPROCESS_TEST_SIZES = [(300, 280), (224, 224), (97, 131), (512, 333), (64, 640),
                         (1, 1), (1, 517), (403, 1), (2, 3), (16, 16), (2000, 35)]


def preprocess_test_images(seed: int = 2):
    """u8 HxWx3 RGB inputs for vit_image_preprocess (vit.cpp:204-305) tests: uniform noise at PREPROCESS_TEST_SIZES, plus one smooth
    400 x 300 image in sixth place (random noise alone under-samples the interpolation arithmetic)."""
    rng = np.random.default_rng(seed)
    imgs = [rng.integers(0, 256, size=(ny, nx, 3), dtype=np.uint8) for ny, nx in PREPROCESS_TEST_SIZES[:5]]
    yy, xx = np.mgrid[0:400, 0:300]
    imgs.append(np.stack([(127 + 120 * np.sin(xx / 17.0)), (127 + 120 * np.cos(yy / 23.0)), ((xx + yy) % 256)], -1).astype(np.uint8))
    imgs += [rng.integers(0, 256, size=(ny, nx, 3), dtype=np.uint8) for ny, nx in PREPROCESS_TEST_SIZES[5:]]
    return imgs


# ------------------------------------------------------------------------------------------------
# True GGUF (v3) container -- the SURVEY.md 8(f) rank-3 extension read by csrc/gguf_file.hpp (key names documented there).
GGUF_MAGIC = b"GGUF"
GGML_TYPE_BF16 = 30  # current ggml; the reference's pinned ggml has no bf16 type
_GGUF_U32, _GGUF_F32, _GGUF_STR, _GGUF_ARR = 4, 6, 8, 9


def f32_to_bf16_bits(x: np.ndarray) -> np.ndarray:
    u = np.ascontiguousarray(x, np.float32).view(np.uint32).astype(np.uint64)
    return ((u + 0x7FFF + ((u >> 16) & 1)) >> 16).astype(np.uint16)  # RNE


def bf16_bits_to_f32(b: np.ndarray) -> np.ndarray:
    return (b.astype(np.uint32) << 16).view(np.float32)


def write_gguf(path: str, vf: VitFile, weight_type: str = "keep", alignment: int = 32) -> None:
    """Write `vf` as GGUF v3.  weight_type: 'keep' (each tensor in its VitFile type; quantised tensors are not supported here),
    'f16', 'f32' or 'bf16' for the block/head matrices (the patch kernel stays f16, 1-D tensors f32)."""
    def gstr(b: bytes) -> bytes:
        return struct.pack("<Q", len(b)) + b

    kv = []

    def kv_u32(k, v):
        kv.append(gstr(k.encode()) + struct.pack("<II", _GGUF_U32, v))

    kv.append(gstr(b"general.architecture") + struct.pack("<I", _GGUF_STR) + gstr(b"vit"))
    kv_u32("general.alignment", alignment)
    kv_u32("general.file_type", vf.ftype)
    for k, v in (("vit.hidden_size", vf.hidden_size), ("vit.num_hidden_layers", vf.num_hidden_layers),
                 ("vit.num_attention_heads", vf.num_attention_heads), ("vit.num_classes", vf.num_classes),
                 ("vit.patch_size", vf.patch_size), ("vit.image_size", vf.img_size)):
        kv_u32(k, v)
    kv.append(gstr(b"vit.layer_norm_eps") + struct.pack("<If", _GGUF_F32, 1e-6))
    if vf.id2label:
        labels = [vf.id2label.get(i, "").encode() for i in range(max(vf.id2label) + 1)]
        kv.append(gstr(b"vit.id2label") + struct.pack("<IIQ", _GGUF_ARR, _GGUF_STR, len(labels)) + b"".join(gstr(x) for x in labels))

    names = [n for n in vf.tensors if not n.endswith(".q8_0_raw")]
    blobs, infos, rel = [], [], 0
    for name in names:
        arr = vf.tensors[name]
        ft = vf.tensor_ftype[name]
        if ft not in (0, 1):
            raise ValueError("write_gguf: quantised tensors are not supported")
        is_mat = arr.ndim >= 2 and name not in ("cls_token", "pos_embed", "patch_embed.proj.bias")
        if is_mat and name != "patch_embed.proj.weight" and weight_type != "keep":
            ft = {"f32": 0, "f16": 1, "bf16": GGML_TYPE_BF16}[weight_type]
        if ft == 0:
            data = np.ascontiguousarray(arr, np.float32).tobytes()
        elif ft == 1:
            data = np.ascontiguousarray(arr, np.float16).tobytes()
        else:
            data = f32_to_bf16_bits(np.asarray(arr, np.float32)).tobytes()
        ne = list(reversed(arr.shape))
        infos.append(gstr(name.encode()) + struct.pack("<I", len(ne)) + b"".join(struct.pack("<Q", d) for d in ne) +
                     struct.pack("<IQ", ft, rel))
        pad = (-len(data)) % alignment
        blobs.append(data + b"\0" * pad)
        rel += len(data) + pad
    head = GGUF_MAGIC + struct.pack("<IQQ", 3, len(names), len(kv)) + b"".join(kv) + b"".join(infos)
    with open(path, "wb") as f:
        f.write(head + b"\0" * ((-len(head)) % alignment))
        for b in blobs:
            f.write(b)


def read_gguf(path: str) -> VitFile:
    """Parse a GGUF v2/v3 ViT container (the Python twin of csrc/gguf_file.hpp, for tooling and tests)."""
    buf = open(path, "rb").read()
    off = 0

    def rd(fmt):
        nonlocal off
        v = struct.unpack_from("<" + fmt, buf, off)
        off += struct.calcsize("<" + fmt)
        return v[0] if len(v) == 1 else v

    def rstr():
        nonlocal off
        n = rd("Q")
        s = buf[off:off + n]
        off += n
        return s.decode()

    if buf[:4] != GGUF_MAGIC:
        raise ValueError("not a GGUF file")
    off = 4
    version, n_tensors, n_kv = rd("I"), rd("Q"), rd("Q")
    if version not in (2, 3):
        raise ValueError(f"unsupported GGUF version {version}")
    scalar = {0: "B", 1: "b", 2: "H", 3: "h", 4: "I", 5: "i", 6: "f", 7: "?", 10: "Q", 11: "q", 12: "d"}
    kv = {}
    for _ in range(n_kv):
        key, vt = rstr(), rd("I")
        if vt == 8:
            kv[key] = rstr()
        elif vt == 9:
            et, cnt = rd("I"), rd("Q")
            kv[key] = [rstr() if et == 8 else rd(scalar[et]) for _ in range(cnt)]
        else:
            kv[key] = rd(scalar[vt])
    vf = VitFile(kv["vit.hidden_size"], kv["vit.num_hidden_layers"], kv["vit.num_attention_heads"], kv["vit.num_classes"],
                 kv["vit.patch_size"], kv.get("vit.image_size", kv.get("vit.img_size")), kv.get("general.file_type", 1))
    vf.id2label = dict(enumerate(kv.get("vit.id2label", [])))
    align = kv.get("general.alignment", 32)
    infos = []
    for _ in range(n_tensors):
        name, nd = rstr(), rd("I")
        ne = [rd("Q") for _ in range(nd)]
        infos.append((name, ne, rd("I"), rd("Q")))
    data0 = off + (-off) % align
    for name, ne, ft, rel in infos:
        shape = tuple(reversed(ne))
        n = int(np.prod(shape))
        o = data0 + rel
        if ft == 0:
            arr = np.frombuffer(buf, np.float32, n, o).reshape(shape)
        elif ft == 1:
            arr = np.frombuffer(buf, np.float16, n, o).reshape(shape)
        elif ft == GGML_TYPE_BF16:
            arr = bf16_bits_to_f32(np.frombuffer(buf, np.uint16, n, o)).reshape(shape)
        elif ft in QUANT_BLOCK_BYTES:
            arr = dequant_blocks(ft, np.frombuffer(buf, np.uint8, n // 32 * QUANT_BLOCK_BYTES[ft], o).copy(), n).reshape(shape)
        else:
            raise ValueError(f"unsupported tensor type {ft}")
        vf.tensors[name] = arr
        vf.tensor_ftype[name] = ft
    return vf


def legacy_to_gguf(src: str, dst: str, weight_type: str = "keep") -> None:
    """Offline converter (no timm, no torch): legacy-ggml ViT file -> GGUF."""
    write_gguf(dst, read(src), weight_type)
