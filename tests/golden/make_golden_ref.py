"""Store what the tests used to read from a live run of the UNMODIFIED reference (oracle/_ref, built by oracle/Makefile), so that
they compare against the reference without needing it at test time.  Run where oracle/_ref is built:
    python tests/golden/make_golden_ref.py

  ref_live.npz   reference logits / probabilities of the seeded images the tests feed (bit-exact pins of the restatement, fresh-image
                 and bf16-weight parity of the engine, the u8 -> preprocess -> predict pipeline), the reference's primitive ops (GELU
                 table on every finite f16, soft-max rows, f16 rounding, norm), ggml's block quantisers + dequantisers on a seeded
                 vector, and the sha256 of the reference quantize binary's q8_0 files.  Outputs that the tests only compare bit for
                 bit are stored as the sha256 of their float32 bytes (digest()), which keeps the fixture small."""
import ctypes as C
import hashlib
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from tests.util import gf, model_path  # noqa: E402
from oracle import ref  # noqa: E402

BIT_EXACT = [("micro", "f16"), ("micro14", "f16"), ("micro", "f32"), ("micro", "q8_0"), ("tiny", "f16")]


def digest(a):
    return np.array(hashlib.sha256(np.ascontiguousarray(a, np.float32).tobytes()).hexdigest())


def sha256(path):
    h = hashlib.sha256()
    with open(path, "rb") as f:
        for chunk in iter(lambda: f.read(1 << 24), b""):
            h.update(chunk)
    return h.hexdigest()


def primitives(out):
    L = ref.lib()
    L.vitref_unary.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_float]
    ref.RefModel(model_path("micro", "f16")).close()   # ggml_init fills the tables
    rng = np.random.default_rng(5)
    x = (rng.standard_normal((64, 197)) * 4).astype(np.float32)
    allh = np.arange(65536, dtype=np.uint16).view(np.float16).astype(np.float32)
    allh = allh[np.isfinite(allh)]
    g = np.empty_like(allh)
    L.vitref_unary(0, allh.ctypes.data, g.ctypes.data, allh.size, 1, 0.0)
    sm, nm = np.empty_like(x), np.empty_like(x)
    L.vitref_unary(1, x.ctypes.data, sm.ctypes.data, 197, 64, 0.0)
    L.vitref_unary(2, x.ctypes.data, nm.ctypes.data, 197, 64, 1e-6)
    out["prim_gelu_sha256"] = digest(g)
    out["prim_softmax_sha256"] = digest(sm)
    out["prim_round_f16_sha256"] = digest(ref.round_f16(x))
    out["prim_norm_sha256"] = digest(nm)


def dequant(out):
    L = ref.lib()
    ref.RefModel(model_path("micro", "f16")).close()
    for name, ft in gf.QUANT_NAMES.items():
        rng = np.random.default_rng(ft)
        n = 32 * 257
        src = (rng.normal(0, 0.05, n) * rng.choice([1.0, 8.0, 0.01], n)).astype(np.float32)
        blocks = np.zeros(n // 32 * gf.QUANT_BLOCK_BYTES[ft], np.uint8)
        hist = np.zeros(16, np.int64)
        quant = getattr(L, f"ggml_quantize_{name}")
        quant.restype = C.c_size_t
        quant.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]
        assert quant(src.ctypes.data, blocks.ctypes.data, n, n, hist.ctypes.data) == blocks.size
        want = np.empty(n, np.float32)
        deq = getattr(L, f"dequantize_row_{name}")
        deq.restype = None
        deq.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        deq(blocks.ctypes.data, want.ctypes.data, n)
        out[f"dequant_{name}_blocks"] = blocks
        out[f"dequant_{name}_want"] = want


def quantize_sha(out):
    with tempfile.TemporaryDirectory() as d:
        for cfg in ("micro", "tiny"):
            dst = os.path.join(d, f"{cfg}.q8_0")
            subprocess.check_call([ref.QUANTIZE_BIN, model_path(cfg, "f16"), dst, str(gf.QUANT_NAMES["q8_0"])],
                                  stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
            out[f"quantize_q8_0_{cfg}_sha256"] = np.array(sha256(dst))


def forwards(out):
    for cfg, ft in BIT_EXACT:                                        # tests/test_oracle.py bit-exact pins: 2 images, seed 77
        m = ref.RefModel(model_path(cfg, ft))
        p, l = m.predict_batch(gf.synthetic_images(2, m.img, seed=77), n_threads=4)
        out[f"s77_{cfg}_{ft}_logits"], out[f"s77_{cfg}_{ft}_probs_sha256"] = l, np.stack([digest(pi) for pi in p])
        m.close()
    m = ref.RefModel(model_path("tiny", "f16"))                      # fresh images of the engine's parity test
    p, l = m.predict_batch(gf.synthetic_images(12, m.img, seed=31337), n_threads=8)
    out["s31337_tiny_f16_logits"], out["s31337_tiny_f16_probs"] = l, p
    rng = np.random.default_rng(4)                                   # u8 -> reference preprocess -> reference predict
    imgs = [rng.integers(0, 256, size=(260, 310, 3), dtype=np.uint8) for _ in range(3)]
    out["u8_s4_tiny_f16_logits"] = np.stack([m.predict(m.preprocess(im), n_threads=8)[1] for im in imgs])
    m.close()
    m = ref.RefModel(model_path("tiny", "bf16w"))                    # the reference's f32 path on bf16-representable weights
    p, l = m.predict_batch(gf.synthetic_images(3, m.img, seed=8), n_threads=8)
    out["s8_tiny_bf16w_logits"] = l
    m.close()


def main():
    out = {}
    primitives(out)
    dequant(out)
    quantize_sha(out)
    forwards(out)
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "ref_live.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
