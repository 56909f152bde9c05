"""CPU tests: pin the plain-C restatement (oracle/vit_oracle.c) against
 (a) the committed golden vectors in tests/golden/ (generated from the unmodified reference by
     tests/golden/make_golden.py), and
 (b) the compiled reference's own outputs (oracle/_ref/libvitref.so), bit for bit, stored in
     tests/golden/ref_live.npz by tests/golden/make_golden_ref.py.
The reference holds no golden vectors of its own for this path (SURVEY.md 4 / 8c: its only end-to-end
example needs real timm weights), so outputs of the reference run here ARE the pin."""
import hashlib
import os

import numpy as np
import pytest

from tests.util import gf, model_path
from oracle import ref, restatement as rs

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
LIVE = np.load(os.path.join(GOLD, "ref_live.npz"))
needs_ref = pytest.mark.skipif(not ref.available(), reason="oracle/_ref not built")


def _sha(path):
    h = hashlib.sha256()
    with open(path, "rb") as f:
        for c in iter(lambda: f.read(1 << 24), b""):
            h.update(c)
    return h.hexdigest()


def _digest(a):
    """sha256 of the float32 bytes: how ref_live.npz stores outputs that are only compared bit for bit."""
    return hashlib.sha256(np.ascontiguousarray(a, np.float32).tobytes()).hexdigest()


def _oracle(cfg, ft):
    path = model_path(cfg, ft)
    vf = gf.read(path)
    return path, vf, rs.OracleModel(vf, gf.tensor_specs)


@pytest.mark.parametrize("cfg,ft", [("micro", "f16"), ("micro14", "f16"), ("micro", "f32"), ("tiny", "f16")])
def test_restatement_matches_golden_bit_exact(cfg, ft):
    g = np.load(os.path.join(GOLD, f"{cfg}_{ft}.npz"))
    path, vf, om = _oracle(cfg, ft)
    assert _sha(path) == str(g["model_sha256"]), "synthetic model writer drifted from the golden fixture"
    rs.set_threads(8)
    imgs = gf.synthetic_images(int(g["n_images"]), vf.img_size, seed=int(g["image_seed"]))
    probs, logits = om.forward_batch(imgs)
    # same libm + same summation order => identical bits on the box that made the fixture;
    # elsewhere (different libm tanhf/expf) allow table-level noise.
    np.testing.assert_allclose(logits, g["logits"], rtol=0, atol=2e-3 * np.abs(g["logits"]).max())
    assert (np.argsort(-logits, 1)[:, :5] == np.argsort(-g["logits"], 1)[:, :5]).all()
    np.testing.assert_allclose(probs, g["probs"], rtol=0, atol=1e-3)


@pytest.mark.parametrize("cfg,ft", [("micro", "q8_0"), ("tiny", "q8_0")])
def test_restatement_matches_golden_q8_0(cfg, ft):
    g = np.load(os.path.join(GOLD, f"{cfg}_{ft}.npz"))
    path, vf, om = _oracle(cfg, ft)
    assert _sha(path) == str(g["model_sha256"])
    imgs = gf.synthetic_images(int(g["n_images"]), vf.img_size, seed=int(g["image_seed"]))
    probs, logits = om.forward_batch(imgs)
    np.testing.assert_allclose(logits, g["logits"], rtol=0, atol=2e-3 * np.abs(g["logits"]).max())


@pytest.mark.parametrize("cfg,ft", [("micro", "f16"), ("micro14", "f16"), ("micro", "f32"), ("micro", "q8_0"),
                                    ("tiny", "f16")])
def test_restatement_bit_exact_vs_compiled_reference(cfg, ft):
    path, vf, om = _oracle(cfg, ft)
    imgs = gf.synthetic_images(2, vf.img_size, seed=77)
    for i in range(2):
        l_ref = LIVE[f"s77_{cfg}_{ft}_logits"][i]
        p, l = om.forward(imgs[i])
        assert np.array_equal(l, l_ref), np.abs(l - l_ref).max()
        assert _digest(p) == str(LIVE[f"s77_{cfg}_{ft}_probs_sha256"][i])


@needs_ref
def test_reference_is_thread_count_invariant():
    path = model_path("micro", "f16")
    m = ref.RefModel(path)
    img = gf.synthetic_images(1, m.img, seed=3)[0]
    outs = [m.predict(img, n_threads=t)[1] for t in (1, 3, 8)]
    assert np.array_equal(outs[0], outs[1]) and np.array_equal(outs[0], outs[2])
    m.close()


def test_primitives_bit_exact_vs_reference_ops():
    rng = np.random.default_rng(5)
    x = (rng.standard_normal((64, 197)) * 4).astype(np.float32)
    # GELU through the f16 table, every finite f16 input (ggml.c:1434-1441, 2197)
    allh = np.arange(65536, dtype=np.uint16).view(np.float16).astype(np.float32)
    allh = allh[np.isfinite(allh)]
    assert _digest(rs.gelu_table(allh)) == str(LIVE["prim_gelu_sha256"])
    # softmax rows (ggml.c:10498-10567)
    assert _digest(rs.softmax_rows(x)) == str(LIVE["prim_softmax_sha256"])
    # f16 rounding (ggml.c:315-332)
    assert _digest(rs.round_f16(x)) == str(LIVE["prim_round_f16_sha256"])
    # norm (ggml.c:8959-9008) == restatement layernorm with w=1,b=0
    ones, zeros = np.ones(197, np.float32), np.zeros(197, np.float32)
    assert _digest(rs.layernorm(x, ones, zeros, 1e-6)) == str(LIVE["prim_norm_sha256"])


def test_model_file_roundtrip_and_shapes():
    path = model_path("micro", "f16")
    vf = gf.read(path)
    assert (vf.hidden_size, vf.num_hidden_layers, vf.num_attention_heads) == (128, 2, 2)
    assert len([k for k in vf.tensors]) == 4 + 12 * 2 + 4
    assert vf.tensors["patch_embed.proj.weight"].dtype == np.float16
    assert vf.tensors["patch_embed.proj.bias"].shape == (1, 128, 1, 1)  # convert-pth-to-ggml.py:150-151
    assert vf.tensors["pos_embed"].shape == (1, vf.n_tokens, 128)
    assert vf.id2label[5] == "LABEL_5"


def test_synthetic_images_are_preprocess_range():
    x = gf.synthetic_images(2, 32, seed=1)
    assert x.dtype == np.float32 and x.shape == (2, 32, 32, 3)
    assert x.min() >= -2.2 and x.max() <= 2.7


@pytest.mark.parametrize("name", ["q4_0", "q4_1", "q5_0", "q5_1", "q8_0"])
def test_block_dequant_matches_ggml(name):
    """The upload-time weight conversion (C++ in the library, numpy in the file tooling) against ggml's own
    ggml_quantize_* / dequantize_row_* (ggml-quants.c:1074-1185) compiled from the reference tree (blocks and their dequantised
    values stored in ref_live.npz): f32 values identical, engine output = their f16 rounding."""
    from tests.util import pkg
    ft = gf.QUANT_NAMES[name]
    rng = np.random.default_rng(ft)
    n = 32 * 257
    src = (rng.normal(0, 0.05, n) * rng.choice([1.0, 8.0, 0.01], n)).astype(np.float32)
    blocks = LIVE[f"dequant_{name}_blocks"]
    want = LIVE[f"dequant_{name}_want"]
    assert blocks.size == n // 32 * gf.QUANT_BLOCK_BYTES[ft]
    got_np = gf.dequant_blocks(ft, blocks, n)
    assert np.array_equal(got_np, want) or np.abs(got_np - want).max() <= 2.0 ** -24 * np.abs(want).max()  # *_1: fma or not
    got_eng = pkg.engine.test_dequant(ft, blocks)
    assert np.array_equal(got_eng, want.astype(np.float16)) or \
        np.abs(got_eng.astype(np.float32) - want).max() <= 2.0 ** -11 * np.abs(want).max()
    assert np.abs(want - src).max() < (0.2 if name.startswith("q4") else 0.1)   # it is a quantisation of src


def test_gguf_writer_reader_round_trip(tmp_path):
    """legacy file -> GGUF (kept types / BF16 matrices) -> read back: hyper-parameters, labels and every tensor survive; BF16 is
    exact for bf16-representable weights (the bf16w synthetic model) and a 8-bit-mantissa rounding otherwise."""
    src = gf.read(model_path("micro", "f16"))
    dst = str(tmp_path / "keep.gguf")
    gf.write_gguf(dst, src, "keep")
    back = gf.read_gguf(dst)
    assert (back.hidden_size, back.num_hidden_layers, back.num_attention_heads, back.num_classes, back.patch_size, back.img_size) == \
        (src.hidden_size, src.num_hidden_layers, src.num_attention_heads, src.num_classes, src.patch_size, src.img_size)
    assert back.id2label[5] == src.id2label[5]
    for name, arr in src.tensors.items():
        assert back.tensor_ftype[name] == src.tensor_ftype[name] and np.array_equal(back.tensors[name], arr), name
    srcb = gf.read(model_path("micro", "bf16w"))
    dstb = str(tmp_path / "bf16.gguf")
    gf.write_gguf(dstb, srcb, "bf16")
    backb = gf.read_gguf(dstb)
    w = "blocks.1.mlp.fc1.weight"
    assert backb.tensor_ftype[w] == gf.GGML_TYPE_BF16 and np.array_equal(backb.tensors[w], srcb.tensors[w])
    assert backb.tensor_ftype["patch_embed.proj.weight"] == 1 and backb.tensor_ftype["norm.bias"] == 0


@pytest.mark.parametrize("cfg", ["vitstr_micro", "vitstr_tiny"])
def test_restatement_equals_the_vitstr_extension_bit_for_bit(cfg):
    """The C restatement with in_chans = 1, head_tokens = 25 against the reference's ViTSTR extension compiled from its own
    sources (oracle/Makefile: libvitstrref.so; its outputs are the committed golden fixture): 25 x classes logits and
    probabilities identical bit for bit."""
    path = model_path(cfg, "f16")
    vf = gf.read(path)
    g = np.load(os.path.join(GOLD, f"{cfg}_f16.npz"))
    assert _sha(path) == str(g["model_sha256"])
    om = rs.OracleModel(vf, gf.tensor_specs, head_tokens=25)
    rs.set_threads(8)
    imgs = gf.synthetic_gray_images(2, vf.img_size, seed=int(g["image_seed"]))
    for i in range(2):
        p_o, l_o = om.forward(imgs[i])
        assert np.array_equal(l_o, g["logits"][i]) and np.array_equal(p_o, g["probs"][i])
    om.close()


# ------------------------------------------------------------------------------------------------
# Offline converters (vit.cpp_b200/convert.py): the timm-free counterparts of convert-pth-to-ggml.py and quantize.cpp
def test_state_dict_converter_reproduces_the_reference_layout(tmp_path):
    """A plain state_dict (safetensors file, or a torch checkpoint) -> model file must be byte-identical to what the writer that
    follows convert-pth-to-ggml.py:105-158 produces for the same weights, for both ftypes; hyper-parameters are inferred from the
    tensor shapes alone; the f32 container keeps the patch kernel f16 (vit.cpp:515).  The reference itself must load the result."""
    from tests.util import pkg
    conv = pkg.convert
    hidden, layers, heads, patch, img = gf.CONFIGS["micro"]
    tens = gf.synth_tensors(hidden, layers, 1000, patch, img, seed=0)
    st = str(tmp_path / "micro.safetensors")
    conv.write_safetensors(st, tens)
    back = conv.read_safetensors(st)
    assert list(back) == list(tens) and all(np.array_equal(back[k], tens[k]) for k in tens)
    assert conv.infer_hparams(back, heads=heads) == (hidden, layers, heads, 1000, patch, img, 3)
    for ftype in (1, 0):
        want = str(tmp_path / f"want{ftype}.gguf")
        got = str(tmp_path / f"got{ftype}.gguf")
        gf.write_synthetic(want, "micro", ftype, seed=0)
        conv.state_dict_to_model_file(back, got, ftype, heads=heads)
        assert open(got, "rb").read() == open(want, "rb").read()
    # torch checkpoint path, with a norm_pre tensor that the reference converter skips
    import torch
    sd = {k: torch.from_numpy(v.copy()) for k, v in tens.items()}
    sd["norm_pre.weight"] = torch.ones(hidden)
    pth = str(tmp_path / "micro.pth")
    torch.save(sd, pth)
    got = str(tmp_path / "from_pth.gguf")
    conv.main([pth, got, "--ftype", "1", "--heads", str(heads)])
    assert open(got, "rb").read() == open(str(tmp_path / "want1.gguf"), "rb").read()
    # a real GGUF container from the same state_dict parses back to the same tensors
    gg = str(tmp_path / "micro.real.gguf")
    conv.state_dict_to_model_file(back, gg, 1, heads=heads, container="gguf")
    vf = gf.read_gguf(gg)
    assert (vf.hidden_size, vf.num_hidden_layers, vf.num_attention_heads) == (hidden, layers, heads)
    assert np.array_equal(vf.tensors["blocks.1.mlp.fc2.weight"], tens["blocks.1.mlp.fc2.weight"].astype(np.float16))
    if ref.available():
        m = ref.RefModel(str(tmp_path / "got1.gguf"))
        assert (m.hidden, m.layers, m.heads, m.classes) == (hidden, layers, heads, 1000)
        m.close()


@pytest.mark.parametrize("cfg", ["micro", "tiny"])
def test_q8_0_quantizer_is_byte_identical_to_the_reference_binary(cfg, tmp_path):
    """convert.quantize_model_file restates quantize.cpp + quantize_row_q8_0_reference; the reference's own `quantize` binary on the
    same f16 file is the golden output (its sha256 is stored in ref_live.npz)."""
    from tests.util import pkg
    got = str(tmp_path / "q8.gguf")
    pkg.convert.quantize_model_file(model_path(cfg, "f16"), got, "q8_0")
    assert _sha(got) == str(LIVE[f"quantize_q8_0_{cfg}_sha256"])
