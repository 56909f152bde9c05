"""GPU parity tests proper: the CUDA path, called through the C ABI (vit_model_load / vit_predict mirror), against
 (1) the committed golden vectors generated from the unmodified reference (tests/golden/make_golden*.py),
 (2) the plain-C restatement (incl. per-layer taps), and (3) the compiled reference itself when oracle/_ref is built.

Tolerances (DESIGN.md section 4): the north star asks for logits "within 1e-3 relative fp16 tolerance" and identical top-k.
 * Metric: per image, max|dlogit| / max|ref logit| (SURVEY.md 7.4).  Two *correct* implementations that are not bit-identical
   already differ by a median of 3e-4 (micro) / 6.4e-4 (tiny) / 7.6e-4 (base) and up to 1.2e-3 on single images: the restatement run
   with double-precision accumulation and the reference's rounding points ("variant 1"; per-image values for the 64 headline images
   are stored in tests/golden/base_f16_b64.npz as `floor`).  "<= 1e-3 on EVERY image" is therefore not attainable by any
   implementation on these weights; what IS attainable, and asserted, is to sit AT that floor: the engine's error distribution must
   stay within 1.1x of the floor distribution on the same images (median and 90th percentile), no image above 1.25e-3, and the
   top-5 index lists must be identical with NO gap-aware exemption on the headline batch.
 * Generic check (small fixtures of 2-12 images): median <= 1e-3, every image <= 1.25e-3 (1.5e-3 for the 2-layer-deep "micro"
   models whose max|logit| is small), L2 <= 1.1e-3, top-5 identical wherever the reference's own top-5 logit gaps exceed 2.5x the
   observed error (reported; 0 exemptions expected), |dp| no larger than the logit deviation allows."""
import os

import numpy as np
import pytest

from tests.util import pkg, gf, model_path
from oracle import ref, restatement as rs

eng = pkg.engine
pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
LIVE = np.load(os.path.join(GOLD, "ref_live.npz"))   # outputs of the compiled reference (tests/golden/make_golden_ref.py)


def rel_err(logits, ref_logits):
    return np.abs(logits - ref_logits).max(axis=1) / np.abs(ref_logits).max(axis=1)


def check_parity(logits, probs, idx, ref_logits, ref_probs, k=5, max_tol=1.25e-3):
    re = rel_err(logits, ref_logits)
    l2 = np.linalg.norm(logits - ref_logits, axis=1) / np.linalg.norm(ref_logits, axis=1)
    assert l2.max() <= 1.1e-3 * (max_tol / 1.25e-3), l2
    assert np.median(re) <= 1e-3, re
    assert re.max() <= max_tol, re
    # probabilities: (a) exactly the soft-max of OUR logits (f32 rounding only); (b) against the reference no further off than
    # the logit deviation allows: |dp_i| = p_i |dl_i - sum_j p_j dl_j| <= 2 p_i (1 - p_i) max|dl| <= 0.5 max|dl| (first order)
    z = logits.astype(np.float64) - logits.max(axis=1, keepdims=True)
    sm = np.exp(z) / np.exp(z).sum(axis=1, keepdims=True)
    assert np.abs(probs - sm).max() <= 2e-3 * sm.max()   # f16-table exp semantics of the reference soft-max (ggml.c:10547)
    dl = np.abs(logits - ref_logits).max(axis=1)
    assert (np.abs(probs - ref_probs).max(axis=1) <= 0.55 * dl + 1e-6).all(), (np.abs(probs - ref_probs).max(axis=1), dl)
    order = np.argsort(-ref_logits, 1)[:, : k + 1]
    exempt = 0
    for b in range(logits.shape[0]):
        gaps = -np.diff(ref_logits[b, order[b]])
        err = np.abs(logits[b] - ref_logits[b]).max()
        if gaps.min() > 2.5 * err:  # otherwise a tie-flip is within the noise of ANY implementation
            assert (idx[b] == order[b, :k]).all(), (b, idx[b], order[b], gaps, err)
        elif not (idx[b] == order[b, :k]).all():
            exempt += 1
    assert exempt <= max(1, logits.shape[0] // 16), f"{exempt} images needed the near-tie exemption"
    return re


@pytest.mark.parametrize("cfg", ["micro", "micro14", "tiny", "base"])
def test_logits_and_topk_match_golden(cfg):
    g = np.load(os.path.join(GOLD, f"{cfg}_f16.npz"))
    m = eng.vit_model_load(model_path(cfg, "f16"), 0, 8)
    imgs = gf.synthetic_images(int(g["n_images"]), m.img_size, seed=int(g["image_seed"]))
    probs, idx, val, logits = eng.vit_predict(m, imgs, 5, want_logits=True)
    check_parity(logits, probs, idx, g["logits"], g["probs"], max_tol=1.5e-3 if cfg.startswith("micro") else 1.25e-3)
    # top-k values are the probabilities at those indices, descending
    assert np.array_equal(val, np.take_along_axis(probs, idx.astype(np.int64), 1))
    assert (np.diff(val, axis=1) <= 0).all()
    assert m.last_launch_count() > 0
    m.close()


@pytest.mark.parametrize("cfg,layer", [("micro", 0), ("micro", 1), ("tiny", 0), ("tiny", 11)])
def test_taps_match_restatement(cfg, layer):
    path = model_path(cfg, "f16")
    vf = gf.read(path)
    om = rs.OracleModel(vf, gf.tensor_specs)
    imgs = gf.synthetic_images(2, vf.img_size, seed=7)
    m = eng.vit_model_load(path, 0, 4)
    probs, logits, taps = eng.vit_predict_debug(m, imgs, layer)
    for b in range(2):
        _, l_o, t_o = om.forward(imgs[b], layer, tuple(eng.TAP_SHAPES))
        for name, tol in [("embed", 1e-5), ("ln1", 2e-3), ("qkv", 2e-3), ("attn", 2e-3), ("x1", 2e-3), ("ln2", 2e-3),
                          ("h", 3e-3), ("x2", 2e-3), ("final_ln", 3e-3), ("x_final", 2e-3)]:
            a, r = taps[name][b], t_o[name]
            assert np.abs(a - r).max() <= tol * np.abs(r).max(), (name, np.abs(a - r).max(), np.abs(r).max())
    m.close()


def test_against_live_reference_fresh_images():
    path = model_path("tiny", "f16")
    m = eng.vit_model_load(path, 0, 16)
    imgs = gf.synthetic_images(12, m.img_size, seed=31337)
    p_ref, l_ref = LIVE["s31337_tiny_f16_probs"], LIVE["s31337_tiny_f16_logits"]
    probs, idx, val, logits = eng.vit_predict(m, imgs, 5, want_logits=True)
    check_parity(logits, probs, idx, l_ref, p_ref)
    m.close()


def test_long_sequence_geometry_vit_large_384():
    """BASELINE.json configs[2] geometry (hidden 1024, 16 heads, 384^2 -> 577 tokens; 2 layers here): exercises the
    577-token attention kernel, D = 1024 LayerNorm and the 1024/3072/4096-wide GEMMs against the restatement."""
    path = model_path("large384x2", "f16")
    vf = gf.read(path)
    om = rs.OracleModel(vf, gf.tensor_specs)
    rs.set_threads(8)
    imgs = gf.synthetic_images(2, vf.img_size, seed=21)
    m = eng.vit_model_load(path, 0, 2)
    probs, logits, taps = eng.vit_predict_debug(m, imgs, 1, taps=("attn", "x2"))
    for b in range(2):
        p_o, l_o, t_o = om.forward(imgs[b], 1, ("attn", "x2"))
        assert np.abs(taps["attn"][b] - t_o["attn"]).max() <= 4e-3 * np.abs(t_o["attn"]).max()  # f16 storage: <= 2 ulp at the top binade
        assert np.abs(logits[b] - l_o).max() <= 2e-3 * np.abs(l_o).max()
        assert np.linalg.norm(logits[b] - l_o) <= 1e-3 * np.linalg.norm(l_o)
        assert logits[b].argmax() == l_o.argmax()
    m.close()


def test_full_depth_vit_large_384_bf16_weights_8_images():
    """BASELINE.json configs[2] at its real size (ViT-L/16-384: 24 layers, hidden 1024, 577 tokens, bf16-representable weights in
    the f32 container): 8 seeded images against the UNMODIFIED reference's logits (tests/golden/large384_bf16w_b8.npz, generated
    by tests/golden/make_golden_dist.py), per image, plus batch-position invariance at a batch that makes every attention CTA loop
    over several heads.  The reference runs this file through its f32 path (f32 activations), the engine feeds f16 activations to
    the tensor cores: the distance is the f16-activation noise of 24 layers (tiny, 12 layers: <= 2.5e-3), not an accumulation
    artefact -- hence 4e-3 here instead of the f16 configs' 1.25e-3."""
    g = np.load(os.path.join(GOLD, "large384_bf16w_b8.npz"))
    n = int(g["n_images"])
    path = model_path("large384", "bf16w")
    m = eng.vit_model_load(path, 0, 12)
    imgs = gf.synthetic_images(12, m.img_size, seed=31)
    fixed = gf.synthetic_images(n, m.img_size, seed=int(g["image_seed"]))
    pos = [0, 1, 3, 5, 6, 8, 10, 11]
    for j, p in enumerate(pos):
        imgs[p] = fixed[j]
    probs, idx, val, logits = eng.vit_predict(m, imgs, 5, want_logits=True)
    re = rel_err(logits[pos], g["logits"])
    l2 = np.linalg.norm(logits[pos] - g["logits"], axis=1) / np.linalg.norm(g["logits"], axis=1)
    print("ViT-L/16-384 bf16w, 8 images vs reference: max-norm", re, "L2", l2)
    assert re.max() <= 4e-3 and np.median(re) <= 3e-3, re
    assert l2.max() <= 2.5e-3, l2
    assert (idx[pos, 0] == g["logits"].argmax(1)).all()
    alone = eng.vit_predict(m, imgs[5:6], 5, want_logits=True)
    assert np.array_equal(alone[3][0], logits[5])
    assert np.isfinite(logits).all()
    if ref.available():  # one image through the live reference on this host: the fixture is not stale
        rm = ref.RefModel(path)
        p_ref, l_ref = rm.predict(imgs[pos[2]], n_threads=32)
        rm.close()
        assert np.abs(l_ref - g["logits"][2]).max() <= 1e-6 * np.abs(l_ref).max()
    m.close()


def test_bf16_weights_in_f32_container_vs_reference_f32_path():
    """BASELINE.json configs[2] weight format: the reference has no bf16 type (SURVEY.md section 0), so the oracle is its f32
    path on a file of bf16-representable f32 weights (f16 patch kernel).  The engine rounds f32 weights to f16 at upload,
    which is EXACT for bf16 values with |w| >= 2^-14, and multiplies them with f16 activations; the reference keeps f32
    activations, so agreement is at the f16-activation noise level (SURVEY.md 7.4: 5e-4..1e-3), far from the 5e-3 a
    bf16-activation design would show.  (f16 x bf16 in one tcgen05.mma is an illegal instruction on B200.)"""
    path = model_path("tiny", "bf16w")
    m = eng.vit_model_load(path, 0, 4)
    imgs = gf.synthetic_images(3, m.img_size, seed=8)
    l_ref = LIVE["s8_tiny_bf16w_logits"]
    probs, idx, val, logits = eng.vit_predict(m, imgs, 5, want_logits=True)
    assert rel_err(logits, l_ref).max() <= 2.5e-3
    assert (np.linalg.norm(logits - l_ref, axis=1) <= 1.5e-3 * np.linalg.norm(l_ref, axis=1)).all()
    assert (idx[:, 0] == l_ref.argmax(1)).all()
    m.close()


def test_batch_invariance_and_ragged_batches():
    """An image's result must not depend on its batch mates or position (independent units, SURVEY.md 8e)."""
    m = eng.vit_model_load(model_path("tiny", "f16"), 0, 9)
    imgs = gf.synthetic_images(9, m.img_size, seed=5)
    p_all, i_all, v_all, l_all = eng.vit_predict(m, imgs, 5, want_logits=True)
    for sl in (slice(0, 1), slice(3, 8), slice(8, 9)):
        p, i, v, l = eng.vit_predict(m, imgs[sl], 5, want_logits=True)
        assert np.array_equal(l, l_all[sl]) and np.array_equal(p, p_all[sl]) and np.array_equal(i, i_all[sl])
    m.close()


def test_full_batch_256_base_parity_at_the_noise_floor():
    """BASELINE.json configs[1] at its real size (ViT-B/16, batch 256).  64 of the 256 images are the seeded fixtures of
    tests/golden/base_f16_b64.npz (reference logits from the unmodified reference + per-image noise floor `floor`, the distance
    of a correct-but-not-bit-identical CPU implementation on the same images); they are scattered over the batch (first / last
    image, both sides of every 32-image boundary) and compared PER IMAGE:
      * engine error distribution <= 1.1 x the floor distribution (median, 90th percentile), no image above 1.25e-3;
      * top-5 index lists identical on all 64 images, no exemption; top-1 identical; |dp| bounded by the logit deviation;
      * the same images alone (batch 64) give bit-identical logits (position / batch-mate invariance);
      * size-independent properties on all 256: probabilities sum to 1, top-k sorted and consistent, everything finite."""
    g = np.load(os.path.join(GOLD, "base_f16_b64.npz"))
    n = int(g["n_images"])
    m = eng.vit_model_load(model_path("base", "f16"), 0, 256)
    base = gf.synthetic_images(n, 224, seed=int(g["image_seed"]))
    imgs = gf.synthetic_images(256, 224, seed=99)
    pos = sorted(set([0, 255] + list(range(31, 256, 32)) + list(range(32, 256, 32)) + list(range(3, 256, 5))))[:n]
    assert len(pos) == n
    for j, p in enumerate(pos):
        imgs[p] = base[j]
    probs, idx, val, logits = eng.vit_predict(m, imgs, 5, want_logits=True)
    re = rel_err(logits[pos], g["logits"])
    floor = g["floor"]
    stats = dict(median=float(np.median(re)), p90=float(np.quantile(re, 0.9)), max=float(re.max()),
                 floor_median=float(np.median(floor)), floor_p90=float(np.quantile(floor, 0.9)), floor_max=float(floor.max()))
    print("base f16 B=256, 64 images vs reference:", stats)
    assert np.median(re) <= 1.1 * np.median(floor), stats
    assert np.quantile(re, 0.9) <= 1.1 * np.quantile(floor, 0.9), stats
    assert re.max() <= 1.25e-3, stats
    order = np.argsort(-g["logits"], 1)[:, :5]
    assert (order == idx[pos]).all(), np.nonzero((order != idx[pos]).any(1))   # all 64 top-5 lists, no exemption
    dl = np.abs(logits[pos] - g["logits"]).max(axis=1)
    assert (np.abs(probs[pos] - g["probs"]).max(axis=1) <= 0.55 * dl + 1e-6).all()
    small = eng.vit_predict(m, base, 5, want_logits=True)
    assert np.array_equal(small[3], logits[pos])
    np.testing.assert_allclose(probs.sum(1), 1.0, atol=1e-3)
    assert (np.diff(val, axis=1) <= 0).all()
    assert np.array_equal(idx[:, 0], probs.argmax(1))
    assert np.isfinite(logits).all()
    m.close()


def test_loader_rejects_wrong_shapes_and_duplicate_names():
    """The reference loader compares all four extents of every tensor with the model's declaration (vit.cpp:633-641, "has wrong
    shape in model file") and keeps tensors in a name-keyed map; vitb200_create must do the same instead of accepting any tensor
    with the right element count: a transposed square weight would load silently and produce garbage."""
    vf = gf.read(model_path("micro", "f16"))

    def transpose_proj(entries):
        for e in entries:
            if e[0] == "blocks.0.attn.qkv.weight":
                e[3] = [e[3][1], e[3][0]]      # [3D, D] instead of [D, 3D]: same element count
    with pytest.raises(eng.VitB200Error) as ei:
        eng.vit_model_from_tensors(vf, edit=transpose_proj)
    assert "wrong shape" in str(ei.value) and "blocks.0.attn.qkv.weight" in str(ei.value)

    def flat_pos(entries):
        for e in entries:
            if e[0] == "pos_embed":
                e[3] = [int(np.prod(e[3]))]    # 1-D with the right count
    with pytest.raises(eng.VitB200Error) as ei:
        eng.vit_model_from_tensors(vf, edit=flat_pos)
    assert "wrong shape" in str(ei.value)

    def duplicate(entries):
        return entries + [entries[5]]
    with pytest.raises(eng.VitB200Error) as ei:
        eng.vit_model_from_tensors(vf, edit=duplicate)
    assert "duplicate tensor" in str(ei.value)

    # and the untouched list loads and matches the file path bit for bit
    m1 = eng.vit_model_from_tensors(vf, max_batch=2)
    m2 = eng.vit_model_load(model_path("micro", "f16"), 0, 2)
    imgs = gf.synthetic_images(2, vf.img_size, seed=3)
    assert np.array_equal(eng.vit_predict(m1, imgs, 5, want_logits=True)[3], eng.vit_predict(m2, imgs, 5, want_logits=True)[3])
    m1.close()
    m2.close()


@pytest.mark.parametrize("classes", [10, 1001, 21843])
def test_class_counts_that_are_not_a_multiple_of_four(classes, tmp_path):
    """ImageNet-21k heads have 21843 classes (the reference runs them); the head GEMM pads the class count to a multiple of 4
    internally (zero weight rows through TMA out-of-bounds fill, zero bias) and every output stays dense [batch][num_classes].
    21843 floats also exceed the 48 KB default of the soft-max kernel's dynamic shared memory (opt-in up to 227 KB)."""
    path = str(tmp_path / f"micro-c{classes}.gguf")
    gf.write_synthetic(path, "micro", 1, classes=classes, seed=5)
    vf = gf.read(path)
    om = rs.OracleModel(vf, gf.tensor_specs)
    imgs = gf.synthetic_images(3, vf.img_size, seed=9)
    m = eng.vit_model_load(path, 0, 4)
    probs, idx, val, logits = eng.vit_predict(m, imgs, 5, want_logits=True)
    assert probs.shape == (3, classes) and logits.shape == (3, classes)
    p_ref, l_ref = om.forward_batch(imgs)
    assert rel_err(logits, l_ref).max() <= 1.5e-3
    assert (idx[:, 0] == l_ref.argmax(1)).all()
    np.testing.assert_allclose(probs.sum(1), 1.0, atol=1e-3)
    assert np.abs(probs - p_ref).max() <= 1e-3
    # k larger than the class count is clamped: the tail is (-1, 0)
    if classes == 10:
        p2, i2, v2 = eng.vit_predict(m, imgs, 12)
        assert (i2[:, 10:] == -1).all() and (v2[:, 10:] == 0).all() and (np.sort(i2[:, :10], 1) == np.arange(10)).all()
    m.close()


def test_fused_layernorm_path_is_bit_identical(monkeypatch):
    """VITB200_FUSED_LN=1 applies the block LayerNorms inside the proj / fc2 residual epilogues (row-group completion counters +
    dedicated LayerNorm warps behind a shared-memory queue).  It is opt-in because it measured slower than the stand-alone kernel,
    but it must stay correct: same arithmetic, so logits are bit-identical, including a ragged batch whose last M tile is partial
    and a geometry with a 128-column N tile (micro: hidden 128)."""
    for cfg, n in (("micro", 5), ("base", 3)):
        imgs = gf.synthetic_images(n, gf.CONFIGS[cfg][4], seed=12)
        monkeypatch.delenv("VITB200_FUSED_LN", raising=False)
        m = eng.vit_model_load(model_path(cfg, "f16"), 0, 8)
        want = eng.vit_predict(m, imgs, 5, want_logits=True)
        m.close()
        monkeypatch.setenv("VITB200_FUSED_LN", "1")
        m = eng.vit_model_load(model_path(cfg, "f16"), 0, 8)
        got = eng.vit_predict(m, imgs, 5, want_logits=True)
        launches = m.last_launch_count()
        m.close()
        assert np.array_equal(got[3], want[3]) and np.array_equal(got[1], want[1])
        L = gf.CONFIGS[cfg][1]
        assert launches == 3 + 1 + 5 * L + 3   # patchify + cls rows + patch GEMM, first LayerNorm, 5 kernels per block, pooled LN + head + soft-max: no other LayerNorm launches except the first block's and the pooled final one


def test_error_paths():
    m = eng.vit_model_load(model_path("micro", "f16"), 0, 2)
    imgs = gf.synthetic_images(3, m.img_size, seed=1)
    with pytest.raises(eng.VitB200Error) as ei:
        eng.vit_predict(m, imgs, 5)  # batch > max_batch
    assert "out of range" in str(ei.value)
    with pytest.raises(eng.VitB200Error):
        eng.vit_predict(m, imgs[:1], 64)  # k too large
    m.close()


_NEEDS_QUANTIZE = pytest.mark.skipif(not os.path.exists(ref.QUANTIZE_BIN), reason="q4 / q5 files are written by the reference's quantize binary (oracle/_ref), not built")


@pytest.mark.parametrize("cfg,fmt", [("micro", "q8_0"), ("tiny", "q8_0"), ("base", "q8_0")] +
                         [pytest.param(c, f, marks=_NEEDS_QUANTIZE) for c, f in
                          [("micro", "q4_0"), ("micro", "q4_1"), ("micro", "q5_0"), ("micro", "q5_1"),
                           ("tiny", "q4_0"), ("tiny", "q5_1"), ("base", "q4_1"), ("base", "q5_0")]])
def test_quantised_model_file_top_k_and_noise_floor(cfg, fmt):
    """BASELINE.json configs[4] format (q8_0) and the other block formats vit_model_load accepts (vit.cpp:645-672: q4_0, q4_1,
    q5_0, q5_1), files written by the reference's own quantize.  The reference multiplies the integer weights with activations
    quantised on the fly to int8; no non-bit-identical implementation gets closer than ~1.6e-2 to that (SURVEY.md 7.4; the
    dequantised-weight x f16-activation recipe measured on the CPU sits at 1.0e-2..2.0e-2 for every format), so the binding
    criteria are identical top-1, gap-aware top-5 and an error at that floor, against the reference's own output."""
    g = np.load(os.path.join(GOLD, f"{cfg}_{fmt}.npz"))
    m = eng.vit_model_load(model_path(cfg, fmt), 0, 4)
    imgs = gf.synthetic_images(int(g["n_images"]), m.img_size, seed=int(g["image_seed"]))
    probs, idx, val, logits = eng.vit_predict(m, imgs, 5, want_logits=True)
    re = rel_err(logits, g["logits"])
    # measured floor of ANY dequantised-weight x f16-activation implementation against the reference's integer dot (CPU, restatement
    # on the dequantised weights): 1.0e-2 .. 2.0e-2; q8_0 (the BASELINE config) sits at the low end
    assert re.max() <= (2.5e-2 if fmt == "q8_0" else 3.5e-2), re
    order = np.argsort(-g["logits"], 1)
    for b in range(imgs.shape[0]):
        gaps = -np.diff(g["logits"][b, order[b, :6]])
        err = np.abs(logits[b] - g["logits"][b]).max()
        if gaps.min() > 2.5 * err:
            assert (idx[b] == order[b, :5]).all()
        assert idx[b, 0] == order[b, 0]
    m.close()


def test_f32_model_file_loads_and_matches_within_f16_weight_rounding():
    """ftype 0 files (f32 block weights, f16 patch kernel): weights are rounded to f16 at upload, activations follow the f16
    recipe; the reference runs f32 x f32 there, so agreement is at the f16-recipe noise level."""
    g = np.load(os.path.join(GOLD, "micro_f32.npz"))
    m = eng.vit_model_load(model_path("micro", "f32"), 0, 4)
    imgs = gf.synthetic_images(int(g["n_images"]), m.img_size, seed=int(g["image_seed"]))
    probs, idx, val, logits = eng.vit_predict(m, imgs, 5, want_logits=True)
    assert rel_err(logits, g["logits"]).max() <= 5e-3
    assert (idx[:, 0] == g["logits"].argmax(1)).all()
    m.close()


def test_smoke_entry_point():
    import __graft_entry__ as ge
    ge.smoke()


@pytest.mark.skipif(not (os.path.exists(ref.VIT_REF_BIN) and os.path.exists(os.path.join(os.path.dirname(ref.VIT_REF_BIN), "vit_b200_cli"))),
                    reason="reference CLI binaries (oracle/_ref) not shipped")
def test_reference_cli_runs_unmodified_on_the_b200_engine(tmp_path):
    """Drop-in check at the CLI level: the reference's own main.cpp + loader + stb_image + bicubic preprocess, linked against
    integration/vit_predict_b200.cpp + libvitb200.so (oracle/_ref/vit_b200_cli), must print the same top-5 lines as the stock
    reference binary (oracle/_ref/vit_ref) for the same model file and image."""
    import subprocess
    rng = np.random.default_rng(12)
    img = rng.integers(0, 256, size=(300, 280, 3), dtype=np.uint8)
    ppm = tmp_path / "img.ppm"
    with open(ppm, "wb") as f:
        f.write(b"P6\n280 300\n255\n" + img.tobytes())
    model = model_path("tiny", "f16")

    def top_lines(binary):
        r = subprocess.run([binary, "-m", model, "-i", str(ppm), "-k", "5", "-t", "4"], capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stderr[-2000:]
        return [l.strip() for l in r.stdout.splitlines() if l.startswith(" > ")]

    want = top_lines(ref.VIT_REF_BIN)
    got = top_lines(os.path.join(os.path.dirname(ref.VIT_REF_BIN), "vit_b200_cli"))
    assert len(want) == 5 and len(got) == 5
    assert [l.split(":")[0] for l in got] == [l.split(":")[0] for l in want]          # same labels, same order
    for g, w in zip(got, want):
        assert abs(float(g.split(":")[1]) - float(w.split(":")[1])) <= 0.011           # printed with %.2f


@pytest.mark.skipif(not ref.available(), reason="oracle/_ref not shipped")
@pytest.mark.parametrize("bilinear", [False, True])
def test_gpu_preprocess_matches_reference_bit_for_bit(bilinear):
    """SURVEY.md 8(f) rank 1: vit_image_preprocess on the GPU (bicubic default / bilinear), including the reference's quirks
    (no half-pixel offset in bicubic, clamp-to-edge, double-precision cubic coefficients, round-to-u8 before normalising)."""
    rng = np.random.default_rng(2)
    sizes = [(300, 280), (224, 224), (97, 131), (512, 333), (64, 640)]  # (ny, nx): down-, identity-, up-scaling, odd aspect
    imgs = [rng.integers(0, 256, size=(ny, nx, 3), dtype=np.uint8) for ny, nx in sizes]
    # a smooth image too (random noise alone under-samples the interpolation arithmetic)
    yy, xx = np.mgrid[0:400, 0:300]
    imgs.append(np.stack([(127 + 120 * np.sin(xx / 17.0)), (127 + 120 * np.cos(yy / 23.0)), ((xx + yy) % 256)], -1).astype(np.uint8))
    path = model_path("tiny", "f16")
    rm = ref.RefModel(path)
    m = eng.vit_model_load(path, 0, 8)
    got, _, _, _, _ = eng.vit_image_preprocess_predict(m, imgs, bilinear=bilinear, predict=False)
    for b, im in enumerate(imgs):
        want = rm.preprocess(im, bilinear=bilinear)
        mism = (got[b] != want)
        # the normalised values are (u8 - mean)/std: any difference is a whole u8 level.  Bicubic (the reference default)
        # reproduces the compiled reference's fused multiply-adds; in the bilinear path gcc fused the three unrolled channel
        # iterations differently from each other, which is not replicated: a few values per 10^4 land one level off.
        assert mism.mean() <= (5e-4 if bilinear else 2e-5), (b, im.shape, float(mism.mean()))
        assert np.abs(got[b] - want).max() <= 1.01 / 57.0
    m.close()
    rm.close()


def test_forward_u8_end_to_end_vs_reference_pipeline():
    """u8 image -> GPU preprocess -> GPU forward  vs  reference preprocess -> reference vit_predict."""
    rng = np.random.default_rng(4)
    imgs = [rng.integers(0, 256, size=(260, 310, 3), dtype=np.uint8) for _ in range(3)]
    path = model_path("tiny", "f16")
    m = eng.vit_model_load(path, 0, 4)
    f32, probs, idx, val, logits = eng.vit_image_preprocess_predict(m, imgs, topk=5)
    for b, l_ref in enumerate(LIVE["u8_s4_tiny_f16_logits"]):
        assert np.abs(logits[b] - l_ref).max() <= 1.25e-3 * np.abs(l_ref).max()
        assert idx[b, 0] == l_ref.argmax()
    m.close()


def test_in_process_sharding_over_all_visible_gpus():
    """SURVEY.md 8e process model: one host thread, one engine per GPU, contiguous image shards, no collective.  With a single
    visible GPU this still exercises the sharding arithmetic (two engines on device 0)."""
    import torch
    n_dev = torch.cuda.device_count()
    devs = list(range(n_dev)) if n_dev > 1 else [0, 0]
    path = model_path("tiny", "f16")
    models = [eng.vit_model_load(path, d, 4) for d in devs]
    imgs = gf.synthetic_images(7, models[0].img_size, seed=6)  # ragged: 7 images over the engines
    probs, idx, val = eng.vit_predict_sharded(models, imgs, 5)
    p1, i1, v1 = eng.vit_predict(models[0], imgs[:4], 5)
    assert np.array_equal(probs[:4], p1) and np.array_equal(idx[:4], i1)
    p2, i2, v2 = eng.vit_predict(models[-1], imgs[4:], 5)
    assert np.array_equal(idx[4:], i2)
    np.testing.assert_allclose(probs[4:], p2, rtol=0, atol=1e-6)
    # pipelined form: two global batches in flight from one host thread, then one wait for everything
    imgs2 = gf.synthetic_images(7, models[0].img_size, seed=7)
    outs = [(np.empty((7, models[0].num_classes), np.float32), np.empty((7, 5), np.int32), np.empty((7, 5), np.float32)) for _ in range(2)]
    eng.vit_predict_sharded_async(models, imgs, *outs[0])
    eng.vit_predict_sharded_async(models, imgs2, *outs[1])
    eng.sync_all(models)
    assert np.array_equal(outs[0][0], probs) and np.array_equal(outs[0][1], idx)
    pb, ib, vb = eng.vit_predict_sharded(models, imgs2, 5)
    assert np.array_equal(outs[1][0], pb) and np.array_equal(outs[1][1], ib) and np.array_equal(outs[1][2], vb)
    for m in models:
        m.close()


def test_gguf_container_loads_and_matches_the_legacy_file(tmp_path):
    """SURVEY.md 8(f) rank 3: the same weights in a true GGUF v3 container (oracle by construction: bit-identical logits to the
    legacy file the reference loads), including BF16 tensors for the bf16 checkpoint case."""
    imgs = gf.synthetic_images(3, 64, seed=17)
    legacy = eng.vit_model_load(model_path("micro", "f16"), 0, 4)
    want = eng.vit_predict(legacy, imgs, 5, want_logits=True)
    dst = str(tmp_path / "micro-f16.gguf")
    gf.legacy_to_gguf(model_path("micro", "f16"), dst)
    m = eng.vit_model_load(dst, 0, 4)
    got = eng.vit_predict(m, imgs, 5, want_logits=True)
    assert np.array_equal(got[3], want[3]) and np.array_equal(got[1], want[1])
    assert m.label(7) == legacy.label(7) == "LABEL_7"
    m.close()
    legacy.close()

    imgs = gf.synthetic_images(2, 224, seed=18)
    legacy = eng.vit_model_load(model_path("tiny", "bf16w"), 0, 2)   # bf16-representable values in the f32 container
    want = eng.vit_predict(legacy, imgs, 5, want_logits=True)
    dst = str(tmp_path / "tiny-bf16.gguf")
    gf.legacy_to_gguf(model_path("tiny", "bf16w"), dst, "bf16")      # the same values as real BF16 tensors (ggml type 30)
    assert os.path.getsize(dst) < 0.6 * os.path.getsize(model_path("tiny", "bf16w"))
    m = eng.vit_model_load(dst, 0, 2)
    got = eng.vit_predict(m, imgs, 5, want_logits=True)
    assert np.array_equal(got[3], want[3])
    m.close()
    legacy.close()


@pytest.mark.parametrize("cfg", ["vitstr_micro", "vitstr_tiny"])
def test_vitstr_extension_matches_the_reference(cfg):
    """SURVEY.md 8(f) rank 4: the reference's ViTSTR extension (extensions/vitstr.cpp) -- same encoder on a 1-channel image,
    classifier (LayerNorm + head + soft-max) over the first 25 tokens -- against fixtures generated by the extension itself
    (tests/golden/make_golden.py) and, when the compiled extension travelled, against a live run.  Same tolerances as the
    classifier: the 25 x 96 logits of an image are one vector for the relative-error metric."""
    g = np.load(os.path.join(GOLD, f"{cfg}_f16.npz"))
    m = eng.vit_model_load(model_path(cfg, "f16"), 0, 4, head_tokens=25)
    assert (m.in_chans, m.head_tokens) == (1, 25)
    n = int(g["n_images"])
    imgs = gf.synthetic_gray_images(n, m.img_size, seed=int(g["image_seed"]))
    probs, idx, val, logits = eng.vit_predict(m, imgs, 5, want_logits=True)
    assert logits.shape == (n, 25, m.num_classes) and idx.shape == (n, 25, 5)
    lf, rf = logits.reshape(n, -1), g["logits"].reshape(n, -1)
    re = np.abs(lf - rf).max(1) / np.abs(rf).max(1)
    assert np.median(re) <= 1e-3 and re.max() <= 1.5e-3, re
    assert (np.linalg.norm(lf - rf, axis=1) <= 1.25e-3 * np.linalg.norm(rf, axis=1)).all()
    # greedy decode = per-token argmax (vitstr.cpp:1029-1052): identical wherever the reference's top-2 gap exceeds the error
    top2 = np.sort(g["logits"], -1)[..., -2:]
    clear = (top2[..., 1] - top2[..., 0]) > 2.5 * np.abs(logits - g["logits"]).max(-1)
    assert clear.mean() > 0.9 and (idx[..., 0] == g["logits"].argmax(-1))[clear].all()
    dl = np.abs(logits - g["logits"]).max(-1)
    assert (np.abs(probs - g["probs"]).max(-1) <= 0.55 * dl + 1e-6).all()
    np.testing.assert_allclose(probs.sum(-1), 1.0, atol=1e-3)
    if ref.vitstr_available():
        rm = ref.VitstrRefModel(model_path(cfg, "f16"))
        extra = gf.synthetic_gray_images(1, m.img_size, seed=77)
        p_ref, l_ref = rm.predict(extra[0], n_threads=8)
        got = eng.vit_predict(m, extra, 5, want_logits=True)[3][0]
        assert np.abs(got - l_ref).max() <= 1.5e-3 * np.abs(l_ref).max()
        rm.close()
    # a 3-channel classifier entry point must refuse this model's input
    with pytest.raises(eng.VitB200Error):
        eng.vit_image_preprocess_predict(m, [np.zeros((40, 40, 3), np.uint8)])
    m.close()


def test_batch_size_sweep_is_bit_identical_and_stable():
    """Every batch size from 1 up past the eager/graph switch (8192 tokens = 41 images of 197 tokens) and the persistent-grid
    boundaries (fewer (image, head) problems than SMs, M tails of the 256-row GEMM tiles): the last image of each batch must
    come out bit-identical to running it alone, three calls in a row (graph capture on the second, replay on the third)."""
    m = eng.vit_model_load(model_path("tiny", "f16"), 0, 64)
    imgs = gf.synthetic_images(64, m.img_size, seed=41)
    alone = {}
    for B in (1, 2, 3, 5, 7, 12, 13, 25, 40, 41, 42, 49, 63, 64):
        want = alone.setdefault(B - 1, eng.vit_predict(m, imgs[B - 1:B], 5, want_logits=True)[3][0])
        for rep in range(3):
            p, i, v, l = eng.vit_predict(m, imgs[:B], 5, want_logits=True)
            assert np.array_equal(l[B - 1], want), (B, rep)
            assert np.isfinite(l).all() and abs(float(p.sum()) - B) < 1e-2 * B
    m.close()


_BENCH_B200 = os.path.join(os.path.dirname(ref.VIT_REF_BIN), "benchmark_b200")


@pytest.mark.skipif(not (os.path.exists(_BENCH_B200) and ref.available()), reason="accuracy harness binary (oracle/_ref) not shipped")
def test_batched_accuracy_harness_on_a_synthetic_image_folder(tmp_path):
    """The reference's accuracy harness (tests/benchmark.cpp: <dataset>/<class>/<image> folders, ../classnames.json, one
    "file,true,predicted" line per image, "Top-1 Accuracy") running batched on the engine (integration/benchmark_b200.cpp: reference
    image decoder, GPU preprocess + forward through vitb200_forward_u8_async, batch 4 here so the two pipeline slots and a ragged
    last batch are exercised).  Expected predictions come from the reference pipeline itself (its preprocess + its vit_predict)."""
    import json
    import subprocess
    rng = np.random.default_rng(21)
    root = tmp_path / "data"
    names = [f"class_{i}" for i in range(1000)]
    (tmp_path / "classnames.json").write_text(json.dumps(names))
    model = model_path("tiny", "f16")
    rm = ref.RefModel(model)
    expect = {}
    dirs = ["class_7", "class_421", "class_900"]
    n_imgs = 0
    for d in dirs:
        (root / d).mkdir(parents=True)
        for j in range(3 if d != "class_900" else 5):
            h, w = int(rng.integers(120, 300)), int(rng.integers(120, 300))
            yy, xx = np.mgrid[0:h, 0:w]
            img = np.stack([(xx * 3 + j * 40) % 256, (yy * 2 + 90) % 256, rng.integers(0, 256, size=(h, w))], -1).astype(np.uint8)
            with open(root / d / f"img{j}.ppm", "wb") as f:
                f.write(b"P6\n%d %d\n255\n" % (w, h) + img.tobytes())
            p_ref, l_ref = rm.predict(rm.preprocess(img), n_threads=8)
            order = np.argsort(-l_ref)
            expect[(d, f"img{j}.ppm")] = (names[int(order[0])], float(l_ref[order[0]] - l_ref[order[1]]), float(np.abs(l_ref).max()))
            n_imgs += 1
        (root / d / "notes.txt").write_text("not an image")
    rm.close()
    out = tmp_path / "pred.txt"
    r = subprocess.run([_BENCH_B200, model, str(root), "4", str(out), "4"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l.split(",") for l in out.read_text().splitlines()]
    assert len(lines) == 3 + 3 + 4                      # num_images_per_class = 4 caps the 5-image class
    correct = 0
    for fname, truth, pred in lines:
        want, gap, scale = expect[(truth, fname)]
        if gap > 2.5e-3 * scale:                        # a top-1 decided by less than the parity noise may legitimately flip
            assert pred == want, (fname, truth, pred, want)
        correct += truth == pred
    acc = [l for l in r.stdout.splitlines() if l.startswith("Top-1 Accuracy:")]
    assert acc and abs(float(acc[0].split(":")[1].strip().rstrip("%")) - 100.0 * correct / len(lines)) < 1e-3


_VITSTR_REF = os.path.join(os.path.dirname(ref.VIT_REF_BIN), "vitstr_ref")
_VITSTR_B200 = os.path.join(os.path.dirname(ref.VIT_REF_BIN), "vitstr_b200_cli")


@pytest.mark.skipif(not (os.path.exists(_VITSTR_REF) and os.path.exists(_VITSTR_B200)), reason="ViTSTR CLI binaries (oracle/_ref) not shipped")
def test_vitstr_cli_runs_unmodified_on_the_b200_engine(tmp_path):
    """Drop-in check for the extension at the CLI level: its own main.cpp + loader + stb_image + grayscale preprocess linked
    against integration/vitstr_predict_b200.cpp + libvitb200.so must decode the same string as the stock extension binary
    (greedy per-token argmax; random weights leave a few near-ties, so all but at most two of the 24 characters must agree)."""
    import re
    import subprocess
    rng = np.random.default_rng(12)
    img = rng.integers(0, 256, size=(120, 300, 3), dtype=np.uint8)
    ppm = tmp_path / "word.ppm"
    with open(ppm, "wb") as f:
        f.write(b"P6\n300 120\n255\n" + img.tobytes())
    model = model_path("vitstr_tiny", "f16")

    def decode(binary):
        r = subprocess.run([binary, "-m", model, "-i", str(ppm), "-t", "4"], capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stderr[-2000:]
        block = r.stdout.split("------------------")[1].strip().splitlines()
        return re.findall(r"LABEL_\d+", block[0]), float(block[1].split(":")[1])

    want, want_score = decode(_VITSTR_REF)
    got, got_score = decode(_VITSTR_B200)
    assert len(want) == 24 and len(got) == len(want)
    assert sum(a == b for a, b in zip(got, want)) >= 22, (got, want)
    assert abs(got_score - want_score) <= 0.011
