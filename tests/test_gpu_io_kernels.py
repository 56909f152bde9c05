"""GPU tests of the kernels at the two ends of the forward pass, each on its own against a float64 numpy reference: the patch embedding
(patchify + the patch GEMM's epilogue, through the `embed` tap) at every patch size and channel count the loader accepts, and the final
soft-max + top-k (vitb200_test_softmax_topk) on both sides of each storage threshold of its working row."""
import numpy as np
import pytest

from tests.util import pkg, gf

eng = pkg.engine
pytestmark = pytest.mark.gpu


# ---- soft-max / top-k ------------------------------------------------------------------------------------------------------------
# class counts on both sides of every storage threshold of the working row: the 48 KB default shared memory (12224 floats next to the
# kernel's static arrays; 12288 floats are exactly 48 KB), the 227 KB opt-in limit (57856 floats), global scratch beyond it
SOFTMAX_CLASSES = [1, 2, 3, 5, 96, 1000, 1001, 12224, 12288, 12289, 21843, 57856, 57857]
ROW_KINDS = ("random", "all_equal", "dup_max", "f16_ties", "one_dominant", "huge")


def _logit_rows(R, C, rng):
    """R rows of C logits, row r of kind ROW_KINDS[r % 6] (row 0 random)."""
    x = np.empty((R, C), np.float32)
    for r in range(R):
        kind = ROW_KINDS[r % len(ROW_KINDS)]
        row = (rng.standard_normal(C) * 3).astype(np.float32)
        if kind == "all_equal":
            row[:] = np.float32(rng.uniform(-5, 5))
        elif kind == "dup_max" and C > 7:            # exact duplicate maxima at 7 and 3: top-2 = (3, 7)
            row[7] = row[3] = row.max() + np.float32(1.5)
        elif kind == "f16_ties":                     # distinct logits whose f16(x - max) coincide: equal probabilities
            row = rng.uniform(-8, -2, C).astype(np.float32)
            cols = rng.choice(C, size=min(C, 12), replace=False)
            row[cols] = np.float32(-1.0) - np.arange(cols.size, dtype=np.float32) * np.float32(2.0 ** -14)
            row[cols[-1]] = 0.0
        elif kind == "one_dominant":                 # every other exponential underflows to 0: p = 1, then zeros by index
            row[int(rng.integers(0, C))] = row.max() + np.float32(80.0)
        elif kind == "huge":
            row = (rng.choice([-1e4, 1e4], C) + rng.uniform(-5, 5, C)).astype(np.float32)
        x[r] = row
    return x


def _softmax_ref(x):
    """The reference soft-max (ggml.c:10533-10558) in float64: e = f16(exp(f16(x - max))) with x - max the f32 difference the
    reference forms, p = e / sum(e)."""
    d = x - x.max(axis=1, keepdims=True)                                  # float32 arithmetic: exact RNE like the kernel
    e = np.exp(d.astype(np.float16).astype(np.float64)).astype(np.float16).astype(np.float64)
    return e, e / e.sum(axis=1, keepdims=True)


@pytest.mark.parametrize("C", SOFTMAX_CLASSES)
def test_softmax_topk_against_float64(C):
    """Probabilities within 2^-10 p + 2^-24 max p of the float64 restatement, >= 99 % of the f16 exponentials bit-identical (the
    kernel's ex2.approx may move an f16 rounding by one ulp; e is read back as f16(p / p_max), exact because the largest e is 1);
    top-k = the first k of a stable sort of the kernel's own probabilities by (-p, index), values = probs[idx], entries past C are
    (-1, 0).  Logits have pitch roundup4(C) with NaN in the padding columns, which the kernel must never read."""
    rng = np.random.default_rng(C)
    ldl = (C + 3) // 4 * 4
    kmax = 16
    for R in (1, 7, 300):
        x = _logit_rows(R, C, rng)
        lg = np.full((R, ldl), np.nan, np.float32)
        lg[:, :C] = x
        probs, idx, val = eng.test_softmax_topk(lg, C, kmax)
        e_ref, p_ref = _softmax_ref(x)
        assert np.isfinite(probs).all()
        err = np.abs(probs.astype(np.float64) - p_ref)
        tol = 2.0 ** -10 * p_ref + 2.0 ** -24 * p_ref.max(axis=1, keepdims=True)
        assert (err <= tol).all(), (R, np.unravel_index(np.argmax(err - tol), err.shape), float((err / tol).max()))
        e_k = (probs.astype(np.float64) / probs.max(axis=1, keepdims=True)).astype(np.float16).astype(np.float64)
        assert (e_k == e_ref).mean() >= 0.99, (R, float((e_k == e_ref).mean()))
        n = min(kmax, C)
        want = np.argsort(-probs, axis=1, kind="stable")[:, :n]
        assert np.array_equal(idx[:, :n], want), (R, np.nonzero((idx[:, :n] != want).any(1))[0][:5])
        assert np.array_equal(val[:, :n], np.take_along_axis(probs, want.astype(np.int64), 1))
        assert (idx[:, n:] == -1).all() and (val[:, n:] == 0).all()
        if C > 7 and R >= 3:   # the duplicate maxima of row 2 come out as (3, 7)
            assert list(idx[2, :2]) == [3, 7]
        if R == 7:             # fewer entries: the same probabilities, a prefix of the same list
            for k in (0, 1, 5):
                p2, i2, v2 = eng.test_softmax_topk(lg, C, k)
                assert np.array_equal(p2, probs)
                assert np.array_equal(i2, idx[:, :k]) and np.array_equal(v2, val[:, :k])


# ---- patch embedding ------------------------------------------------------------------------------------------------------------
# (hidden, patch P, image side S, channels, batch): every patch size / channel count the loader accepts; hidden 192 leaves a partial
# 128-column N tile; M = batch * (S / P)^2 spans two or more 256-row tiles with a partial last one
PATCH_CASES = [(128, 8, 64, 3, 9), (128, 14, 56, 3, 37), (128, 16, 64, 3, 37), (192, 16, 224, 3, 3), (128, 32, 128, 3, 37),
               (128, 16, 96, 1, 15), (128, 8, 64, 1, 9)]


@pytest.fixture(scope="module")
def patch_models(tmp_path_factory):
    d = tmp_path_factory.mktemp("patch_models")
    paths = {}

    def get(hidden, P, S, ch):
        key = (hidden, P, S, ch)
        if key not in paths:
            paths[key] = str(d / f"h{hidden}-p{P}-s{S}-c{ch}.gguf")
            gf.write_synthetic(paths[key], (hidden, 1, hidden // 64, P, S), 1, classes=40, seed=P + S + ch, in_chans=ch)
        return paths[key]
    return get


def _embed_ref(vf, imgs, ch):
    """Token rows X[b, 1 + p] = A W^T + bias + pos[1 + p] in float64 on the f16-rounded pixels, im2col k = c P^2 + ky P + kx."""
    P, S, D = vf.patch_size, vf.img_size, vf.hidden_size
    G, B = S // P, imgs.shape[0]
    x = imgs.reshape(B, G, P, G, P, ch).astype(np.float16).astype(np.float64)             # [b][py][ky][px][kx][c]
    A = x.transpose(0, 1, 3, 5, 2, 4).reshape(B, G * G, ch * P * P)                       # [b][py*G + px][c][ky][kx]
    W = vf.tensors["patch_embed.proj.weight"].astype(np.float64).reshape(D, ch * P * P)
    bias = vf.tensors["patch_embed.proj.bias"].astype(np.float64).reshape(D)
    pos = vf.tensors["pos_embed"].astype(np.float64).reshape(-1, D)
    return A @ W.T + bias + pos[1:]


def _check_embed(embed, vf, imgs, ch):
    D = vf.hidden_size
    ref = _embed_ref(vf, imgs, ch)
    tok = embed[:, 1:].astype(np.float64)
    bound = 2e-5 * max(1.0, np.abs(ref).max())
    assert np.abs(tok - ref).max() <= bound, (float(np.abs(tok - ref).max()), bound, np.unravel_index(np.abs(tok - ref).argmax(), ref.shape))
    cls = vf.tensors["cls_token"].astype(np.float32).reshape(D) + vf.tensors["pos_embed"].astype(np.float32).reshape(-1, D)[0]
    assert np.array_equal(embed[:, 0], np.broadcast_to(cls, (imgs.shape[0], D)))


def _images(ch, B, S, seed):
    return gf.synthetic_images(B, S, seed=seed) if ch == 3 else gf.synthetic_gray_images(B, S, seed=seed)


@pytest.mark.parametrize("hidden,P,S,ch,B", PATCH_CASES)
def test_patch_embedding_against_float64(hidden, P, S, ch, B, patch_models, monkeypatch):
    """(a) The default path (patchify kernel for P, C + TMA-fed GEMM, EPI_PATCH_F32) within the f32-output bar of test_gemm_against_numpy,
    class-token rows bit-equal to f32(cls + pos[0]); (b) for P = 16, C = 3 the opt-in gathered variant (VITB200_PATCH_GATHER=1, read per
    call) to the same bound; (d) for C = 3 the u8 path, whose preprocess kernel writes the patch matrix itself (padding columns included
    for P = 14): its logits must be bit-identical to vit_predict on the f32 images it returns."""
    monkeypatch.delenv("VITB200_PATCH_GATHER", raising=False)
    monkeypatch.delenv("VITB200_CTA_GROUP", raising=False)
    path = patch_models(hidden, P, S, ch)
    vf = gf.read(path)
    imgs = _images(ch, B, S, seed=P * 100 + S)
    m = eng.vit_model_load(path, 0, B)
    assert m.in_chans == ch
    _, _, taps = eng.vit_predict_debug(m, imgs, 0, taps=("embed",))
    _check_embed(taps["embed"], vf, imgs, ch)
    if P == 16 and ch == 3:
        monkeypatch.setenv("VITB200_PATCH_GATHER", "1")
        _, _, gathered = eng.vit_predict_debug(m, imgs, 0, taps=("embed",))
        monkeypatch.delenv("VITB200_PATCH_GATHER")
        # same f16 operands, but not bit-identical to (a): its A producers fill the three channels of one 4-row group of kernel rows
        # into consecutive pipeline stages, so the 64-wide K blocks reach the f32 accumulator in the order (ky group, channel)
        # instead of k order -- a different f32 summation order (about 2e-6 apart on these cases), held to the same bound
        _check_embed(gathered["embed"], vf, imgs, ch)
    if ch == 3:
        rng = np.random.default_rng(S + P)
        u8 = [rng.integers(0, 256, size=(int(rng.integers(1, 2 * S)), int(rng.integers(1, 2 * S)), 3), dtype=np.uint8) for _ in range(B)]
        f32, _, idx_u8, _, logits_u8 = eng.vit_image_preprocess_predict(m, u8, topk=5)
        _, idx, _, logits = eng.vit_predict(m, f32, 5, want_logits=True)
        assert np.array_equal(logits_u8, logits) and np.array_equal(idx_u8, idx)
    m.close()


@pytest.mark.parametrize("hidden,P,S,ch,B", PATCH_CASES)
def test_patch_embedding_one_cta_gemms(hidden, P, S, ch, B, patch_models, monkeypatch):
    """(c) The same check with VITB200_CTA_GROUP=1 set before the model is created: every GEMM runs its 1-CTA instantiation."""
    monkeypatch.delenv("VITB200_PATCH_GATHER", raising=False)
    monkeypatch.setenv("VITB200_CTA_GROUP", "1")
    path = patch_models(hidden, P, S, ch)
    vf = gf.read(path)
    imgs = _images(ch, B, S, seed=P * 100 + S)
    m = eng.vit_model_load(path, 0, B)
    _, _, taps = eng.vit_predict_debug(m, imgs, 0, taps=("embed",))
    m.close()
    _check_embed(taps["embed"], vf, imgs, ch)
