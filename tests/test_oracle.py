"""CPU tests (-m "not gpu") that PIN the oracle: oracle/restatement.py (plain-torch restatement) and
oracle/vq_oracle.c (C restatement of the VQ search) against tests/golden/*.pt, which oracle/make_golden.py
produced by running the unmodified reference.
"""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from oracle import restatement as R, synth
from oracle.make_golden import vq_inputs

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _load(name):
    return torch.load(os.path.join(GOLDEN, name), map_location="cpu", weights_only=False)


def _check_sample(t, s, rtol=2e-5):
    flat = t.reshape(-1)
    assert list(t.shape) == s["shape"]
    got = flat[:: s["step"]]
    assert torch.allclose(got, s["values"], rtol=rtol, atol=rtol * float(s["values"].abs().max()))
    assert abs(flat.double().norm().item() - s["norm"]) <= rtol * s["norm"]


@pytest.fixture(scope="module")
def vq_lib():
    from seed_b200.build import ORACLE_LIB, build_oracle

    build_oracle()
    lib = C.CDLL(ORACLE_LIB)
    lib.vq_oracle_argmin.restype = C.c_int
    return lib


def c_oracle(lib, z16, cb16, mode):
    zn = z16.contiguous().view(torch.int16).numpy().view(np.uint16)
    cn = cb16.contiguous().view(torch.int16).numpy().view(np.uint16)
    ids = np.zeros(zn.shape[0], dtype=np.int64)
    margin = np.zeros(zn.shape[0], dtype=np.float32)
    rc = lib.vq_oracle_argmin(zn.ctypes.data_as(C.c_void_p), cn.ctypes.data_as(C.c_void_p), zn.shape[0], cn.shape[0],
                              zn.shape[1], mode, ids.ctypes.data_as(C.c_void_p), margin.ctypes.data_as(C.c_void_p))
    assert rc == 0
    return torch.from_numpy(ids), torch.from_numpy(margin)


# ---------------------------------------------------------------------------------------------
# VQ: C oracle vs the reference's VectorQuantizer2.forward outputs (golden) in both dtypes
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("tag", ["spread", "default_init"])
def test_c_vq_oracle_matches_reference_vectors(vq_lib, tag):
    g = _load("vq_reference_expr.pt")[tag]
    z, cb = vq_inputs(tag)
    s = g["codebook_sample"]
    assert torch.equal(z, g["z"]) and list(cb.shape) == s["shape"]
    assert torch.equal(cb.reshape(-1)[:: s["step"]], s["values"])        # the codebook is the one the ids came from
    ids32, m32 = c_oracle(vq_lib, z, cb, 1)
    ids16, m16 = c_oracle(vq_lib, z, cb, 0)
    # exact wherever the oracle's own top-2 margin is not a floating-point tie; report would-be flips
    neq32 = ids32 != g["ids_fp32"]
    neq16 = ids16 != g["ids_fp16"]
    assert int(neq32.sum()) == 0, f"fp32 mode: {int(neq32.sum())} ids differ, margins {m32[neq32][:8]}"
    assert int(neq16.sum()) == 0, f"fp16 mode: {int(neq16.sum())} ids differ, margins {m16[neq16][:8]}"
    if tag == "default_init":
        # the degenerate case SURVEY.md section 7 describes: in half precision every distance collapses to |z|^2
        assert (g["ids_fp16"] == 0).float().mean() > 0.5


def test_c_vq_oracle_rejects_bad_args(vq_lib):
    assert vq_lib.vq_oracle_argmin(None, None, 1, 1, 32, 0, None, None) == -1


def test_torch_vq_expression_equals_c_oracle_on_random_rows(vq_lib):
    g = torch.Generator().manual_seed(5)
    z = (torch.randn(300, 32, generator=g) * 0.3).half()
    cb = (torch.randn(2048, 32, generator=g) * 0.3).half()
    ids32, _ = c_oracle(vq_lib, z, cb, 1)
    ref32, margin = R.vq_forward(z.float(), cb.float())
    safe = margin > 1e-5
    assert torch.equal(ids32[safe], ref32[safe])


# ---------------------------------------------------------------------------------------------
# encoder restatement vs golden (reference outputs)
# ---------------------------------------------------------------------------------------------
def _encoder_vs_golden(name):
    g = _load(name)
    c = g["config"]
    sd = synth.encoder_state_dict(c["vit_depth"], c["qformer_layers"], c["detok_depth"])
    x = synth.images(c["batch"])
    with torch.no_grad():
        out = R.encode(x, sd, c["vit_depth"], c["qformer_layers"])
        emb = R.detokenize(g["ids"], sd, c["detok_depth"])
    assert torch.equal(out["ids"], g["ids"])
    assert torch.allclose(out["z"].reshape(-1, 32), g["z"], atol=2e-5)
    _check_sample(out["vit"], g["vit"])
    _check_sample(out["image_embeds"], g["image_embeds"])
    _check_sample(out["query_output_up"], g["query_output_up"])
    if isinstance(g["qformer"], dict):
        _check_sample(out["qformer"], g["qformer"])
    else:
        assert torch.allclose(out["qformer"], g["qformer"], atol=5e-5)
    assert torch.allclose(emb, g["image_embeds_out"], atol=5e-5, rtol=1e-4)


def test_encoder_restatement_matches_golden_reduced():
    _encoder_vs_golden("encoder_d2_q2.pt")


def test_encoder_restatement_matches_golden_full_depth():
    """full 39-block ViT-g + 12-layer Q-Former + 4 de-tokenizer blocks, 2 images (about a minute on 8 cores)."""
    _encoder_vs_golden("encoder_full.pt")


def test_encoder_restatement_matches_reference_on_fresh_seeds():
    """the reference's get_codebook_indices / get_codebook_entry outputs on other weight and image seeds, with a
    de-tokenizer block (tests/golden/encoder_v1_q2_d1_seed77.pt)"""
    g = _load("encoder_v1_q2_d1_seed77.pt")
    c = g["config"]
    vd, ql, dd = c["vit_depth"], c["qformer_layers"], c["detok_depth"]
    sd = synth.encoder_state_dict(vd, ql, dd, seed=c["weights_seed"])
    x = synth.images(c["batch"], seed=c["images_seed"])
    with torch.no_grad():
        out = R.encode(x, sd, vd, ql)
        emb2 = R.detokenize(g["ids"], sd, dd)
    assert torch.equal(g["ids"], out["ids"])
    assert torch.allclose(g["query_output_up"], out["query_output_up"], atol=1e-5)
    assert torch.allclose(g["image_embeds_out"], emb2, atol=1e-5)


# ---------------------------------------------------------------------------------------------
# LLaMA restatement vs golden (reference llama_xformer outputs, prefill + one cached decode step)
# ---------------------------------------------------------------------------------------------
def test_llama_restatement_matches_golden():
    g = _load("llama_tiny.pt")
    c = g["config"]
    sd = synth.llama_state_dict(c["hidden"], c["layers"], c["ffn"], c["vocab"])
    with torch.no_grad():
        logits, hidden, past = R.llama_forward(sd, g["input_ids"], c["heads"], c["layers"])
        assert torch.allclose(logits, g["logits"], atol=2e-5, rtol=1e-4)
        assert torch.allclose(past[0][0], g["k0"], atol=1e-5)
        assert torch.allclose(past[1][1], g["v1"], atol=1e-5)
        nxt = logits[:, -1].argmax(-1, keepdim=True)
        assert torch.equal(nxt, g["next_ids"])
        logits2, _, _ = R.llama_forward(sd, nxt, c["heads"], c["layers"], past=past)
        assert torch.allclose(logits2, g["decode_logits"], atol=2e-5, rtol=1e-4)


def test_synth_is_deterministic_and_fp16_representable():
    a = synth.encoder_state_dict(1, 1, 0)
    b = synth.encoder_state_dict(1, 1, 0)
    for k in a:
        assert torch.equal(a[k], b[k])
        assert torch.equal(a[k], a[k].half().float()), k
    ids = synth.prompt_ids(2, 64, n_image_spans=1)
    assert ids[0, 1] == 32000 + 8192 and ids[0, 34] == 32000 + 8193
    assert ((ids[0, 2:34] >= 32000) & (ids[0, 2:34] < 32000 + 8192)).all()


# ----------------------------------------------------------------------------------------------
# resize oracle (oracle/resize_oracle.c) pinned against the installed Pillow -- the third-party code the
# reference's transforms actually execute (models/transforms.py:4-19, seed_llama_tokenizer.py:50-56)
# ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("filt", [2, 3])
@pytest.mark.parametrize("h,w", [(224, 224), (300, 400), (1000, 800), (64, 48), (225, 223), (1, 1), (7, 1000),
                                 (500, 333), (100, 224), (449, 448), (3000, 17), (501, 5), (500, 5), (5, 3000)])
def test_resize_oracle_matches_pillow(h, w, filt):
    from PIL import Image

    from seed_b200.build import ORACLE_LIB, build_oracle

    build_oracle()
    lib = C.CDLL(ORACLE_LIB)
    rng = np.random.default_rng(h * 31 + w + filt)
    img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    if h > 4:
        img[: h // 3] = (img[: h // 3] // 128) * 255
    ref = np.asarray(Image.fromarray(img, "RGB").resize((224, 224), Image.BILINEAR if filt == 2 else Image.BICUBIC))
    out = np.zeros((224, 224, 3), np.uint8)
    rc = lib.resize_oracle_u8(img.ctypes.data_as(C.c_void_p), h, w, 224, 224, filt, out.ctypes.data_as(C.c_void_p))
    assert rc == 0
    assert np.array_equal(out, ref)


# --------------------------------------------------------------------------------------------------
# sampler oracle (oracle/sampler_oracle.py): pinned against the published Philox vectors and against the
# `transformers` warpers the reference's generate() call runs (scripts/seed_llama_inference_8B.py:26-38)
# --------------------------------------------------------------------------------------------------
def test_philox_known_answers_and_c_host_function():
    from oracle import sampler_oracle as S

    # Random123 kat_vectors, philox4x32 with 10 rounds
    assert S.philox4x32_10((0, 0, 0, 0), (0, 0)) == [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]
    assert S.philox4x32_10((0xffffffff,) * 4, (0xffffffff,) * 2) == [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]
    assert S.philox4x32_10((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0)) == \
        [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]
    from seed_b200 import lib as L

    for seed, off, row in [(0, 0, 0), (1234, 5, 2), (2 ** 40 + 7, 2 ** 33 + 1, 3), (2 ** 63, 99, 0)]:
        u = S.philox_uniform(seed, off, row)
        assert 0.0 < float(u) <= 1.0
        assert float(u) == L.philox_uniform(seed, off, row)       # the library's host-side Philox (no GPU needed)


def test_sampler_oracle_matches_transformers_warpers():
    from transformers.generation.logits_process import TemperatureLogitsWarper, TopPLogitsWarper

    from oracle import sampler_oracle as S

    g = torch.Generator().manual_seed(3)
    for V, T, P in [(50, 1.0, 0.5), (1000, 0.7, 0.9), (40194, 1.0, 0.5), (333, 1.3, 0.05), (64, 1.0, 1.0)]:
        logits = (torch.randn(1, V, generator=g) * 3.0).half().float()     # fp16 logits: tied scores do occur
        ids = torch.zeros((1, 1), dtype=torch.long)
        warped = TemperatureLogitsWarper(T)(ids, logits.clone())
        if P < 1.0:
            warped = TopPLogitsWarper(P)(ids, warped)
        ref_probs = torch.softmax(warped, dim=-1)[0].double().numpy()
        x = logits[0].numpy()
        q, keep, margin = S.warp(x, T, P, ties="sort")                 # HF's rule incl. its (stable-sort) tie split
        assert margin > 1e-7                                           # the comparison below is not a coin flip
        assert (keep == (ref_probs > 0)).all()
        assert np.abs(q - ref_probs).max() < 1e-6
        # the threshold form used by the kernel: a superset that differs only by tokens tied with the least kept score
        _, keep_all, _ = S.warp(x, T, P)
        assert (keep_all | ~keep).all() and (x[keep_all & ~keep] == x[keep].min()).all()
    # tied scores at the nucleus boundary: HF's stable CPU sort keeps a suffix of the tie group, the threshold form all
    x = np.array([1.0, 3.0, 1.0, 1.0, 0.0], dtype=np.float32)
    _, keep_hf, _ = S.warp(x, 1.0, 0.9, ties="sort")
    _, keep_all, _ = S.warp(x, 1.0, 0.9, ties="all")
    assert keep_all.tolist() == [True, True, True, True, False] and keep_hf.sum() <= keep_all.sum() and keep_hf[1]
    # greedy = torch.argmax (first maximal index)
    x = np.array([0.5, 2.0, 2.0, -1.0], dtype=np.float32)
    assert S.sample_ref(x, False)[0] == int(torch.from_numpy(x).argmax()) == 1
