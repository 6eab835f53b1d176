"""TEST INFRASTRUCTURE ONLY -- generate tests/golden/*.pt by running the UNMODIFIED reference code
(/root/reference, through oracle/ref_shim.py) on the seeded synthetic weights of oracle/synth.py.

The reference ships no tests, golden vectors or fixtures (SURVEY.md section 4), so these files are the
known-answer vectors for the path.  Run in the build container (the GPU box has no /root/reference):

    python -m oracle.make_golden [--full]

Each file records the generating configuration, the reference outputs, and enough of the intermediate
activations (strided samples + norms) to localise a mismatch.
"""
from __future__ import annotations

import os
import sys
import time

import torch

from . import ref_shim, synth

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def _sample(t: torch.Tensor, max_elems: int = 4096) -> dict:
    flat = t.reshape(-1)
    step = max(1, flat.numel() // max_elems)
    return {"shape": list(t.shape), "step": step, "values": flat[::step].clone(), "norm": flat.double().norm().item(),
            "mean": flat.double().mean().item()}


def encoder_golden(name: str, vit_depth: int, qformer_layers: int, detok_depth: int, batch: int) -> None:
    t0 = time.time()
    model = ref_shim.build_reference_quantizer(vit_depth, qformer_layers, detok_depth)
    sd = synth.encoder_state_dict(vit_depth, qformer_layers, detok_depth)
    missing, unexpected = model.load_state_dict(sd, strict=False)
    allowed = ("pos_embed", "blocks.", "Qformer.cls", "Qformer.bert.embeddings.position_ids")
    bad = [k for k in missing if not k.startswith(allowed)]
    assert not bad and not unexpected, (bad, unexpected)
    x = synth.images(batch)
    taps = {}
    hooks = [
        model.visual_encoder.register_forward_hook(lambda m, i, o: taps.__setitem__("vit", o.detach())),
        model.ln_vision.register_forward_hook(lambda m, i, o: taps.__setitem__("image_embeds", o.detach())),
        model.Qformer.bert.register_forward_hook(lambda m, i, o: taps.__setitem__("qformer", o.last_hidden_state.detach())),
        model.encode_task_layer.register_forward_hook(lambda m, i, o: taps.__setitem__("z", o.detach())),
    ]
    with torch.no_grad():
        ids, query_up = model.get_codebook_indices(x)
        embeds = model.get_codebook_entry(ids)
    for h in hooks:
        h.remove()
    z = taps["z"].reshape(-1, 32)
    cb = sd["quantize.embedding.weight"]
    d = (z ** 2).sum(1, keepdim=True) + (cb ** 2).sum(1) - 2 * z @ cb.t()
    top2 = torch.topk(d, 2, dim=1, largest=False).values
    out = {
        "config": {"vit_depth": vit_depth, "qformer_layers": qformer_layers, "detok_depth": detok_depth,
                   "batch": batch, "weights_seed": 1234, "images_seed": 1234, "dtype": "fp32 (reference CPU mode)",
                   "reference": "models/seed_qformer/qformer_quantizer.py get_codebook_indices/get_codebook_entry"},
        "ids": ids.clone(), "z": z.clone(), "margin": (top2[:, 1] - top2[:, 0]).clone(),
        "query_output_up": _sample(query_up), "image_embeds_out": embeds.clone(),
        "vit": _sample(taps["vit"]), "image_embeds": _sample(taps["image_embeds"]),
        "qformer": taps["qformer"].clone() if taps["qformer"].numel() <= 100000 else _sample(taps["qformer"], 65536),
    }
    os.makedirs(GOLDEN_DIR, exist_ok=True)
    torch.save(out, os.path.join(GOLDEN_DIR, name))
    print(f"{name}: ids[0,:8]={ids[0, :8].tolist()} z_std={z.std():.3f} min_margin={out['margin'].min():.2e} "
          f"({time.time() - t0:.0f}s)")


def encoder_fresh_seed_golden(name: str = "encoder_v1_q2_d1_seed77.pt") -> None:
    """get_codebook_indices / get_codebook_entry outputs on weights and images of other seeds than the files above,
    with a de-tokenizer block: 1 ViT block, 2 Q-Former layers, 1 de-tokenizer block, 2 images."""
    vd, ql, dd, batch, wseed, iseed = 1, 2, 1, 2, 77, 78
    model = ref_shim.build_reference_quantizer(vd, ql, dd)
    model.load_state_dict(synth.encoder_state_dict(vd, ql, dd, seed=wseed), strict=False)
    x = synth.images(batch, seed=iseed)
    with torch.no_grad():
        ids, query_up = model.get_codebook_indices(x)
        embeds = model.get_codebook_entry(ids)
    out = {
        "config": {"vit_depth": vd, "qformer_layers": ql, "detok_depth": dd, "batch": batch, "weights_seed": wseed,
                   "images_seed": iseed, "dtype": "fp32 (reference CPU mode)",
                   "reference": "models/seed_qformer/qformer_quantizer.py get_codebook_indices/get_codebook_entry"},
        "ids": ids.clone(), "query_output_up": query_up.clone(), "image_embeds_out": embeds.clone(),
    }
    torch.save(out, os.path.join(GOLDEN_DIR, name))
    print(f"{name}: ids[0,:8]={ids[0, :8].tolist()} query_output_up {tuple(query_up.shape)}")


def llama_golden(name: str = "llama_tiny.pt") -> None:
    L = ref_shim.load_llama_module()
    from transformers.models.llama.configuration_llama import LlamaConfig

    hidden, layers, heads, ffn, vocab = 512, 2, 4, 1408, 1056
    cfg = LlamaConfig(vocab_size=vocab, hidden_size=hidden, intermediate_size=ffn, num_hidden_layers=layers,
                      num_attention_heads=heads, num_key_value_heads=heads, rms_norm_eps=1e-6,
                      max_position_embeddings=2048, hidden_act="silu", pad_token_id=0)
    cfg.use_cache = True
    model = L.LlamaForCausalLM(cfg).eval()
    sd = synth.llama_state_dict(hidden, layers, ffn, vocab)
    missing, unexpected = model.load_state_dict(sd, strict=False)
    assert not unexpected and all("rotary_emb" in k for k in missing), (missing, unexpected)
    ids = synth.prompt_ids(2, 48, n_image_spans=1, text_vocab=vocab - 66, n_codes=64)
    with torch.no_grad():
        out = model(input_ids=ids, use_cache=True, return_dict=True)
        nxt = out.logits[:, -1].argmax(-1, keepdim=True)
        out2 = model(input_ids=nxt, past_key_values=out.past_key_values, use_cache=True, return_dict=True)
    res = {
        "config": {"hidden": hidden, "layers": layers, "heads": heads, "ffn": ffn, "vocab": vocab, "seed": 1234,
                   "reference": "models/llama_xformer.py LlamaForCausalLM.forward (xformers stubbed by SDPA)"},
        "input_ids": ids, "logits": out.logits.clone(), "next_ids": nxt, "decode_logits": out2.logits.clone(),
        "k0": out.past_key_values[0][0].clone(), "v1": out.past_key_values[1][1].clone(),
    }
    torch.save(res, os.path.join(GOLDEN_DIR, name))
    print(f"{name}: logits {tuple(out.logits.shape)} next {nxt.flatten().tolist()}")


VQ_CASES = {"spread": (512, 0.28, 99), "default_init": (128, None, 98)}       # rows of z, codebook std, seed


def vq_inputs(tag: str) -> tuple[torch.Tensor, torch.Tensor]:
    """z [n,32] and the 8192 x 32 codebook (both fp16) of VQ case `tag`.  The codebooks are drawn here rather than
    stored (512 KB each); vq_golden keeps a strided sample of each so that a changed draw is caught."""
    n, cstd, seed = VQ_CASES[tag]
    g = torch.Generator().manual_seed(seed)
    z = (torch.randn(n, 32, generator=g) * 0.28).half()
    if cstd is None:    # the reference's default init, U(-1/n_e, 1/n_e) (qformer_quantizer.py:39)
        cb = (torch.rand(8192, 32, generator=g, dtype=torch.float64) * 2 - 1) / 8192
    else:
        cb = torch.randn(8192, 32, generator=g) * cstd
    return z, cb.half()


def vq_golden(name: str = "vq_reference_expr.pt") -> None:
    """The reference distance/argmin expression itself (qformer_quantizer.py:94-98) in fp32 and in half."""
    qq = ref_shim.load_quantizer_module()
    res = {}
    for tag in VQ_CASES:
        z, cb = vq_inputs(tag)
        n, n_codes = z.shape[0], cb.shape[0]
        vq = qq.VectorQuantizer2(n_codes, 32, beta=0.25)
        vq.embedding.weight.data = cb.float()
        with torch.no_grad():
            _, _, ids32 = vq(z.float().view(n // 32, 32, 32))
            vq16 = vq.half()
            _, _, ids16 = vq16(z.view(n // 32, 32, 32))
        res[tag] = {"z": z, "codebook_sample": _sample(cb), "ids_fp32": ids32.flatten().clone(),
                    "ids_fp16": ids16.flatten().clone()}
        print(f"{name}/{tag}: fp32 vs fp16 agreement {(ids32 == ids16).float().mean():.4f}")
    torch.save(res, os.path.join(GOLDEN_DIR, name))


def main() -> None:
    assert ref_shim.available(), "the reference must be mounted at /root/reference"
    torch.manual_seed(0)
    vq_golden()
    llama_golden()
    encoder_golden("encoder_d2_q2.pt", 2, 2, 1, 2)
    encoder_fresh_seed_golden()
    if "--full" in sys.argv:
        encoder_golden("encoder_full.pt", 39, 12, 4, 2)


if __name__ == "__main__":
    main()
