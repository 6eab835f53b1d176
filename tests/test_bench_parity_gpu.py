"""Parity at the bench configuration (BASELINE.json config #2: B = 256, full depth) beyond the two golden images:

* a 16-image sample of the bench batch through the CPU oracle (oracle/restatement.py, fp32 = the reference's CPU mode):
  ids exact above the margin, z within tolerance;
* the reference's *GPU* mode (`fp16: True`: `model.half()`, ViT + ln_vision under CUDA autocast, the rest in plain fp16 --
  models/seed_llama_tokenizer.py:58-59,86-87, qformer_quantizer.py:288-307) restated with torch on the GPU box as a
  second oracle (SURVEY.md section 8c): how far that mode sits from fp32, how far this build sits from fp32, and the
  id agreement between all three.  The numbers are printed as one JSON line.
"""
import json

import pytest
import torch
import torch.nn.functional as F

from oracle import restatement as R, synth

pytestmark = pytest.mark.gpu
ID_MARGIN_EPS = 0.02
VIT_DEPTH, QF_LAYERS = 39, 12
PICK = list(range(5, 256, 16))          # 16 of the 256 bench images


def rel(a, b):
    a, b = a.float().cpu(), b.float().cpu()
    return ((a - b).norm() / b.norm()).item()


@pytest.fixture(scope="module")
def full():
    from models.seed_qformer.qformer_quantizer import Blip2QformerQuantizer

    sd = synth.encoder_state_dict(VIT_DEPTH, QF_LAYERS, 0)
    x = synth.images(256, seed=1000).half()                      # bench.py's rank-0 batch
    out = {}
    for vq_mode in (1, 0):                                        # 1: fp32 VQ arithmetic (CPU mode), 0: fp16 (GPU mode)
        model = Blip2QformerQuantizer(sd, device="cuda", max_batch=256, gemm_ctas=2, vq_mode=vq_mode)
        ids, z = model.encode_ids(x.cuda(), return_z=True)
        torch.cuda.synchronize()
        out[vq_mode] = (ids.cpu(), z.float().cpu().view(256, 32, 32))
        del model
        torch.cuda.empty_cache()
    with torch.no_grad():
        ref = R.encode(x[PICK].float(), sd, VIT_DEPTH, QF_LAYERS)
    return sd, x, out, ref


def test_bench_batch_sample_matches_the_cpu_oracle_at_full_depth(full):
    sd, x, out, ref = full
    ids, z = out[1]
    ids, z = ids[PICK].reshape(-1), z[PICK]
    ref_ids, margin = ref["ids"].reshape(-1), ref["margin"].reshape(-1)
    neq = ids != ref_ids
    bad = neq & (margin > ID_MARGIN_EPS)
    assert not bad.any(), f"{int(bad.sum())} ids differ above the margin: {margin[bad][:8].tolist()}"
    assert (z - ref["z"]).abs().max().item() <= 1e-2
    # the bench default (fp16 VQ arithmetic = the reference's GPU mode) may only differ on near ties
    ids16 = out[0][0][PICK].reshape(-1)
    assert ((ids16 != ref_ids) & (margin > ID_MARGIN_EPS)).sum().item() == 0
    print(f"bench-batch sample: {int(neq.sum())}/{ids.numel()} ids flipped (fp32 VQ), "
          f"{int((ids16 != ref_ids).sum())} (fp16 VQ), {int((margin <= ID_MARGIN_EPS).sum())} tokens under the margin")


def reference_gpu_mode_encode(x16, sd16):
    """get_codebook_indices as the reference runs it on a GPU: every parameter fp16, ViT + ln_vision under autocast."""
    with torch.no_grad():
        with torch.autocast("cuda", dtype=torch.float16):
            vit = R.vit_forward_features(x16, sd16, VIT_DEPTH)
            image_embeds = F.layer_norm(vit, (1408,), sd16["ln_vision.weight"], sd16["ln_vision.bias"], 1e-5)
        qout = R.qformer_forward(image_embeds.half(), sd16, QF_LAYERS)
        z = F.linear(torch.tanh(F.linear(qout, sd16["encode_task_layer.0.weight"], sd16["encode_task_layer.0.bias"])),
                     sd16["encode_task_layer.2.weight"], sd16["encode_task_layer.2.bias"])
        ids, _ = R.vq_forward(z, sd16["quantize.embedding.weight"])
    return {"ids": ids.view(x16.shape[0], -1), "z": z, "vit": vit, "image_embeds": image_embeds, "qformer": qout}


def test_reference_gpu_mode_as_a_second_oracle(full):
    sd, x, out, ref = full
    sd16 = {k: v.to(device="cuda", dtype=torch.float16) for k, v in sd.items() if v.is_floating_point()}
    ac = reference_gpu_mode_encode(x[PICK].cuda(), sd16)
    del sd16
    torch.cuda.empty_cache()
    ref_ids, margin = ref["ids"].reshape(-1), ref["margin"].reshape(-1)
    ac_ids = ac["ids"].cpu().reshape(-1)
    ours32, ours16 = out[1][0][PICK].reshape(-1), out[0][0][PICK].reshape(-1)
    z_ours = out[1][1][PICK]
    report = {
        "images": len(PICK), "tokens": int(ref_ids.numel()), "tokens_under_margin_0.02": int((margin <= ID_MARGIN_EPS).sum()),
        "ids_differing": {
            "reference_gpu_mode_vs_fp32_oracle": int((ac_ids != ref_ids).sum()),
            "reference_gpu_mode_vs_fp32_oracle_above_margin": int(((ac_ids != ref_ids) & (margin > ID_MARGIN_EPS)).sum()),
            "this_build_fp32_vq_vs_fp32_oracle": int((ours32 != ref_ids).sum()),
            "this_build_fp16_vq_vs_fp32_oracle": int((ours16 != ref_ids).sum()),
            "this_build_fp16_vq_vs_reference_gpu_mode": int((ours16 != ac_ids).sum()),
        },
        "z_max_abs_err": {"reference_gpu_mode_vs_fp32": (ac["z"].float().cpu() - ref["z"]).abs().max().item(),
                          "this_build_vs_fp32": (z_ours - ref["z"]).abs().max().item()},
        "rel_frobenius_vs_fp32": {k: rel(ac[k], ref[k]) for k in ("vit", "image_embeds", "qformer")},
        "note": "reference GPU mode = model.half(), ViT + ln_vision under torch.autocast(fp16), Q-Former / heads / VQ in "
                "plain fp16 (restated with torch on this GPU); fp32 oracle = oracle/restatement.py on the host",
    }
    print(json.dumps(report))
    # this build keeps scores / statistics / accumulators in fp32 where the reference's GPU mode rounds to fp16: it
    # must sit at least as close to the fp32 oracle as that mode does (with slack for rounding noise)
    assert report["z_max_abs_err"]["this_build_vs_fp32"] <= max(1e-2, 1.5 * report["z_max_abs_err"]["reference_gpu_mode_vs_fp32"])
    assert report["ids_differing"]["this_build_fp32_vq_vs_fp32_oracle"] <= report["ids_differing"]["reference_gpu_mode_vs_fp32_oracle"] + 2
