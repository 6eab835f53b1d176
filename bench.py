#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric on the B200 path.

    python bench.py --gpus 1 --steps 10 --warmup 3                      # images/s, ViT-g/14 + Q-Former + VQ, B=256
    python bench.py --workload llama_prefill --steps 10 --warmup 3      # tokens/s, LLaMA-7B prefill, S=2048
    python bench.py --impl reference ...                                 # the reference algorithm on the host CPU
    torchrun --nproc-per-node N ... bench.py --gpus N ...                # one rank per GPU, weak scaling
    python bench.py ... --dump-outputs DIR                               # + the last timed step's outputs as .npy

One "step" is one pass of the hot path over one batch of synthetic input:
  encode        : 256 images/GPU -> [256,32] ids (config #2 of BASELINE.json); at N > 1 every rank encodes its own
                  shard and one NCCL all-gather returns all ids to every rank (config #4's data-parallel pattern);
  llama_prefill : one S=2048 prompt (with a 34-token image span) through random-init LLaMA-7B (config #3).
With the default workload the line also carries `secondary` records for the LLaMA half of BASELINE.json's metric
(llama_prefill, llama_decode) and for the chained config #4 (pipeline), measured at the same N by the same rules.
`value` is timed with CUDA events with the inputs already resident in HBM; `e2e` is the same metric through the
reference-facing Python API (models.seed_llama_tokenizer.ImageTokenizer.encode / models.llama_xformer
.LlamaForCausalLM.forward) starting from PINNED HOST buffers and ending with the ids / last-token logits on
the host, copies inside the timed region.  Prints ONE JSON line on rank 0.

--dump-outputs DIR writes, on rank 0, what each arm's timed path returned in its last timed step as DIR/<name>.npy
(integer outputs such as ids as float64, which holds them exactly, the rest as float32; at most 64 MB in all).  Inputs
and weights are seeded, so two builds run with the same arguments can be compared output for output.  Outputs too
large to keep whole are a fixed seeded sample: 64 positions of the prefill logits, 16 images of the preprocess batch.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)
sys.dont_write_bytecode = True      # the benchmark writes nothing into the tree it runs from (no __pycache__)

VIT_DEPTH, QF_LAYERS = 39, 12
# algorithmic work per image (2 FLOP per MAC), SURVEY.md section 8d / DESIGN.md
T_TOK, D, FF = 257, 1408, 6144
GEMM_FLOPS_PER_IMAGE = (
    2 * 256 * 588 * D                                                   # patch embed
    + VIT_DEPTH * 2 * T_TOK * (D * 3 * D + D * D + 2 * D * FF)         # qkv, proj, fc1, fc2
    + 6 * 2 * T_TOK * D * 1536                                          # cross-attention K|V of 6 layers
    + QF_LAYERS * 2 * 32 * (768 * 2304 + 768 * 768 + 2 * 768 * 3072)   # self qkv, out, FFN
    + 6 * 2 * 32 * (2 * 768 * 768)                                      # cross q, out
    + 2 * 32 * (768 * 768 + 768 * 32)                                   # encode_task_layer
)
ATTN_FLOPS_PER_IMAGE = (VIT_DEPTH * 4 * 16 * T_TOK * T_TOK * 88 + QF_LAYERS * 4 * 12 * 32 * 32 * 64
                        + 6 * 4 * 12 * 32 * T_TOK * 64)
ENCODE_FLOPS_PER_IMAGE = GEMM_FLOPS_PER_IMAGE + ATTN_FLOPS_PER_IMAGE + 2 * 32 * 8192 * 32


def measured_peaks():
    p = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"tflops_burst": d.get("bf16_tflops"), "tflops_sustained": d.get("bf16_tflops_sustained"),
                "hbm_gbs": d.get("hbm_gbs"), "source": "MEASURED_PEAKS.json (of measured)"}
    return {"tflops_burst": 1590.0, "tflops_sustained": 1400.0, "hbm_gbs": 6650.0,
            "source": "B200_PROFILING.md fallback (of fallback)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=lambda: [self.lines.append(l) for l in self.proc.stdout], daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def __exit__(self, *a):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], [], set()
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


def dist_setup(n_gpus: int):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist

        # stdout carries exactly one JSON line: NCCL's version banner (NCCL_DEBUG=VERSION, which some images export)
        # goes to stdout too
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return world, rank, local


def barrier_sync(world):
    if world > 1:
        import torch.distributed as dist

        dist.barrier()
    torch.cuda.synchronize()


def max_over_ranks(ms: float, world: int) -> float:
    if world == 1:
        return ms
    import torch.distributed as dist

    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


LAST_LOCAL_MS = [0.0]


def timed(fn, steps, warmup, world):
    """W untimed + K timed calls bracketed by barrier + synchronize; CUDA events; max over ranks (ms).
    The rank-local duration of the last call is left in LAST_LOCAL_MS[0] (per-rank statistics at N > 1)."""
    for _ in range(warmup):
        fn()
    barrier_sync(world)
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(steps):
        fn()
    e.record()
    barrier_sync(world)
    LAST_LOCAL_MS[0] = s.elapsed_time(e)
    return max_over_ranks(LAST_LOCAL_MS[0], world)


OUTPUTS = {}                    # --dump-outputs: name -> host array of the last timed step
DUMP_LIMIT_BYTES = 64 << 20


def keep_outputs(**tensors):
    """host copies of the last timed step's outputs, taken right after the timed region (the e2e and profiling calls
    that follow may reuse the buffers the outputs live in)"""
    for name, t in tensors.items():
        t = t.detach().cpu()
        OUTPUTS[name] = (t.float() if t.is_floating_point() else t.double()).numpy()


def seeded_rows(n: int, k: int) -> torch.Tensor:
    """a fixed sample of min(k, n) of n row indices, sorted: the same rows on every run of every build"""
    return torch.randperm(n, generator=torch.Generator().manual_seed(0))[:k].sort().values


def write_outputs(directory: str) -> None:
    import numpy as np

    total = sum(a.nbytes for a in OUTPUTS.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"bench.py: outputs of {total / 2**20:.1f} MB exceed the {DUMP_LIMIT_BYTES >> 20} MB of "
                         "--dump-outputs; use a smaller --batch")
    os.makedirs(directory, exist_ok=True)
    for name, a in OUTPUTS.items():
        np.save(os.path.join(directory, name + ".npy"), a)


def workload_config(args, world):
    """`config` of the JSON line -- built by ONE function for both arms (--impl seedb200 / reference), so the two
    lines name the same workload key for key; arm-specific facts (CPU sample size, kernel options) live outside it."""
    B = args.batch
    if args.workload == "encode":
        return {"workload": f"encode_b{B}_per_gpu", "global_batch": B * world, "vq_arithmetic": args.vq,
                "detail": "224x224 -> ViT-g/14 (39 blocks) + causal Q-Former (12 layers) + 8192-way VQ -> 32 ids/image",
                "weights": "seeded synthetic (seed_b200/synth.py; codebook N(0,0.28) instead of U(+-1/8192))",
                "parallelism": f"dp{world}" + (" + NCCL all-gather of ids" if world > 1 else ""),
                "l2": "inputs not flushed explicitly: each step streams ~2 GB of activations, 16x the 126 MB L2"}
    if args.workload == "llama_prefill":
        return {"workload": f"llama7b_prefill_s{args.seq}", "global_batch": world, "seq_len": args.seq,
                "detail": "random-init h4096/L32/H32/FFN11008/V40194, B=1, one 34-token image span, logits for all positions",
                "parallelism": f"dp{world} (independent replicas, no collective)",
                "l2": "13.5 GB of weights stream through L2 every step"}
    if args.workload == "llama_decode":
        return {"workload": f"llama13b_p{args.prompt}_decode{args.new_tokens}", "global_batch": world,
                "seq_len": args.prompt + args.new_tokens,
                "detail": f"random-init h5120/L40/H40/FFN13824/V40194, B=1, {args.prompt}-token prompt with 4 image spans, "
                          f"{args.new_tokens} greedy tokens (1 prefill + {args.new_tokens - 1} cached decode steps)",
                "parallelism": f"dp{world} (independent replicas, no collective)",
                "l2": "26 GB of weights stream from HBM every token (207x the L2)"}
    if args.workload == "pipeline":
        return {"workload": f"pipeline_encode_b{B}_to_llama7b_prefill_s{args.seq}", "global_batch": B * world,
                "seq_len": args.seq,
                "detail": "config #4: encode B images/GPU -> all-gather ids -> id->token arithmetic -> 60 image spans + text "
                          "-> one 7B prefill per rank, ids never leave the device",
                "parallelism": f"dp{world} + NCCL all-gather of ids", "l2": "activations >> L2"}
    return {"workload": f"preprocess_b{B}", "global_batch": B * world, "parallelism": f"dp{world}",
            "detail": "uint8 480x640x3 -> Pillow-exact bicubic 224x224 -> CLIP normalise -> fp16",
            "l2": f"inputs {B * 480 * 640 * 3 / 1e6:.0f} MB per step (> L2 at B=256)"}


def per_rank_stats(ms: float, world: int):
    """min / median / max over ranks of one rank-local duration (ms): shows whether an N>1 efficiency loss is skew
    between ranks (power capping) or a uniformly slower step (the collective)."""
    if world == 1:
        return None
    import torch.distributed as dist

    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    allv = [torch.zeros_like(t) for _ in range(world)]
    dist.all_gather(allv, t)
    v = sorted(float(x.item()) for x in allv)
    return {"min": round(v[0], 3), "median": round(v[len(v) // 2], 3), "max": round(v[-1], 3)}


# --------------------------------------------------------------------------------------------------
# CPU legs: the oracle port of the reference algorithm (the only place bench.py executes oracle/)
# --------------------------------------------------------------------------------------------------
def host_cores() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def tune_cpu_threads(sd) -> int:
    """The oracle port is plain torch on the host; on many-core boxes torch with every hardware thread is far from
    its best (measured: 8 threads of an 8-core container 1.08 images/s, 128 threads of the GPU box 0.02-0.47).  Give
    the CPU baseline its best thread count: time a 4-block slice at a few counts and keep the fastest."""
    from oracle import restatement as R
    from seed_b200 import synth

    n = host_cores()
    cands = sorted({c for c in (n, n // 2, n // 4, 32, 16, 8) if 1 <= c <= n}, reverse=True)
    x = synth.images(2, seed=3)
    best, best_t = n, float("inf")
    with torch.no_grad():
        for c in cands:
            torch.set_num_threads(c)
            R.encode(x, sd, 2, 2)
            t0 = time.perf_counter()
            R.encode(x, sd, 4, 2)
            t = time.perf_counter() - t0
            if t < best_t:
                best, best_t = c, t
    torch.set_num_threads(best)
    return best


def tune_cpu_threads_gemm() -> int:
    """same idea for the LLaMA port (GEMM dominated): fastest thread count on a 2048 x 4096 x 4096 fp32 matmul"""
    n = host_cores()
    cands = sorted({c for c in (n, n // 2, n // 4, 32, 16, 8) if 1 <= c <= n}, reverse=True)
    a, b = torch.randn(2048, 4096), torch.randn(4096, 4096)
    best, best_t = n, float("inf")
    for c in cands:
        torch.set_num_threads(c)
        torch.mm(a, b)
        t0 = time.perf_counter()
        torch.mm(a, b); torch.mm(a, b)
        t = time.perf_counter() - t0
        if t < best_t:
            best, best_t = c, t
    torch.set_num_threads(best)
    return best


ENC_GFLOP_FIXED = 0.424 + 12.75 + 0.056          # patch embed + Q-Former + heads/VQ (SURVEY 8d), per image
ENC_GFLOP_PER_BLOCK = 13.342


def cpu_encode_images_per_s(sd, n_images: int, target_s: float = 20.0):
    """Times oracle/restatement.py on a bounded sample of the workload.  `n_images` > 0 forces the sample size;
    0 sizes it from the (timed) warm-up image so that the leg costs ~target_s even on a slow or contended host:
    batches of 4 images (1 if an image takes > 6 s) until target_s has elapsed, at most 32 images."""
    from oracle import restatement as R
    from seed_b200 import synth

    tune_cpu_threads(sd)
    with torch.no_grad():
        x1 = synth.images(1, seed=4241)
        t0 = time.perf_counter()
        R.encode(x1, sd, VIT_DEPTH, QF_LAYERS)          # warm-up, also the probe
        probe = time.perf_counter() - t0
        if n_images > 0:
            x = synth.images(n_images, seed=4242)
            t0 = time.perf_counter()
            R.encode(x, sd, VIT_DEPTH, QF_LAYERS)
            dt = time.perf_counter() - t0
            return n_images / dt, dt, n_images
        bs = 4 if probe < 6.0 else 1
        done, t0 = 0, time.perf_counter()
        while done < 32:
            R.encode(synth.images(bs, seed=4242 + done), sd, VIT_DEPTH, QF_LAYERS)
            done += bs
            if time.perf_counter() - t0 >= target_s:
                break
        dt = time.perf_counter() - t0
    return done / dt, dt, done


def reference_arm(args, world, rank):
    """--impl reference: the reference algorithm (oracle port: /root/reference is Python and does not travel to
    the GPU box; oracle/restatement.py is pinned to it by tests/golden) on the host cores, same metric/config."""
    if rank != 0:
        return None
    from seed_b200 import synth

    cores = host_cores()
    torch.set_num_threads(cores)
    if args.workload == "encode":
        from oracle import restatement as R

        sd = synth.encoder_state_dict(VIT_DEPTH, QF_LAYERS, 0)
        cores = tune_cpu_threads(sd)
        x = synth.images(1, seed=1)
        with torch.no_grad():
            t0 = time.perf_counter(); R.encode(x, sd, VIT_DEPTH, QF_LAYERS); probe = time.perf_counter() - t0
        n_calls = max(1, args.steps + args.warmup)
        budget = args.ref_seconds / n_calls           # seconds per step so that the whole run ends within minutes
        depth, nb = VIT_DEPTH, max(1, min(args.batch, int(budget / max(probe, 1e-3))))
        if probe > budget:
            # even one full-depth image does not fit the per-step budget on this host: time a depth-truncated
            # ViT (same blocks, fewer of them) and scale by the algorithmic FLOPs of the missing blocks
            per_block = probe * ENC_GFLOP_PER_BLOCK / (ENC_GFLOP_FIXED + VIT_DEPTH * ENC_GFLOP_PER_BLOCK)
            depth = max(2, min(VIT_DEPTH, int((budget - probe * ENC_GFLOP_FIXED / (ENC_GFLOP_FIXED + VIT_DEPTH * ENC_GFLOP_PER_BLOCK)) / max(per_block, 1e-6))))
        scale_full = (ENC_GFLOP_FIXED + VIT_DEPTH * ENC_GFLOP_PER_BLOCK) / (ENC_GFLOP_FIXED + depth * ENC_GFLOP_PER_BLOCK)
        x = synth.images(nb, seed=1234)
        with torch.no_grad():
            for _ in range(args.warmup):
                R.encode(x, sd, depth, QF_LAYERS)
            t0 = time.perf_counter()
            for _ in range(args.steps):
                R.encode(x, sd, depth, QF_LAYERS)
            dt = (time.perf_counter() - t0) * scale_full
        value = nb * args.steps / dt
        sample = f"{nb} images/step (of the {args.batch}-image batch), fp32, torch {torch.get_num_threads()} threads"
        if depth != VIT_DEPTH:
            sample += f"; ViT truncated to {depth} of {VIT_DEPTH} blocks and the time scaled x{scale_full:.2f} by algorithmic FLOPs (host too slow for a full-depth image per step)"
        return dict(metric="images/sec SEED encode+VQ", value=value, unit="images/s", ms_per_step=1e3 * dt / args.steps,
                    sample=sample, cores=cores)
    else:
        from oracle import restatement as R

        cores = tune_cpu_threads_gemm()
        layers = 2       # layer-truncated 7B (fp32 7B = 26.6 GB of weights and minutes per prompt on the host)
        sd = synth.llama_state_dict(4096, layers, 11008, 40194)
        ids = synth.prompt_ids(1, args.seq, 1)
        with torch.no_grad():
            for _ in range(max(1, min(args.warmup, 1))):
                R.llama_forward(sd, ids, 32, layers)
            t0 = time.perf_counter()
            n = max(1, min(args.steps, 3))
            for _ in range(n):
                R.llama_forward(sd, ids, 32, layers)
            dt = (time.perf_counter() - t0) / n
        # scale the per-layer time to 32 layers (+ embedding / lm_head measured as part of the 2-layer run)
        per_layer = dt / (layers + 0.8)
        full = per_layer * (32 + 0.8)
        value = args.seq / full
        sample = (f"{layers}-layer slice of LLaMA-7B, S={args.seq}, fp32, scaled to 32 layers by measured time per layer "
                  f"(lm_head+embedding counted as 0.8 layer)")
        return dict(metric="tokens/sec LLaMA-7B prefill", value=value, unit="tokens/s", ms_per_step=1e3 * full,
                    sample=sample, cores=cores)


# --------------------------------------------------------------------------------------------------
# GPU arms
# --------------------------------------------------------------------------------------------------
def encode_arm(args, world, rank, local, keep=None):
    from models.seed_llama_tokenizer import ImageTokenizer, all_gather_ids
    from seed_b200 import lib as L, synth

    B = args.batch
    dev = torch.device("cuda", local)
    sd = synth.encoder_state_dict(VIT_DEPTH, QF_LAYERS, 0)
    tok = ImageTokenizer(model_path=sd, device=dev, fp16=True, max_batch=B, gemm_ctas=args.ctas,
                         vq_mode=L.VQ_FP32 if args.vq == "fp32" else L.VQ_FP16)
    if keep is not None:
        keep["tok"], keep["sd"] = tok, sd
    # id parity against the reference's own output (tests/golden/encoder_full.pt), same weights
    parity = None
    gpath = os.path.join(REPO, "tests", "golden", "encoder_full.pt")
    if rank == 0 and os.path.exists(gpath):
        g = torch.load(gpath, map_location="cpu", weights_only=False)
        ids = tok.encode(synth.images(g["config"]["batch"]).to(dev)).cpu()
        neq = ids != g["ids"]
        parity = {"tokens": int(ids.numel()), "equal": int((~neq).sum()),
                  "differ_above_margin_0.02": int((neq.reshape(-1) & (g["margin"] > 0.02)).sum()),
                  "vq_mode": args.vq, "against": "reference fp32 ids (tests/golden/encoder_full.pt)"}
    host = synth.images(B, seed=1000 + rank).half().pin_memory()
    x = host.to(dev)
    out = {}

    def step_device():
        ids = tok.encode(x)
        if world > 1:
            ids = all_gather_ids(ids)
        out["ids"] = ids

    def step_e2e():
        xi = host.to(dev, non_blocking=True)
        ids = tok.encode(xi)
        if world > 1:
            ids = all_gather_ids(ids)
        out["ids_host"] = ids.cpu()

    step_device(); torch.cuda.synchronize()
    L.reset_launch_count()
    with ClockSampler(local) as cs:
        ms = timed(step_device, args.steps, args.warmup, world)
    if args.dump_outputs:
        keep_outputs(encode_ids=out["ids"])
    rank_ms = per_rank_stats(LAST_LOCAL_MS[0] / args.steps, world)
    launches = L.launch_count() // (args.steps + args.warmup)
    clocks = cs.summary()
    ms_e2e = timed(step_e2e, args.steps, max(1, args.warmup), world)
    # roofline of the dominant kernel (tcgen05 GEMM): one more identical step with every GEMM launch bracketed
    # by CUDA events on its stream
    torch.cuda.synchronize()
    L.profile_begin()
    tok.encode(x)
    prof = L.profile_end()
    peaks = measured_peaks()
    gemm_ms, gemm_n = prof["gemm"]["ms"], prof["gemm"]["launches"]
    gemm_flops = GEMM_FLOPS_PER_IMAGE * B
    ach = gemm_flops / (gemm_ms * 1e-3) / 1e12
    traffic, traffic_src = None, None
    for name in ("r02_gemm_traffic.json", "r01_gemm_traffic.json"):
        tp = os.path.join(REPO, "profiles", name)
        if os.path.exists(tp):
            traffic = json.load(open(tp)).get("dram_bytes_per_launch_avg")
            traffic_src = f"static: ncu --set full capture committed as profiles/{name} (dram__bytes_read.sum + dram__bytes_write.sum per launch, average over the ViT shapes); not measured in this run"
            break
    roofline = {"kernel": "sb::gemm_tcgen05_kernel", "bound": "tensor", "achieved": round(ach, 1),
                "peak": peaks["tflops_sustained"], "unit": "TFLOP/s", "frac": round(ach / peaks["tflops_sustained"], 4),
                "traffic": traffic, "traffic_source": traffic_src,
                "peak_source": peaks["source"] + ", sustained figure (kernel timed inside a long step)",
                "launches_per_step": gemm_n, "gemm_ms_per_step": round(gemm_ms, 3),
                "algorithmic_gflop_per_launch": round(gemm_flops / gemm_n / 1e9, 2),
                "avg_launch_ms": round(gemm_ms / gemm_n, 4), "share_of_step": round(gemm_ms / (ms / args.steps), 3),
                "attention_ms_per_step": round(prof["attention"]["ms"], 3),
                "whole_step_tflops": round(ENCODE_FLOPS_PER_IMAGE * B / (ms / args.steps * 1e-3) / 1e12, 1)}
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:      # reported at N=1 only
        v, dt, n_cpu = cpu_encode_images_per_s(sd, args.cpu_images)
        cpu = {"value": round(v, 3), "unit": "images/s", "cores": torch.get_num_threads(), "kind": "port",
               "sample": f"{n_cpu} of the {B} images, full depth, fp32, oracle/restatement.py, {dt:.1f} s, "
                         f"{torch.get_num_threads()} of {host_cores()} host threads (fastest of a short sweep)"}
    total = B * world * args.steps
    res = {
        "metric": "images/sec SEED encode+VQ", "value": round(total / (ms * 1e-3), 2), "unit": "images/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms / args.steps, 3),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
        "config": workload_config(args, world), "kernel_options": {"gemm_cta_group": args.ctas or 1},
        "clocks": clocks,
        "e2e": {"value": round(total / (ms_e2e * 1e-3), 2), "unit": "images/s",
                "h2d_bytes_per_step": B * world * 3 * 224 * 224 * 2, "d2h_bytes_per_step": B * world * 32 * 8 * world,
                "api": "models.seed_llama_tokenizer.ImageTokenizer.encode(pinned.to(cuda)) -> ids.cpu()"},
        "gpu_launches": int(launches) * args.steps,
        "roofline": roofline, "cpu_baseline": cpu, "id_parity": parity,
    }
    if rank_ms is not None:
        res["per_rank_ms_per_step"] = rank_ms
    return res


def random_llama(dev, rank, h, nl, nh, ffn, V, max_seq, ctas):
    """random-init llama_xformer weights generated on the device (HF key names), wrapped by the product class"""
    from transformers.models.llama.configuration_llama import LlamaConfig
    from models.llama_xformer import LlamaForCausalLM

    cfg = LlamaConfig(vocab_size=V, hidden_size=h, intermediate_size=ffn, num_hidden_layers=nl,
                      num_attention_heads=nh, num_key_value_heads=nh, rms_norm_eps=1e-6, max_position_embeddings=4096)
    g = torch.Generator(device=dev).manual_seed(1234 + rank)

    def rnd(*shape, std=0.02, mean=0.0):
        return (torch.randn(*shape, device=dev, generator=g, dtype=torch.float32) * std + mean).half()

    sd = {"model.embed_tokens.weight": rnd(V, h), "model.norm.weight": rnd(h, std=0.05, mean=1.0),
          "lm_head.weight": rnd(V, h)}
    for l in range(nl):
        p = f"model.layers.{l}."
        for n in ("q_proj", "k_proj", "v_proj", "o_proj"):
            sd[p + f"self_attn.{n}.weight"] = rnd(h, h)
        sd[p + "mlp.gate_proj.weight"] = rnd(ffn, h)
        sd[p + "mlp.up_proj.weight"] = rnd(ffn, h)
        sd[p + "mlp.down_proj.weight"] = rnd(h, ffn)
        sd[p + "input_layernorm.weight"] = rnd(h, std=0.05, mean=1.0)
        sd[p + "post_attention_layernorm.weight"] = rnd(h, std=0.05, mean=1.0)
    model = LlamaForCausalLM(cfg, sd, device=dev, max_batch=1, max_seq=max_seq, gemm_ctas=ctas)
    del sd
    torch.cuda.empty_cache()
    return model


def llama_decode_arm(args, world, rank, local):
    """BASELINE.json config #5: random-init 13B llama_xformer, interleaved 4-image prompt, prefill + 128 generated
    tokens (greedy), batch 1.  A step = one generate() call = ONE C call (prefill, on-device sampler, CUDA-graph
    replayed decode steps); value = generated tokens/s over prefill+decode."""
    from seed_b200 import lib as L, synth

    dev = torch.device("cuda", local)
    h, nl, nh, ffn, V = 5120, 40, 40, 13824, 40194
    P, NEW = args.prompt, args.new_tokens
    model = random_llama(dev, rank, h, nl, nh, ffn, V, P + NEW + 8, args.ctas)
    ids_host = synth.prompt_ids(1, P, 4, seed=99 + rank).pin_memory()
    ids = ids_host.to(dev)
    out = {}
    gen = dict(max_new_tokens=NEW, do_sample=False, eos_token_id=-1)       # fixed length: no early stop on eos

    def step_device():
        out["seq"] = model.generate(input_ids=ids, **gen)

    def step_e2e():
        out["host"] = model.generate(input_ids=ids_host.to(dev, non_blocking=True), **gen).cpu()

    step_device(); torch.cuda.synchronize()
    used_graph = model._llm.used_graph
    L.reset_launch_count()
    with ClockSampler(local) as cs:
        ms = timed(step_device, args.steps, args.warmup, world)
    if args.dump_outputs:
        keep_outputs(llama_decode_sequence=out["seq"])
    rank_ms = per_rank_stats(LAST_LOCAL_MS[0] / args.steps, world)
    launches = L.launch_count() // (args.steps + args.warmup)
    clocks = cs.summary()
    ms_e2e = timed(step_e2e, args.steps, max(1, args.warmup), world)
    # decode-only time per token: whole generate minus the prefill forward, both between CUDA events
    e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
    torch.cuda.synchronize()
    e0.record()
    model.forward(input_ids=ids, use_cache=True, last_logits_only=True)
    e1.record()
    model.generate(input_ids=ids, **gen)
    e2.record(); torch.cuda.synchronize()
    prefill_ms = e0.elapsed_time(e1)
    dec_ms = (e1.elapsed_time(e2) - prefill_ms) / (NEW - 1)
    peaks = measured_peaks()
    weight_bytes = 2.0 * (nl * (4 * h * h + 3 * h * ffn) + h * V)      # every weight once per token (+ one embedding row)
    kv_bytes = 2.0 * 2 * nl * nh * 128 * (P + NEW / 2)
    ach = (weight_bytes + kv_bytes) / (dec_ms * 1e-3) / 1e9
    total_tok = NEW * world * args.steps
    res = {
        "metric": "tokens/sec LLaMA-13B prefill+decode", "value": round(total_tok / (ms * 1e-3), 1), "unit": "tokens/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms / args.steps, 3),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
        "config": workload_config(args, world),
        "kernel_options": {"gemm_cta_group": args.ctas or 1, "decode_step": "CUDA graph replay" if used_graph == 1 else "eager launches"},
        "clocks": clocks,
        "e2e": {"value": round(total_tok / (ms_e2e * 1e-3), 1), "unit": "tokens/s", "h2d_bytes_per_step": P * 8,
                "d2h_bytes_per_step": (P + NEW) * 8,
                "api": "models.llama_xformer.LlamaForCausalLM.generate(pinned ids.to(cuda), max_new_tokens) -> seq.cpu()"},
        "gpu_launches": int(launches) * args.steps,
        "roofline": {"kernel": "sb::gemv_kernel (whole cached decode step incl. sampler)", "bound": "hbm", "achieved": round(ach, 1),
                     "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": round(ach / peaks["hbm_gbs"], 4), "traffic": None,
                     "peak_source": peaks["source"], "decode_ms_per_token": round(dec_ms, 4),
                     "prefill_ms": round(prefill_ms, 3),
                     "algorithmic_bytes_per_token": int(weight_bytes + kv_bytes)},
        "cpu_baseline": None,
    }
    if rank_ms is not None:
        res["per_rank_ms_per_step"] = rank_ms
    del model
    torch.cuda.empty_cache()
    return res


def preprocess_arm(args, world, rank, local):
    """SURVEY 8f row 1: uint8 HWC images (640x480, the COCO-style size) -> bicubic resize 224 -> normalise -> fp16 on
    the GPU (seedb200_preprocess_run), bit-exact with the reference's torchvision+Pillow `processor`."""
    import numpy as np
    from PIL import Image
    from torchvision import transforms

    from seed_b200 import lib as L

    dev = torch.device("cuda", local)
    B, H, W = args.batch, 480, 640
    rng = np.random.default_rng(5 + rank)
    host = torch.from_numpy(rng.integers(0, 256, (B, H, W, 3), dtype=np.uint8)).pin_memory()
    x = host.to(dev)
    plan = L.Preprocess(H, W, 224, "bicubic", max_batch=B)
    out = {}

    def step_device():
        out["y"] = plan(x)

    def step_e2e():
        out["y"] = plan(host.to(dev, non_blocking=True))
        out["sum"] = out["y"][:, :, ::56, ::56].float().sum().cpu()      # small device->host read of the result

    step_device(); torch.cuda.synchronize()
    L.reset_launch_count()
    with ClockSampler(local) as cs:
        ms = timed(step_device, args.steps, args.warmup, world)
    if args.dump_outputs:
        keep_outputs(preprocess_pixels_sample=out["y"][seeded_rows(B, 16).to(dev)])
    launches = L.launch_count() // (args.steps + args.warmup)
    clocks = cs.summary()
    ms_e2e = timed(step_e2e, args.steps, max(1, args.warmup), world)
    peaks = measured_peaks()
    alg_bytes = B * (H * W * 3 + 3 * 224 * 224 * 2)
    ach = alg_bytes / (ms / args.steps * 1e-3) / 1e9
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        ref = transforms.Compose([transforms.Resize((224, 224), interpolation=3), transforms.ToTensor(),
                                  transforms.Normalize((0.48145466, 0.4578275, 0.40821073), (0.26862954, 0.26130258, 0.27577711))])
        n_cpu = min(B, 64)
        pil = [Image.fromarray(host[i].numpy(), "RGB") for i in range(n_cpu)]
        t0 = time.perf_counter()
        res = [ref(p).half() for p in pil]
        dt = time.perf_counter() - t0
        same = bool(torch.equal(torch.stack(res).view(torch.int16), out["y"][:n_cpu].cpu().view(torch.int16)))
        cpu = {"value": round(n_cpu / dt, 1), "unit": "images/s", "cores": 1, "kind": "reference",
               "sample": f"{n_cpu} of the {B} images through torchvision+Pillow (the reference's own processor), one thread",
               "bit_exact_vs_gpu": same}
    total = B * world * args.steps
    return {
        "metric": "images/sec preprocess (resize+normalise)", "value": round(total / (ms * 1e-3), 1), "unit": "images/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms / args.steps, 4),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": workload_config(args, world),
        "clocks": clocks,
        "e2e": {"value": round(total / (ms_e2e * 1e-3), 1), "unit": "images/s", "h2d_bytes_per_step": B * world * H * W * 3,
                "d2h_bytes_per_step": 4 * world, "api": "seed_b200.lib.Preprocess(pinned uint8.to(cuda)) -> checksum.cpu()"},
        "gpu_launches": int(launches) * args.steps,
        "roofline": {"kernel": "sb::resize_h_kernel + sb::resize_v_norm_kernel", "bound": "hbm", "achieved": round(ach, 1),
                     "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": round(ach / peaks["hbm_gbs"], 4), "traffic": None,
                     "peak_source": peaks["source"], "algorithmic_bytes_per_step": alg_bytes},
        "cpu_baseline": cpu,
    }


def llama_arm(args, world, rank, local, keep=None):
    from seed_b200 import lib as L, synth

    dev = torch.device("cuda", local)
    h, nl, nh, ffn, V, S = 4096, 32, 32, 11008, 40194, args.seq
    model = random_llama(dev, rank, h, nl, nh, ffn, V, S, args.ctas)
    if keep is not None:
        keep["llama7b"] = model
    ids_host = synth.prompt_ids(1, S, 1, seed=77 + rank).pin_memory()
    ids = ids_host.to(dev)
    out = {}

    def step_device():
        out["o"] = model.forward(input_ids=ids, use_cache=False)          # full [1,S,V] logits: the reference contract

    def step_e2e():
        o = model.forward(input_ids=ids_host.to(dev, non_blocking=True), use_cache=False)
        out["last"] = o.logits[:, -1].float().cpu()

    step_device(); torch.cuda.synchronize()
    L.reset_launch_count()
    with ClockSampler(local) as cs:
        ms = timed(step_device, args.steps, args.warmup, world)
    if args.dump_outputs:
        keep_outputs(llama_prefill_logits_sample=out["o"].logits[0, seeded_rows(S, 64).to(dev)])
    rank_ms = per_rank_stats(LAST_LOCAL_MS[0] / args.steps, world)
    launches = L.launch_count() // (args.steps + args.warmup)
    clocks = cs.summary()
    ms_e2e = timed(step_e2e, args.steps, max(1, args.warmup), world)
    L.profile_begin(); model.forward(input_ids=ids, use_cache=False); prof = L.profile_end()
    peaks = measured_peaks()
    lin_flops = 2.0 * S * (nl * (4 * h * h + 3 * h * ffn) + h * V)
    attn_flops = nl * 4.0 * nh * S * S * 128 * 0.5
    ach = lin_flops / (prof["gemm"]["ms"] * 1e-3) / 1e12
    total_tok = S * world * args.steps
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        import copy

        a2 = copy.copy(args); a2.steps, a2.warmup, a2.workload = 1, 1, "llama_prefill"
        r = reference_arm(a2, 1, 0)
        cpu = {"value": round(r["value"], 2), "unit": r["unit"], "cores": r["cores"], "kind": "port", "sample": r["sample"]}
    res = {
        "metric": "tokens/sec LLaMA-7B prefill", "value": round(total_tok / (ms * 1e-3), 1), "unit": "tokens/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms / args.steps, 3),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
        "config": workload_config(args, world), "kernel_options": {"gemm_cta_group": args.ctas or 1},
        "clocks": clocks,
        "e2e": {"value": round(total_tok / (ms_e2e * 1e-3), 1), "unit": "tokens/s", "h2d_bytes_per_step": S * 8,
                "d2h_bytes_per_step": V * 4,
                "api": "models.llama_xformer.LlamaForCausalLM.forward(pinned ids.to(cuda)) -> logits[:, -1].cpu()"},
        "gpu_launches": int(launches) * args.steps,
        "roofline": {"kernel": "sb::gemm_tcgen05_kernel", "bound": "tensor", "achieved": round(ach, 1),
                     "peak": peaks["tflops_sustained"], "unit": "TFLOP/s",
                     "frac": round(ach / peaks["tflops_sustained"], 4), "traffic": None,
                     "peak_source": peaks["source"], "launches_per_step": prof["gemm"]["launches"],
                     "gemm_ms_per_step": round(prof["gemm"]["ms"], 3),
                     "attention_ms_per_step": round(prof["attention"]["ms"], 3),
                     "whole_step_tflops": round((lin_flops + attn_flops) / (ms / args.steps * 1e-3) / 1e12, 1)},
        "cpu_baseline": cpu,
    }
    if rank_ms is not None:
        res["per_rank_ms_per_step"] = rank_ms
    return res


def pipeline_arm(args, world, rank, local, tok=None, model=None):
    """BASELINE.json config #4 as one device-resident chain: every rank encodes its 256 images, ONE NCCL all-gather
    hands all ids to every rank, the id -> token arithmetic writes 60 `<img>`+32 ids+`</img>` spans (of the gathered
    images, rank r takes images [60 r, 60 r + 60)) between text tokens of an S=2048 prompt, and the rank's LLaMA-7B
    replica prefills it.  No id touches the host (scripts/seed_llama_inference_8B.py:94-103 does a string round trip)."""
    from models.seed_llama_tokenizer import ImageTokenizer, SeedImageTokenMixin, all_gather_ids
    from seed_b200 import lib as L, synth

    B, S = args.batch, args.seq
    dev = torch.device("cuda", local)
    if tok is None:
        tok = ImageTokenizer(model_path=synth.encoder_state_dict(VIT_DEPTH, QF_LAYERS, 0), device=dev, fp16=True,
                             max_batch=B, gemm_ctas=args.ctas)
    if model is None:
        model = random_llama(dev, rank, 4096, 32, 32, 11008, 40194, S, args.ctas)
    n_span = min(60, (S - 8) // 34, B * world)
    host = synth.images(B, seed=1000 + rank).half().pin_memory()
    text_host = torch.randint(0, 32000, (1, S), generator=torch.Generator().manual_seed(5 + rank)).pin_memory()
    x, text = host.to(dev), text_host.to(dev)
    out = {}

    def chain(images, prompt):
        ids = tok.encode(images)                                   # [B,32] int64 on the device
        if world > 1:
            ids = all_gather_ids(ids)                              # [world*B,32] on every rank
        first = (rank * n_span) % max(1, ids.shape[0] - n_span + 1)
        spans = prompt[0, 8:8 + n_span * 34].view(n_span, 34)
        SeedImageTokenMixin.image_ids_to_tokens(ids[first:first + n_span], 32000, out=spans)
        return model.forward(input_ids=prompt, use_cache=False, last_logits_only=True)

    def step_device():
        out["o"] = chain(x, text)

    def step_e2e():
        o = chain(host.to(dev, non_blocking=True), text_host.to(dev, non_blocking=True))
        out["last"] = o.logits[:, -1].float().cpu()

    step_device(); torch.cuda.synchronize()
    L.reset_launch_count()
    with ClockSampler(local) as cs:
        ms = timed(step_device, args.steps, args.warmup, world)
    if args.dump_outputs:
        keep_outputs(pipeline_last_logits=out["o"].logits)
    rank_ms = per_rank_stats(LAST_LOCAL_MS[0] / args.steps, world)
    launches = L.launch_count() // (args.steps + args.warmup)
    clocks = cs.summary()
    ms_e2e = timed(step_e2e, args.steps, max(1, args.warmup), world)
    step_s, e2e_s = ms / args.steps * 1e-3, ms_e2e / args.steps * 1e-3
    flops = ENCODE_FLOPS_PER_IMAGE * B + 2.0 * S * 32 * (4 * 4096 * 4096 + 3 * 4096 * 11008) + 2.0 * 4096 * 40194 \
        + 32 * 4.0 * 32 * S * S * 128 * 0.5
    peaks = measured_peaks()
    res = {
        "metric": "images/sec SEED encode+VQ feeding one LLaMA-7B prefill per rank", "value": round(B * world / step_s, 2),
        "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(ms / args.steps, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f16", "data": "synthetic", "config": workload_config(args, world),
        "prefill_tokens_per_s": round(S * world / step_s, 1), "image_spans_per_prompt": n_span,
        "clocks": clocks,
        "e2e": {"value": round(B * world / e2e_s, 2), "unit": "images/s",
                "h2d_bytes_per_step": world * (B * 3 * 224 * 224 * 2 + S * 8), "d2h_bytes_per_step": world * 40194 * 4,
                "api": "ImageTokenizer.encode(pinned.to(cuda)) -> all_gather_ids -> image_ids_to_tokens(out=prompt span) "
                       "-> LlamaForCausalLM.forward(last_logits_only) -> logits.cpu()"},
        "gpu_launches": int(launches) * args.steps,
        "roofline": {"kernel": "whole chain (tcgen05 GEMMs dominate)", "bound": "tensor",
                     "achieved": round(flops / step_s / 1e12, 1), "peak": peaks["tflops_sustained"], "unit": "TFLOP/s",
                     "frac": round(flops / step_s / 1e12 / peaks["tflops_sustained"], 4), "traffic": None,
                     "peak_source": peaks["source"]},
        "cpu_baseline": None,
    }
    if rank_ms is not None:
        res["per_rank_ms_per_step"] = rank_ms
    return res


def compact(r):
    """a secondary record: the same fields as a full line minus the boilerplate"""
    keep = ("metric", "value", "unit", "steps", "warmup", "ms_per_step", "config", "kernel_options", "clocks", "e2e",
            "gpu_launches", "roofline", "cpu_baseline", "per_rank_ms_per_step", "prefill_tokens_per_s",
            "image_spans_per_prompt")
    return {k: r[k] for k in keep if k in r and r[k] is not None}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="seedb200", choices=["seedb200", "reference"])
    ap.add_argument("--workload", default="encode",
                    choices=["encode", "llama_prefill", "llama_decode", "pipeline", "preprocess"])
    ap.add_argument("--batch", type=int, default=256, help="images per GPU per step (encode)")
    ap.add_argument("--seq", type=int, default=2048, help="prompt length (llama_prefill)")
    ap.add_argument("--prompt", type=int, default=256, help="prompt length (llama_decode)")
    ap.add_argument("--new-tokens", type=int, default=128, help="generated tokens (llama_decode)")
    ap.add_argument("--ctas", type=int, default=2, help="tcgen05 cta_group of the GEMMs (1 or 2)")
    ap.add_argument("--vq", default="fp16", choices=["fp16", "fp32"], help="VQ distance arithmetic")
    ap.add_argument("--cpu-images", type=int, default=0, help="images timed by the cpu_baseline leg (0 = ~20 s worth)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-secondary", action="store_true",
                    help="encode workload only: skip the LLaMA half of BASELINE.json's metric (secondary records)")
    ap.add_argument("--ref-seconds", type=float, default=150.0, help="wall-clock budget of the --impl reference run")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step of every arm as DIR/<name>.npy (seedb200 arm)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the seedb200 arm")
    args.warmup = max(args.warmup, 3) if args.impl == "seedb200" else args.warmup

    if args.impl == "reference":
        world = int(os.environ.get("WORLD_SIZE", "1"))
        rank = int(os.environ.get("RANK", "0"))
        r = reference_arm(args, world, rank)
        if r is None:
            return
        line = {"impl": "reference", "metric": r["metric"], "value": round(r["value"], 3), "unit": r["unit"],
                "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": round(r["ms_per_step"], 2), "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": workload_config(args, max(world, args.gpus)),
                "note": "reference algorithm on the host CPU (oracle port of /root/reference, pinned by tests/golden); "
                        "no GPU involved; every step is a BOUNDED SAMPLE of the workload: " + r["sample"],
                "cpu_baseline": {"value": round(r["value"], 3), "unit": r["unit"], "cores": r["cores"], "kind": "port",
                                 "sample": r["sample"]},
                "e2e": {"value": round(r["value"], 3), "unit": r["unit"], "h2d_bytes_per_step": 0,
                        "d2h_bytes_per_step": 0}}
        print(json.dumps(line), flush=True)
        return

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the seedb200 arm has no CPU fallback; use --impl reference)")
    world, rank, local = dist_setup(args.gpus)
    if args.workload == "encode":
        # headline: images/s through encode -> VQ.  BASELINE.json's metric has a second half (tokens/s through
        # llama_xformer: 7B prefill, config #3; 13B prefill + 128-step decode, config #5) and a chained config (#4):
        # they ride in the same line as `secondary` records, measured by the same rules at the same N.
        import copy

        keep = {}
        res = encode_arm(args, world, rank, local, keep=keep)
        if not args.no_secondary:
            sec = {}
            a2 = copy.copy(args)
            a2.workload, a2.steps = "llama_prefill", min(args.steps, 10)
            sec["llama_prefill"] = compact(llama_arm(a2, world, rank, local, keep=keep))
            a3 = copy.copy(args)
            a3.workload, a3.steps = "pipeline", min(args.steps, 5)
            sec["pipeline"] = compact(pipeline_arm(a3, world, rank, local, tok=keep["tok"], model=keep["llama7b"]))
            keep.clear()
            import gc

            gc.collect()
            torch.cuda.empty_cache()
            a4 = copy.copy(args)
            a4.workload, a4.steps = "llama_decode", min(args.steps, 3)
            sec["llama_decode"] = compact(llama_decode_arm(a4, world, rank, local))
            res["secondary"] = sec
    else:
        arm = {"llama_prefill": llama_arm, "llama_decode": llama_decode_arm, "pipeline": pipeline_arm,
               "preprocess": preprocess_arm}[args.workload]
        res = arm(args, world, rank, local)
    if world > 1:
        import torch.distributed as dist

        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        if args.dump_outputs:
            write_outputs(args.dump_outputs)
        print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
