#!/usr/bin/env python
"""Benchmark of the MetaMorph hot path (contract: task statement + BASELINE.json).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path (default N=1)
    python bench.py ... --dump-outputs DIR                    # + the last timed step's outputs as DIR/*.npy
    python bench.py --impl reference --gpus N ...             # the reference's own code on the host cores (oracle/_ref)
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (config.workload): BASELINE.json configs[1] at N=1 — LLaMA-3-8B + SigLIP-SO400M-14@384, bf16
instruction-tune step (forward + backward + AdamW), seq_len 4096, batch 4 per GPU, 4 images per sample
(2 prompt-side, 2 answer-side), synthetic seeded data, random-init weights. N>1: the same per-GPU batch
on every rank (weak scaling, configs[2] shape at N=8 with --batch 8), one gradient all-reduce per bucket.
Metric: interleaved tokens/sec of the whole job (sum over ranks of B*T per step / max-over-ranks time).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "interleaved tokens/sec (train step) LLaMA-3-8B+SigLIP seq4096"
UNIT = "tokens/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=4, help="samples per GPU")
    ap.add_argument("--seq-len", type=int, default=4096)
    ap.add_argument("--images-per-sample", type=int, default=4, help="half prompt-side, half answer-side")
    ap.add_argument("--layers", type=int, default=32, help="debug only: fewer layers => invalid as a result")
    ap.add_argument("--save-gu-layers", type=int, default=int(os.environ.get("MM_SAVE_GU_LAYERS", "32")))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-decode", action="store_true")
    ap.add_argument("--no-shard", action="store_true", help="A/B only: replicate the optimizer state (round-1 behaviour)")
    ap.add_argument("--no-fused-allgather", action="store_true", help="A/B only: NCCL all-gather instead of the AdamW kernel's own broadcast")
    ap.add_argument("--extra-configs", default="auto", choices=["auto", "on", "off"],
                    help="BASELINE configs 3 (batch 8/GPU) and 5 (T=8192, 8 frames) as extra keys; auto = at 8 GPUs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed to DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


# ------------------------------------------------------------------------------------------------
# algorithmic FLOPs (SURVEY.md §8d): 6*P per token + causal-halved attention + forward-only vision
# ------------------------------------------------------------------------------------------------
def train_flops_per_step(B, T, n_images, L=32, H=4096, I=14336, V=128258, Hq=32, Hkv=8, dh=128):
    per_layer = H * (Hq * dh + 2 * Hkv * dh + Hq * dh) + 3 * H * I
    P = L * per_layer + H * V
    per_token = 6 * P + 6 * L * H * T
    vision = 2 * 729 * (27 * (4 * 1152 ** 2 + 2 * 1152 * 4304) + 588 * 1152) + 27 * 4 * 729 ** 2 * 1152
    return B * T * per_token + n_images * vision


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""

    def __init__(self, gpu_index):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# CPU baseline = THE REFERENCE'S OWN CODE on the host cores (oracle/ref_bench.py runs the copy that oracle/build_ref.py
# vendors into oracle/_ref; it is a separate process so that `metamorph` resolves to the reference, not to this
# repository's alias package). Falls back to the oracle port (oracle/restatement.py) only if that copy is missing.
# ------------------------------------------------------------------------------------------------
def _run_ref_bench(argv, timeout):
    cmd = [sys.executable, os.path.join(ROOT, "oracle", "ref_bench.py")] + argv
    env = dict(os.environ)
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT"):
        env.pop(k, None)
    try:
        res = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, env=env)
    except subprocess.TimeoutExpired:
        return None, "oracle/ref_bench.py timed out"
    rows = []
    for line in res.stdout.splitlines():
        line = line.strip()
        if line.startswith("{"):
            try:
                rows.append(json.loads(line))
            except ValueError:
                pass
    summ = next((r for r in reversed(rows) if "summary" in r), None)
    if summ is None or "error" in summ:
        return None, (summ or {}).get("error") or (res.stderr.strip().splitlines() or ["no output"])[-1][:300]
    return summ, None


def _train_sample_desc(summ, secs):
    return (f"the reference's own MetaMorphLlamaForCausalLM.forward + loss.backward() ({summ['root']}; torch {summ['torch']} CPU, "
            f"{summ['dtype']}, {summ['attention']} attention): full width, depth-reduced to {summ['layers']} LLaMA layer(s) + lm_head over all "
            f"rows + both losses + {summ['siglip_layers']} SigLIP layers on {summ['images']} images, B=1, T={summ['seq_len']}; "
            f"{secs:.2f} s per sample on {summ['threads']} of {summ['host_threads']} host threads (fastest of a 1-second "
            f"thread-count calibration); tokens/s = (algorithmic FLOPs of the sample / seconds) / (algorithmic FLOPs per "
            f"token of the 32-layer + 27-layer step), i.e. a LABELLED EXTRAPOLATION by FLOP ratio")


def reference_train_tokens_per_s(summ, secs, T):
    return (summ["sample_flops"] / secs) / (train_flops_per_step(1, T, 4) / T)


def cpu_port_sample(T=1024, layers=1):
    """Fallback only (no oracle/_ref on this box): one full-width decoder layer of the oracle PORT, fwd+bwd, fp32."""
    import torch
    from oracle import restatement as R
    H, I, Hq, Hkv, dh = 4096, 14336, 32, 8, 128
    g = torch.Generator().manual_seed(0)
    p = {}
    for i in range(layers):
        q = f"model.layers.{i}."
        p[q + "input_layernorm.weight"] = torch.ones(H)
        p[q + "post_attention_layernorm.weight"] = torch.ones(H)
        for n, shp in (("self_attn.q_proj", (Hq * dh, H)), ("self_attn.k_proj", (Hkv * dh, H)),
                       ("self_attn.v_proj", (Hkv * dh, H)), ("self_attn.o_proj", (H, Hq * dh)),
                       ("mlp.gate_proj", (I, H)), ("mlp.up_proj", (I, H)), ("mlp.down_proj", (H, I))):
            p[q + n + ".weight"] = (torch.randn(shp, generator=g) * 0.02).requires_grad_(True)
    p["model.norm.weight"] = torch.ones(H)
    x = (torch.randn(1, T, H, generator=g) * 0.1).requires_grad_(True)
    t0 = time.time()
    out = R.llama_forward(p, x, torch.arange(T)[None], torch.ones(1, T, dtype=torch.bool), layers, Hq, Hkv,
                          1e-5, 500000.0)
    out.square().mean().backward()
    dt = time.time() - t0
    flops_sample = T * (6 * layers * (H * (2 * Hq * dh + 2 * Hkv * dh) + 3 * H * I) + 6 * layers * H * T)
    return dt, (flops_sample / dt) / (train_flops_per_step(1, T, 0) / T)


def cpu_train_baseline(T):
    """cpu_baseline of the default run: one bounded sample of the reference's own train step per dtype (fp32 and bf16)."""
    summ, err = _run_ref_bench(["train", "--steps", "1", "--warmup", "0", "--seq-len", str(T), "--dtype", "auto",
                                "--budget-s", "1e9"], timeout=900)
    if summ is None:
        dt, tok_s = cpu_port_sample()
        return {"value": tok_s, "unit": UNIT, "cores": os.cpu_count(), "kind": "port",
                "sample": f"oracle/_ref unavailable ({err}); oracle port: 1 full-width layer fwd+bwd, B=1, T=1024, {dt:.1f} s, "
                          "extrapolated by FLOP ratio"}
    secs = summ["seconds"][0]
    out = {"value": reference_train_tokens_per_s(summ, secs, T), "unit": UNIT, "cores": summ["threads"], "kind": "reference",
           "sample": _train_sample_desc(summ, secs), "dtype": summ["dtype"], "measured_seconds": secs,
           "probe_seconds_by_dtype": summ["probe_seconds"], "depth": {"llama_layers": summ["layers"], "siglip_layers": summ["siglip_layers"]}}
    for name, t in summ["probe_seconds"].items():
        out[f"value_{name}_first_sample"] = reference_train_tokens_per_s(summ, t, T)
    return out


def cpu_decode_baseline():
    """Reference `generate()` -> `greedy_decode` WITHOUT a KV cache (metamorph_llama.py:502-597), batch 1, P=128, 32 new
    tokens, full width, 2 decoder layers; extrapolated to 32 layers by the ratio of executed FLOPs."""
    summ, err = _run_ref_bench(["decode", "--new-tokens", "32", "--prompt-len", "128", "--layers", "2", "--dtype", "f32"],
                               timeout=900)
    if summ is None:
        return {"error": err, "kind": "reference"}
    H, I, V = 4096, 14336, 128258
    per_layer = H * (32 * 128 + 2 * 8 * 128 + 32 * 128) + 3 * H * I
    P, n = summ["prompt_len"], summ["new_tokens"]
    full = sum(2 * (32 * per_layer + H * V) * (P + t) + 4 * 32 * H * (P + t) ** 2 // 2 for t in range(n))
    secs_full = summ["seconds"] * full / summ["executed_flops"]
    return {"value": n / secs_full, "unit": "tokens/s", "cores": summ["threads"], "kind": "reference",
            "measured_seconds": summ["seconds"], "new_tokens": n,
            "sample": f"the reference's own generate() -> greedy_decode, no KV cache ({summ['root']}), batch 1, prompt {P}, {n} new text "
                      f"tokens, full width, {summ['layers']} of 32 decoder layers, {summ['dtype']}: {summ['seconds']:.2f} s on "
                      f"{summ['threads']} of {summ['host_threads']} host threads; extrapolated to 32 layers by executed-FLOP ratio "
                      f"({full / summ['executed_flops']:.2f}x). The reference decodes one sequence at a time."}


def decode_bench(model, dev, peaks, batch=8, prompt_len=128, new_positions=512):
    """BASELINE.json configs[3]: 512-position greedy decode, batch 8, KV cache, mixed text + 4 x 64 visual-token
    embeddings per sequence. Weights are random, so emission follows a forced schedule (SURVEY.md section 8d);
    every step still runs lm_head + argmax + the vision head / projector feedback."""
    import torch
    from metamorph_b200.constants import IMAGE_END_TOKEN_ID, IMAGE_START_TOKEN_ID
    g = torch.Generator().manual_seed(4321)
    prompts = torch.randint(0, 128000, (batch, prompt_len), generator=g)
    sched = []
    text = lambda n: torch.randint(0, 128000, (n,), generator=g).tolist()  # noqa: E731
    for _ in range(4):
        sched += text(30) + [IMAGE_START_TOKEN_ID] + [7] * 64 + [IMAGE_END_TOKEN_ID]
    sched += text(new_positions - len(sched))
    forced = torch.tensor([sched[:new_positions]] * batch, dtype=torch.int32)
    emb = model.get_model().embed_tokens(prompts.to(dev))
    model.eval()
    times = []
    for it in range(2):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        ids, imgs = model.greedy_decode(None, None, emb, max_new_tokens=new_positions - 1, output_image=True,
                                        forced_tokens=forced)
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1))
    total_ms = min(times)
    tim = model._decode.last_timing
    ms = tim["decode_ms"]                    # the 512 decode steps (device time), prefill/capture excluded
    n_vis = sum(int(x.shape[0]) for x in imgs)
    n_txt = sum(int(x.numel()) for x in ids)
    steps = new_positions
    P = 7504666624
    kv_bytes = sum(2 * 8 * 128 * 2 * 32 * (prompt_len + t) for t in range(steps)) * batch
    bytes_total = steps * (P * 2 + (4096 * 4096 + 4096 * 1152 + 1152 * 4096 + 4096 * 4096) * 2) + kv_bytes
    hbm = peaks.get("hbm_gbs", 6650.0)
    achieved = bytes_total / (ms / 1e3) / 1e9
    model.train()
    return {"metric": f"decode tokens/sec (512 new positions incl. 256 visual embeddings, batch {batch}, KV cache)",
            "value": batch * steps / (ms / 1e3), "unit": "tokens/s", "ms_per_step": ms / steps,
            "visual_embeddings": n_vis, "text_tokens": n_txt, "prompt_len": prompt_len,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": hbm, "unit": "GB/s", "frac": achieved / hbm,
                         "bytes_per_step": bytes_total / steps},
            "total_ms_incl_prefill_and_graph_capture": total_ms, "graph_capture_ms": tim["capture_ms"],
            "cuda_graph": tim["cuda_graph"],
            "timed": f"CUDA events around the 512 decode steps (prefill of the {batch}x128-token prompts and the one-off "
                     "graph capture are reported separately)"}


def preprocess_bench(dev, peaks, n_images=16, h=480, w=640, iters=20):
    """SURVEY.md section 8f row N1: the step's 16 images (640x480 RGB uint8) through the on-GPU SigLIP pre-processing,
    end to end from host memory (pinned staging -> H2D -> two resampling passes + normalisation), against the reference's
    CPU chain (Pillow BICUBIC resize + the HF processor's arithmetic) on one host core per image, as its dataset
    workers run it."""
    import time
    import numpy as np
    import torch
    from metamorph_b200.preprocess import ImageBatchPipeline, SiglipGpuImageProcessor
    from oracle import preprocess as op                       # checker / CPU leg only
    imgs = [op.synthetic_image(h, w, 100 + i) for i in range(n_images)]
    proc = SiglipGpuImageProcessor(device=dev)
    pipe = ImageBatchPipeline(proc)
    out = pipe.submit(imgs).result()
    torch.cuda.synchronize()
    ok = bool(np.array_equal(out[0].cpu().numpy(), op.siglip_preprocess(imgs[0])))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for _ in range(iters):
        out = pipe.submit(imgs).result()
    e1.record()
    torch.cuda.synchronize()
    wall = (time.perf_counter() - t0) / iters
    dev_ms = e0.elapsed_time(e1) / iters
    in_bytes = sum(im.size for im in imgs)
    side = max(h, w)
    alg_bytes = in_bytes + n_images * (2 * side * 384 * 3 + 3 * 384 * 384 * 4)   # raw read + uint8 intermediate w/r + fp32 write
    cpu = None
    try:
        from PIL import Image
        t0 = time.perf_counter()
        for im in imgs:
            sq = op.expand2square(im)
            r8 = np.asarray(Image.fromarray(sq).resize((384, 384), resample=Image.BICUBIC))
            op.rescale_normalize(r8)
        dt = time.perf_counter() - t0
        cpu = {"value": n_images / dt, "unit": "images/s", "cores": 1, "kind": "reference",
               "sample": f"{n_images} images {w}x{h}: expand2square + Pillow BICUBIC resize + HF rescale/normalise arithmetic"}
    except Exception:  # noqa: BLE001
        t0 = time.perf_counter()
        for im in imgs[:4]:
            op.siglip_preprocess(im)
        cpu = {"value": 4 / (time.perf_counter() - t0), "unit": "images/s", "cores": 1, "kind": "port",
               "sample": "4 images through oracle/preprocess.py (numpy)"}
    hbm = peaks.get("hbm_gbs", 6650.0)
    return {"metric": "SigLIP image pre-processing, host uint8 -> device fp32 [N,3,384,384]", "bit_exact_vs_oracle": ok,
            "value": n_images / wall, "unit": "images/s", "device_ms_per_batch": dev_ms, "wall_ms_per_batch": wall * 1e3,
            "images_per_batch": n_images, "input": f"{w}x{h} RGB uint8", "h2d_bytes_per_batch": in_bytes,
            "roofline": {"bound": "hbm", "achieved": alg_bytes / (dev_ms / 1e3) / 1e9, "peak": hbm, "unit": "GB/s",
                         "frac": alg_bytes / (dev_ms / 1e3) / 1e9 / hbm,
                         "note": "launch/latency-bound: 2 small launches per image, ~60 MB per batch"},
            "cpu_baseline": cpu}


DUMP_PARAM_SAMPLES = 4096      # per trainable tensor: ~200 tensors at 32 layers x 4096 x 4 B, a few MB
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir, step_out, model):
    """What the last timed step computed, as .npy files that two builds can be compared on: every value
    TrainEngine.step returned (float64), and the trainable parameters it updated, as a fixed, seeded sample of
    DUMP_PARAM_SAMPLES elements per tensor in named_parameters() order (float32; the full 8 B weights are 16 GB)."""
    import numpy as np
    import torch
    arrays = {}
    for k, v in step_out.items():
        arrays[k] = np.asarray(v.detach().cpu().double().numpy() if torch.is_tensor(v) else v, dtype=np.float64)
    g = torch.Generator().manual_seed(0)
    sample = []
    for _, p in model.named_parameters():
        if not p.requires_grad:
            continue
        idx = torch.randint(0, p.numel(), (min(DUMP_PARAM_SAMPLES, p.numel()),), generator=g)
        sample.append(p.detach().reshape(-1)[idx.to(p.device)].float().cpu())
    arrays["updated_params_sample"] = torch.cat(sample).numpy()
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_MAX_BYTES, f"--dump-outputs: {total} bytes > {DUMP_MAX_BYTES}"
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, f"{k}.npy"), a)


def run_reference_impl(args):
    """`--impl reference`: the reference's own CPU implementation of the path on the host cores, same metric/config.
    Every step is one bounded sample (see oracle/ref_bench.py); rank 0 alone runs it."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    T = args.seq_len
    summ, err = _run_ref_bench(["train", "--steps", str(args.steps), "--warmup", str(args.warmup), "--seq-len", str(T),
                                "--dtype", "auto", "--budget-s", "240"], timeout=1500)
    if summ is not None:
        secs = sum(summ["seconds"]) / len(summ["seconds"])
        v = reference_train_tokens_per_s(summ, secs, T)
        cpu = {"value": v, "unit": UNIT, "cores": summ["threads"], "kind": "reference", "sample": _train_sample_desc(summ, secs),
               "dtype": summ["dtype"], "probe_seconds_by_dtype": summ["probe_seconds"]}
        dtype = summ["dtype"]
    else:
        vals, ts = [], []
        for i in range(args.warmup + args.steps):
            dt, tok_s = cpu_port_sample()
            if i >= args.warmup:
                vals.append(tok_s)
                ts.append(dt)
        v, secs, dtype = sum(vals) / len(vals), sum(ts) / len(ts), "f32"
        cpu = {"value": v, "unit": UNIT, "cores": os.cpu_count(), "kind": "port",
               "sample": f"oracle/_ref unavailable ({err}); oracle port (oracle/restatement.py, torch fp32): 1 full-width decoder "
                         "layer fwd+bwd, B=1, T=1024 per step; extrapolated by algorithmic-FLOP ratio"}
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * secs,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": dtype,
            "data": "synthetic",
            "config": {"workload": f"LLaMA-3-8B + SigLIP-SO400M instruction-tune step, seq {T}, batch {args.batch}/GPU "
                                   "(reference arm: each step = one bounded full-width, depth-reduced CPU sample of the reference's "
                                   "own forward+backward at the same T; value extrapolated by FLOP ratio, see cpu_baseline.sample)",
                       "seq_len": T},
            "cpu_baseline": cpu,
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)
    return 0


# ------------------------------------------------------------------------------------------------
def main():
    args = parse()
    if args.impl == "reference":
        return run_reference_impl(args)

    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device: the product path has no CPU fallback"}))
        return 1
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    # NCCL writes its banner ("NCCL version ...") to stdout when the communicator is created: keep stdout for the
    # single JSON line by pointing fd 1 at stderr until the timed runs are done
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    from metamorph_b200 import ops, synthetic
    from metamorph_b200._lib import call, lib, reset_launch_count
    from metamorph_b200.engine.trainer import TrainEngine
    call("mm_check_device")

    # SURVEY section 8f N1, measured before the 8 B model and its optimizer state fill the HBM
    preprocess = None
    if rank == 0 and world == 1 and not args.no_decode:
        try:
            pk = {}
            try:
                with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
                    pk = json.load(f)
            except Exception:  # noqa: BLE001
                pass
            preprocess = preprocess_bench(dev, pk)
        except Exception as e:  # noqa: BLE001
            preprocess = {"error": repr(e)[:300]}

    torch.manual_seed(0)
    cfg = synthetic.make_config(llama=dict(num_hidden_layers=args.layers), max_len=args.seq_len)
    model = synthetic.build_model(cfg, device=dev)
    engine = TrainEngine(model, lr=6.93e-5, weight_decay=0.0, max_grad_norm=None, total_steps=1000,
                         n_save_gu_layers=min(args.save_gu_layers, args.layers), shard_optimizer=not args.no_shard,
                         fused_allgather=not args.no_fused_allgather)
    B, T = args.batch, args.seq_len
    host_batch = synthetic.train_batch(B, T, n_prompt_images=args.images_per_sample // 2,
                                       n_answer_images=args.images_per_sample - args.images_per_sample // 2,
                                       seed=1234 + 1000 * rank)
    n_images = host_batch["images"].shape[0]
    dev_batch = dict(host_batch)
    dev_batch["images"] = host_batch["images"].to(dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(batch, steps, read_loss, profile_gemm=False):
        barrier()
        reset_launch_count()
        if profile_gemm:
            ops.GEMM_PROFILE = []
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        last = out = None
        for _ in range(steps):
            out = engine.step(batch)
            if read_loss:
                last = float(out["loss"])          # device -> host read of the step's result
            else:
                last = out["loss"]
        e1.record()
        barrier()
        prof = ops.GEMM_PROFILE
        ops.GEMM_PROFILE = None
        ms = e0.elapsed_time(e1)
        launches = reset_launch_count()
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t)
        return ms, launches, prof, float(last), out

    for _ in range(args.warmup):
        engine.step(dev_batch)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms, launches, prof, loss_val, step_out = timed(dev_batch, args.steps, read_loss=False, profile_gemm=True)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, step_out, model)    # before the e2e steps below update the weights again
    tokens_per_step = world * B * T
    value = tokens_per_step * args.steps / (ms / 1e3)

    # roofline of the dominant kernel family (tcgen05 GEMM): algorithmic flops / measured launch time
    gemm_ms = sum(a.elapsed_time(b) for a, b, _ in prof)
    gemm_flops = sum(f for _, _, f in prof)
    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:  # noqa: BLE001
        pass
    peak = peaks.get("bf16_tflops_sustained")
    peak_src = "MEASURED_PEAKS.json bf16_tflops_sustained (kernel timed inside a long step)"
    if peak is None:
        peak, peak_src = 1400.0, "fallback (B200_PROFILING.md sustained)"
    achieved = gemm_flops / (gemm_ms / 1e3) / 1e12 if gemm_ms > 0 else 0.0
    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "r02_gemm_ncu_summary.json")) as f:
            traffic = json.load(f).get("dram_bytes_per_launch")
    except Exception:  # noqa: BLE001
        pass
    step_flops = train_flops_per_step(B, T, n_images, L=args.layers)
    roofline = {"bound": "tensor", "kernel": "gemm_tcgen05_kernel (all dense contractions of the step)",
                "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                "traffic": traffic, "peak_source": peak_src, "launches": len(prof),
                "gemm_share_of_step": gemm_ms / ms if ms > 0 else None,
                "step_algorithmic_tflop": step_flops / 1e12,
                "step_achieved_tflops_per_gpu": step_flops * args.steps / (ms / 1e3) / 1e12,
                "step_frac_of_peak": step_flops * args.steps / (ms / 1e3) / 1e12 / peak}

    e2e = None
    if not args.no_e2e:
        ms2, _, _, _, _ = timed(host_batch, args.steps, read_loss=True)
        h2d = host_batch["images"].numel() * 2 + (host_batch["input_ids"].numel() * 4 * 3)
        e2e = {"value": tokens_per_step * args.steps / (ms2 / 1e3), "unit": UNIT, "ms_per_step": ms2 / args.steps,
               "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": 4,
               "api": "metamorph_b200.engine.trainer.TrainEngine.step(host batch: pinned images + int tensors)"}

    # BASELINE.json configs[2] (global batch 64 = 8 samples per GPU at 8 GPUs) and configs[4] (8 frames, seq 8192) as the
    # judge asked: driver-visible extra keys of the 8-GPU line. The headline `value` keeps the per-GPU batch of the N=1 run
    # (weak scaling: fixed work per GPU), so the driver's efficiency figure stays meaningful.
    extra = {}
    peak_alloc_gb = round(torch.cuda.max_memory_allocated() / 1e9, 1)       # of the headline configuration
    peak_reserved_gb = round(torch.cuda.max_memory_reserved() / 1e9, 1)
    if args.extra_configs == "on" or (args.extra_configs == "auto" and world == 8):
        for key, (b_x, t_x, imgs_x) in (("config3_batch8", (8, args.seq_len, args.images_per_sample)),
                                        ("config5_seq8192_8frames", (2, 8192, 8))):
            try:
                torch.cuda.empty_cache()
                torch.cuda.reset_peak_memory_stats()
                # activations of the bigger shape on top of what is resident: run it only if EVERY rank has the room (an
                # out-of-memory error on one rank in the middle of a step would leave the others inside a collective)
                tok_x = b_x * t_x
                need = tok_x * (args.layers * (40960 + 57344 * min(args.save_gu_layers, args.layers) / max(args.layers, 1))
                                + 4 * 57344 + 3 * 128264) + (6 << 30)
                free = torch.tensor([torch.cuda.mem_get_info()[0]], dtype=torch.float64, device=dev)
                if world > 1:
                    dist.all_reduce(free, op=dist.ReduceOp.MIN)
                if float(free) < need:
                    extra[key] = {"skipped": f"needs ~{need / 1e9:.0f} GB free per GPU, {float(free) / 1e9:.0f} GB available"}
                    continue
                model.config.tokenizer_model_max_length = t_x
                hb = synthetic.train_batch(b_x, t_x, n_prompt_images=imgs_x // 2, n_answer_images=imgs_x - imgs_x // 2,
                                           seed=4321 + 1000 * rank)
                db = dict(hb)
                db["images"] = hb["images"].to(dev)
                for _ in range(2):
                    engine.step(db)
                ms_x, _, _, loss_x, _ = timed(db, 3, read_loss=False)
                fl = train_flops_per_step(b_x, t_x, b_x * imgs_x, L=args.layers)
                extra[key] = {"value": world * b_x * t_x * 3 / (ms_x / 1e3), "unit": UNIT, "ms_per_step": ms_x / 3,
                              "batch_per_gpu": b_x, "global_batch": world * b_x, "seq_len": t_x, "images_per_sample": imgs_x,
                              "steps": 3, "warmup": 2, "loss": loss_x,
                              "step_achieved_tflops_per_gpu": fl * 3 / (ms_x / 1e3) / 1e12,
                              "peak_hbm_gb": round(torch.cuda.max_memory_allocated() / 1e9, 1)}
            except Exception as e:  # noqa: BLE001 - an extra line must never cost the headline
                extra[key] = {"error": repr(e)[:300]}
                torch.cuda.empty_cache()
        model.config.tokenizer_model_max_length = args.seq_len
        torch.cuda.reset_peak_memory_stats()

    cpu = None
    cpu_decode = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_train_baseline(T)
        if not args.no_decode:
            cpu_decode = cpu_decode_baseline()

    decode = None
    if rank == 0 and world == 1 and not args.no_decode:
        try:
            decode = decode_bench(model, dev, peaks)
            decode["cpu_baseline"] = cpu_decode
        except Exception as e:  # noqa: BLE001 - secondary metric must not lose the headline line
            decode = {"error": repr(e)[:300]}
        if "error" not in decode:
            # beyond BASELINE's batch 8: 32 sequences share every weight byte of the step (four n8 tiles of the same MMAs)
            try:
                d32 = decode_bench(model, dev, peaks, batch=32)
                decode["batch32"] = {k: d32[k] for k in ("metric", "value", "unit", "ms_per_step", "roofline")}
            except Exception as e:  # noqa: BLE001 - an extra key must not lose the batch-8 decode line
                decode["batch32"] = {"error": repr(e)[:300]}

    sys.stdout.flush()
    os.dup2(saved_stdout, 1)
    os.close(saved_stdout)
    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                "config": {"workload": f"LLaMA-3-8B({args.layers}L)+SigLIP-SO400M-14@384 bf16 instruction-tune step "
                                       f"(fwd+bwd+AdamW fp32 master), seq_len {T}, batch {B}/GPU, {n_images // B} images/sample "
                                       "(64 visual tokens each), synthetic seeded inputs, random-init weights",
                           "global_batch": world * B, "seq_len": T, "parallelism": f"dp{world}",
                           "l2_policy": "inputs+weights (>100 GB/step) far exceed the 126 MB L2; no flush needed",
                           "max_grad_norm": None,
                           "optimizer": "AdamW fused into the backward sweep, fp32 master/m/v " +
                                        ((f"sharded over the {world} ranks (ZeRO-1: " + ("" if getattr(engine, "fused_reduce", False) else "NCCL reduce-scatter -> ") + "AdamW on the slice, "
                                          + ("IN-SWITCH gradient sum (multimem.ld_reduce) + " if getattr(engine, "fused_reduce", False) else "")
                                          + ("the same kernel broadcasts the updated slice into every replica (symmetric memory"
                                             + (", NVSwitch multicast)" if engine.fused_allgather and int(engine.layer_buckets[0].symm.multicast_ptr or 0) and engine.use_multicast else ", P2P stores)")
                                             if engine.fused_allgather else "-> NCCL all-gather") + ")")
                                         if engine.shard_world > 1 else "on this GPU"),
                           "optimizer_state_gb_per_gpu": round(engine.optimizer_state_bytes() / 1e9, 2),
                           "recompute": f"gate/up GEMM recomputed in {args.layers - min(args.save_gu_layers, args.layers)} of {args.layers} layers; norms always",
                           "lm_head_rows": "lm_head+CE run on the %d of %d rows that carry a label (identical loss/grads; "
                                           "algorithmic FLOPs below still count all rows)" % engine.hot.last_head_rows,
                           "loss": loss_val,
                           "peak_hbm_gb": peak_alloc_gb, "peak_hbm_reserved_gb": peak_reserved_gb},
                "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "decode": decode, "preprocess": preprocess, "gpu_launches": launches, "clocks": clocks}
        line.update(extra)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
