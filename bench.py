#!/usr/bin/env python
"""bench.py — images/sec of the ControlAR conditional-decoding hot path (BASELINE.json metric) on N GPUs.

One "step" = one pass of the hot path over one batch of synthetic input: control map -> DINOv2 + adapter_mlp ->
prefill -> N-1 KV-cache decode steps with CFG + top-k sampling -> VQGAN decode of the token grids, i.e. exactly
`generate()` + `decode_code()` of autoregressive/sample/sample_t2i.py:163-176, through this repo's drop-in modules.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--config 2|3|4|4t] [--dump-outputs DIR]

  --config 2  (default) BASELINE.json configs[1]: XL + DINOv2-small canny, 512x512, batch 8 per GPU
  --config 3  configs[2]: XL + DINOv2-base depth, 512x512, batch 8 per GPU (64 images on 8 GPUs)
  --config 4  configs[3]: XL canny_MR 768x512 (W x H, 1536 tokens, RoPE table side 48), batch 4; 4t = 512x768 (tall)

N > 1 is launched with torchrun (one rank per GPU); every rank generates its own `--batch` images (weak scaling)
and the int32 token grids are all-gathered once over NCCL.  `--dump-outputs DIR` saves what the last timed step returned to its
caller (rank 0's token grids and decoded images); inputs, weights and sampling seeds depend only on the arguments, so two builds
run with the same arguments can be compared output for output.  `--impl reference` times the CPU restatement of the
reference path (oracle/, kind "port": the reference is Python and /root/reference does not exist on the GPU box)
on the host cores.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True        # no __pycache__ beside the sources: bench.py leaves the tree as build() left it

import torch


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--size", type=int, default=512)
    ap.add_argument("--height", type=int, default=0, help="non-square generation (config 4: --height 512 --width 768); default --size")
    ap.add_argument("--width", type=int, default=0)
    ap.add_argument("--adapter-size", default="small", choices=["small", "base"], help="DINOv2-small (config 2) or -base (config 3)")
    ap.add_argument("--condition-type", default="canny", help="canny | depth | hed | lineart | seg (config 3: depth)")
    ap.add_argument("--model", default="GPT-XL")
    ap.add_argument("--cfg-scale", type=float, default=4.0)
    ap.add_argument("--top-k", type=int, default=2000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-eager", action="store_true", help="skip the reference PyTorch-eager measurement on the GPU (gpu_eager_baseline)")
    ap.add_argument("--ref-compile", action="store_true", help="also time the reference's torch.compile(mode='reduce-overhead') path (minutes of compile)")
    ap.add_argument("--config", default="2", choices=["2", "3", "4", "4t"], help="BASELINE.json config preset (sets size/batch/adapter/condition)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the token grids and images of the last timed step (rank 0) to DIR/<name>.npy as float32")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs applies to the timed GPU path (--impl ours)")
    if a.config == "3":
        a.adapter_size, a.condition_type = "base", "depth"
    elif a.config in ("4", "4t"):
        a.batch = 4
        a.height, a.width = (512, 768) if a.config == "4" else (768, 512)
    return a


WORKLOADS = {
    "2": "configs[1]: LlamaGen-XL t2i + DINOv2-small canny, 512x512 (1024 tokens), batch=8/GPU, cfg 4.0, top-k 2000",
    "3": "configs[2]: LlamaGen-XL t2i + DINOv2-base depth, 512x512 (1024 tokens), batch=8/GPU (64 images on 8 GPUs), cfg 4.0, top-k 2000",
    "4": "configs[3]: LlamaGen-XL canny_MR 768x512 (W x H; 1536 tokens, 32 rows x 48 columns, RoPE table side 48), batch=4, cfg 4.0, top-k 2000, incl. VQGAN decode",
    "4t": "configs[3] (tall): LlamaGen-XL canny_MR 512x768 (W x H; 1536 tokens, 48 rows x 32 columns, linear RoPE index), batch=4, cfg 4.0, top-k 2000, incl. VQGAN decode",
}
WORKLOAD = WORKLOADS["2"]


# ---------------------------------------------------------------------------------------------------------------
# clocks sampler (recipe: /opt/skills/guides/B200_PROFILING.md)
# ---------------------------------------------------------------------------------------------------------------
class ClockSampler:
    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}",
                 "--query-gpu=clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
                 "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
                 "clocks_event_reasons.sw_power_cap", "--format=csv,noheader,nounits", "-lms", "200"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = max([float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()] or [0.0])
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": reasons,
                "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------------------
# CPU baseline = the oracle port (the reference is Python; /root/reference does not exist on the GPU box), SURVEY.md 8(d):
# full batch (B_eff = 2B rows), prefill + 32 sampled decode steps (median of 3 groups) + DINOv2 and VQ decode of one image each,
# extrapolated x(N-1) — the reference's decode-step cost is position independent (it attends over all S slots every step,
# gpt_t2i.py:276-286)
# ---------------------------------------------------------------------------------------------------------------
def _dims(args):
    H_img, W_img = (args.height or args.size), (args.width or args.size)
    return H_img, W_img, H_img // 16, W_img // 16


_CPU_CACHE = {}


def cpu_reference_images_per_sec(args, n_decode_steps=32, repeats=3, threads=None):
    from oracle.weights import GPTSpec, make_gpt_state_dict, make_vq_state_dict, dinov2_shapes, _fill
    from oracle.ar_oracle import AROracle, cfg_combine, sample_from_logits
    from oracle.vision_oracle import dinov2_adapter_oracle, vq_decode_oracle
    from controlar_b200.synthetic import text_inputs, control_map
    cores = threads or min(os.cpu_count() or 1, 32)     # more threads than this only thrash on the shared GPU hosts
    torch.set_num_threads(cores)
    dims = {"GPT-XL": (1280, 36, 20), "GPT-L": (1024, 24, 16), "GPT-B": (768, 12, 12)}[args.model]
    H_img, W_img, gh, gw = _dims(args)
    g = max(gh, gw)
    spec = GPTSpec(dim=dims[0], n_layer=dims[1], n_head=dims[2], vocab_size=16384, cls_token_num=120, block_size=g * g,
                   model_type="t2i", adapter_size=args.adapter_size, condition_type=args.condition_type)
    if "orc" not in _CPU_CACHE:                       # procedural XL weights take ~20 s to draw: once per process
        _CPU_CACHE["orc"] = AROracle(spec, make_gpt_state_dict(spec, 0, with_adapter=False), torch.bfloat16)
        _CPU_CACHE["vsd"] = make_vq_state_dict(0)
    orc = _CPU_CACHE["orc"]
    B, N, T = args.batch, gh * gw, 120
    cond, masks = text_inputs(T, spec.caption_dim, B, 1)
    ctype = "canny" if args.condition_type in ("canny", "seg") else "depth"
    cmap = control_map(1, H_img, W_img, 2, ctype)
    hidden = 384 if args.adapter_size == "small" else 768
    dsd = _fill(dinov2_shapes(hidden, prefix="model."), 0, 0.02)
    t0 = time.perf_counter()
    feat = dinov2_adapter_oracle(dsd, cmap[:1], args.condition_type, torch.bfloat16, heads=hidden // 64).float()
    t_dino = (time.perf_counter() - t0) * B
    t0 = time.perf_counter()
    ctrl = orc.mlp(orc.r(feat), "adapter_mlp").repeat(B, 1, 1)
    cc = torch.cat([cond, torch.zeros_like(cond) + orc.w["cls_embedding.uncond_embedding"]])
    cic = torch.cat([ctrl, torch.zeros_like(ctrl)])
    orc.setup_caches(2 * B, T + N)
    orc.apply_emb_masks(torch.cat([masks, masks]))
    lg = orc.prefill(cc, cic, 1.0)[:, -1]
    tok, _ = sample_from_logits(cfg_combine(lg, args.cfg_scale), top_k=args.top_k)
    t_prefill = time.perf_counter() - t0
    per_step = []
    i = 0
    for _ in range(repeats):
        t0 = time.perf_counter()
        for _ in range(n_decode_steps):
            t = tok.view(-1)
            lg = orc.decode(torch.cat([t, t]), T + i)
            tok, _ = sample_from_logits(cfg_combine(lg, args.cfg_scale), top_k=args.top_k)
            i += 1
        per_step.append((time.perf_counter() - t0) / n_decode_steps)
    t_step = sorted(per_step)[len(per_step) // 2]
    vsd = _CPU_CACHE["vsd"]
    codes = torch.randint(0, 16384, (1, N))
    t0 = time.perf_counter()
    vq_decode_oracle(vsd, codes, [1, 8, gh, gw])
    t_vq = (time.perf_counter() - t0) * B
    total = t_dino + t_prefill + t_step * (N - 1) + t_vq
    spread = (max(per_step) - min(per_step)) / t_step
    sample = (f"CPU port of the reference (oracle/), bf16 AR + fp32 VQ, full batch {B} (B_eff {2 * B}): prefill {t_prefill:.1f}s, "
              f"{repeats} x {n_decode_steps} sampled decode steps, median {t_step:.3f}s/step (spread {100 * spread:.0f}%) extrapolated x{N - 1}, "
              f"DINOv2-{args.adapter_size} 1 img {t_dino / B:.2f}s x{B}, VQ decode 1 img {t_vq / B:.1f}s x{B}; images/s = {B} / total")
    return B / total, cores, sample


# ---------------------------------------------------------------------------------------------------------------
# Reference GPU baseline (SURVEY.md 8(d)): the UNMODIFIED reference modules from oracle/_ref (oracle/install_ref.sh, run by build()) run
# eagerly on this GPU through the reference's own generate() + decode_code() (sample_t2i.py:163-176).  Warm-up 1 short call,
# then the median of 3 full calls, CUDA events.  The north_star target (>= 4x) is defined against this number.
# ---------------------------------------------------------------------------------------------------------------
def gpu_eager_reference(args, dev, cond_d, masks_d, cmap_d, n_calls=3, compile_too=False):
    ref_root = os.path.join(ROOT, "oracle", "_ref")
    if not os.path.isdir(os.path.join(ref_root, "autoregressive", "models")):
        return {"unavailable": "oracle/_ref missing: build() makes it where a checkout of the reference exists (oracle/install_ref.sh)"}
    import contextlib, io, tempfile, warnings
    warnings.filterwarnings("ignore")
    H_img, W_img, gh, gw = _dims(args)
    g = max(gh, gw)
    N, B = gh * gw, args.batch
    old_cwd, old_path = os.getcwd(), list(sys.path)
    out = {}
    try:
        from transformers import Dinov2Config, Dinov2Model
        hidden = 384 if args.adapter_size == "small" else 768
        with tempfile.TemporaryDirectory() as tmp:
            d = os.path.join(tmp, "autoregressive", "models", f"dinov2-{args.adapter_size}")      # dinov2_adapter.py:13 loads it relative to CWD
            os.makedirs(d)
            Dinov2Model(Dinov2Config(hidden_size=hidden, num_hidden_layers=12, num_attention_heads=hidden // 64, mlp_ratio=4, patch_size=14,
                                     image_size=518, layerscale_value=1.0, qkv_bias=True, layer_norm_eps=1e-6)).save_pretrained(d)
            os.chdir(tmp)
            sys.path.insert(0, ref_root)
            for k in [k for k in sys.modules if k.split(".")[0] in ("autoregressive", "tokenizer", "utils")]:
                del sys.modules[k]
            with contextlib.redirect_stdout(io.StringIO()):
                from autoregressive.models.gpt_t2i import GPT_models as REF_GPT
                from autoregressive.models.generate import generate as ref_generate
                from tokenizer.tokenizer_image.vq_model import VQ_models as REF_VQ
                torch.manual_seed(0)
                gpt = REF_GPT[args.model](block_size=g * g, cls_token_num=120, model_type="t2i", condition_type=args.condition_type,
                                          adapter_size=args.adapter_size).eval()
            gpt.output.weight.data.normal_(0, 0.02)
            gpt = gpt.to(dev, torch.bfloat16)
            vq = REF_VQ["VQ-16"](codebook_size=16384, codebook_embed_dim=8).to(dev).eval()
            os.chdir(old_cwd)
        kw = dict(cfg_scale=args.cfg_scale, temperature=1.0, top_k=args.top_k, top_p=1.0, sample_logits=True)

        def call(n_tokens, fn):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            with torch.no_grad():
                toks = fn(gpt, cond_d, n_tokens, masks_d, condition=cmap_d, **kw)
                if n_tokens == N:
                    vq.decode_code(toks, [B, 8, gh, gw])
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1)
        call(32, ref_generate)                                 # warm-up (cuBLAS / cuDNN handles, allocator)
        ms = sorted(call(N, ref_generate) for _ in range(n_calls))
        med = ms[len(ms) // 2]
        out = {"value": B / (med * 1e-3), "unit": "images/s", "ms_per_batch": med, "ms_per_decode_step": med / N, "calls": n_calls,
               "spread": (ms[-1] - ms[0]) / med, "impl": "reference modules (oracle/_ref, unmodified) PyTorch eager, bf16 AR + fp32 VQ, "
               f"torch {torch.__version__}", "config": f"{args.model} {W_img}x{H_img} batch {B} cfg {args.cfg_scale} top-k {args.top_k}"}
        if compile_too:
            try:
                import autoregressive.models.generate as G
                G.decode_one_token = torch.compile(G.decode_one_token, mode="reduce-overhead", fullgraph=True)    # sample_t2i.py:85-91
                call(32, ref_generate); call(32, ref_generate)
                ms2 = sorted(call(N, ref_generate) for _ in range(n_calls))
                out["compiled_reduce_overhead"] = {"value": B / (ms2[len(ms2) // 2] * 1e-3), "unit": "images/s", "ms_per_batch": ms2[len(ms2) // 2]}
            except Exception as e:       # noqa: BLE001 — informational arm
                out["compiled_reduce_overhead"] = {"unavailable": str(e)[:200]}
        del gpt, vq
        torch.cuda.empty_cache()
    except Exception as e:               # noqa: BLE001 — the baseline must never take the bench line down
        out = {"unavailable": f"{type(e).__name__}: {str(e)[:300]}"}
    finally:
        os.chdir(old_cwd)
        sys.path[:] = old_path
        for k in [k for k in sys.modules if k.split(".")[0] in ("autoregressive", "tokenizer", "utils") and "controlar_b200" not in k]:
            del sys.modules[k]
    return out


# ---------------------------------------------------------------------------------------------------------------
def _config_block(args, world):
    H_img, W_img, gh, gw = _dims(args)
    return {"workload": WORKLOADS[args.config] if (args.model, args.cfg_scale, args.top_k) == ("GPT-XL", 4.0, 2000) and
            (args.config != "2" or (H_img, W_img, args.batch, args.adapter_size, args.condition_type) == (512, 512, 8, "small", "canny"))
            else f"{args.model} t2i + DINOv2-{args.adapter_size} {args.condition_type}, {W_img}x{H_img}, batch={args.batch}/GPU",
            "global_batch": world * args.batch, "tokens_per_image": gh * gw,
            "parallelism": f"dp{world} (batch sharded, one all-gather of token grids)",
            "l2": "working set larger than L2 (weights 1.5 GB + KV cache up to 3.4 GB stream every decode step)",
            "sampling": {"cfg_scale": args.cfg_scale, "top_k": args.top_k, "temperature": 1.0, "top_p": 1.0}}


DUMP_BYTES = 64_000_000        # cap on everything --dump-outputs writes, .npy headers included (64 MB, decimal)
NPY_HEADER = 128               # bytes np.save puts in front of a 1- to 4-d float array


def dump_outputs(path, arrays):
    """One float32 DIR/<name>.npy per output, smallest first; each output may use an even share of what DUMP_BYTES has left, so the
    budget the small ones leave unused goes to the larger.  An output larger than its share is cut to a fixed seeded sample of its
    elements, whose flat indices go to DIR/<name>_index.npy (float64: 12 bytes per sampled element with the value)."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    left = DUMP_BYTES
    for i, (name, t) in enumerate(sorted(arrays.items(), key=lambda kv: kv[1].numel())):
        share = left // (len(arrays) - i)
        a = t.float().numpy()
        if a.nbytes + NPY_HEADER > share:
            idx = np.sort(np.random.default_rng(0).choice(a.size, (share - 2 * NPY_HEADER) // 12, replace=False))
            np.save(os.path.join(path, name + "_index.npy"), idx.astype(np.float64))
            left -= idx.size * 8 + NPY_HEADER
            a = a.reshape(-1)[idx]
        np.save(os.path.join(path, name + ".npy"), a)
        left -= a.nbytes + NPY_HEADER


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # one step = the bounded CPU sample of the workload (cpu_reference_images_per_sec: the full batch, prefill + 3 x 32 decode steps,
    # about a minute of host work): one untimed sample if warm-up is requested, then exactly `steps` timed ones
    vals = []
    n_warm = 0
    if args.warmup > 0:
        cpu_reference_images_per_sec(args, n_decode_steps=4, repeats=1)        # touches every weight page once
        n_warm = 1
    while len(vals) < args.steps:
        ips, cores, sample = cpu_reference_images_per_sec(args)
        vals.append(ips)
    v = sorted(vals)[len(vals) // 2]
    line = {"metric": "images/sec", "value": v, "unit": "images/s", "n_gpus": args.gpus, "steps": len(vals), "warmup": n_warm,
            "ms_per_step": 1000.0 * args.batch / v, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic", "impl": "reference", "config": _config_block(args, args.gpus),
            "cpu_baseline": {"value": v, "unit": "images/s", "cores": cores, "kind": "port", "sample": sample,
                             "all_samples": vals},
            "e2e": {"value": v, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def run_ours(args):
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    from controlar_b200.build import build
    if rank == 0:
        build()
    if world > 1:
        dist.barrier()
    from controlar_b200 import _lib
    from controlar_b200.autoregressive.models.gpt_t2i import GPT_models
    from controlar_b200.autoregressive.models.generate import generate
    from controlar_b200.tokenizer.tokenizer_image.vq_model import VQ_models
    from controlar_b200.parallel import gather_token_grids, rank_seed
    from controlar_b200.synthetic import text_inputs, control_map     # seeded synthetic inputs

    torch.manual_seed(0)
    H_img, W_img = (args.height or args.size), (args.width or args.size)
    gh, gw = H_img // 16, W_img // 16
    g = max(gh, gw)                                   # RoPE table side = image_size / 16 (sample_t2i_MR.py:72-74)
    N, T, B = gh * gw, 120, args.batch
    gpt = GPT_models[args.model](block_size=g * g, cls_token_num=T, model_type="t2i", condition_type=args.condition_type,
                                 adapter_size=args.adapter_size).eval()
    gpt.output.weight.data.normal_(0, 0.02)          # the reference zero-inits the head (gpt_t2i.py:377)
    for blk in gpt.adapter.model.encoder.layer:      # HF init has layerscale 1.0
        blk.layer_scale1.lambda1.data.fill_(1.0); blk.layer_scale2.lambda1.data.fill_(1.0)
    gpt = gpt.to(dev, torch.bfloat16)
    vq = VQ_models["VQ-16"](codebook_size=16384, codebook_embed_dim=8).to(dev).eval()
    cond_h, masks_h = text_inputs(T, 2048, B, 1000 + rank, torch.bfloat16)
    cmap_h = control_map(B, H_img, W_img, 2000 + rank, args.condition_type, torch.bfloat16)
    cond_h, masks_h, cmap_h = cond_h.pin_memory(), masks_h.pin_memory(), cmap_h.pin_memory()
    img_h = torch.empty((B, 3, H_img, W_img), dtype=torch.float32).pin_memory()
    cond_d, masks_d, cmap_d = cond_h.to(dev), masks_h.to(dev), cmap_h.to(dev)
    kw = dict(cfg_scale=args.cfg_scale, temperature=1.0, top_k=args.top_k, top_p=1.0, sample_logits=True)
    lib = _lib.lib()
    t_decode = []

    def one_step(step_idx, host_io):
        if host_io:
            c, m, x = cond_h.to(dev, non_blocking=True), masks_h.to(dev, non_blocking=True), cmap_h.to(dev, non_blocking=True)
        else:
            c, m, x = cond_d, masks_d, cmap_d
        # rank seed mirrors sample_c2i_ddp.py:47 (global_seed * world + rank), advanced per step
        toks = generate(gpt, c, N, emb_masks=m, condition=x, seed=rank_seed(step_idx, world, rank), **kw)
        allt = gather_token_grids(toks)                  # the single NCCL all-gather of finished token grids (world > 1)
        img = vq.decode_code(toks, [B, 8, gh, gw])
        if host_io:
            img_h.copy_(img, non_blocking=True)
        return toks, img

    def timed(n_steps, host_io, first_idx):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n_steps):
            last = one_step(first_idx + i, host_io)
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms), last

    for i in range(args.warmup):
        one_step(i, False)
    torch.cuda.synchronize()
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    lib.car_launch_count(1)
    ms, (last_toks, last_img) = timed(args.steps, False, args.warmup)
    launches = int(lib.car_launch_count(0))
    outputs = {"tokens": last_toks.cpu(), "images": last_img.cpu()} if args.dump_outputs and rank == 0 else None
    ms_e2e, _ = timed(args.steps, True, args.warmup + args.steps)
    # decode-loop roofline: time the device-side decode loop alone (prefill excluded) with CUDA events on the stream
    # the kernels are launched on (torch's current stream is the stream handed to the library)
    st = gpt._car_state
    cc = torch.cat([cond_d, torch.zeros_like(cond_d) + gpt.cls_embedding.uncond_embedding])
    ctrl = gpt._car_encoder.forward(cmap_d, apply_mlp=True)
    cic = torch.cat([ctrl, torch.zeros_like(ctrl)])
    from controlar_b200.engine import make_sampling
    sp = make_sampling(1.0, args.top_k, 1.0, True, args.cfg_scale, -1, 7)
    dec_ms = []
    ts_buf = torch.zeros(N, dtype=torch.int64, device=dev)
    st.set_step_timer(ts_buf)                         # one 8-byte store per token by one thread: ms/step versus context length
    for _ in range(max(min(args.steps, 5), 3)):
        st.prefill(cc, cic, 1.0, all_rows=False)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); st.generate(sp, N, None, dev); e1.record()
        torch.cuda.synchronize()
        dec_ms.append(e0.elapsed_time(e1))
    st.set_step_timer(None)
    dec_ms = sorted(dec_ms)[len(dec_ms) // 2]
    # algorithmic bytes (SURVEY.md 8(d)): decode iteration k (k = 0 .. N-2) decodes position T + k with context n = T + 1 + k
    step_bytes = sum(st.step_bytes(T + 1 + k) for k in range(N - 1))
    ts = ts_buf.cpu().tolist()                        # last launch: ts[s] = start of iteration s; iteration k spans ts[k] .. ts[k+1]
    clk = clocks.stop() if rank == 0 else None
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    achieved = step_bytes / (dec_ms * 1e-3) / 1e9
    # per-step table: mean ms/step and HBM fraction over windows of 32 iterations, and at the last iteration (n = T + N - 1)
    table = []
    for k0 in list(range(0, N - 2, 128)) + [N - 2 - 32]:
        k1 = min(k0 + 32, N - 2)
        if k1 <= k0 or ts[k1] <= ts[k0]:
            continue
        ms_k = (ts[k1] - ts[k0]) * 1e-6 / (k1 - k0)
        by = sum(st.step_bytes(T + 1 + k) for k in range(k0, k1)) / (k1 - k0)
        table.append({"n": T + 1 + (k0 + k1) // 2, "ms_per_step": round(ms_k, 4), "frac": round(by / (ms_k * 1e-3) / 1e9 / peak, 4)})
    # numeric DRAM traffic of the decode kernel: ncu --set full of a short launch of the same kernel (committed summary), scaled by
    # the algorithmic bytes of this launch (ncu replays each kernel ~40 times: a 1023-token launch cannot be captured whole)
    traffic, traffic_note = None, "no ncu summary found (profiles/r2_pk_traffic.json)"
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "r2_pk_traffic.json")))
        ratio = float(tj["dram_bytes"]) / float(tj["algorithmic_bytes"])
        traffic = ratio * step_bytes
        traffic_note = (f"dram__bytes_read.sum + dram__bytes_write.sum = {ratio:.3f} x algorithmic bytes in the ncu --set full capture of a "
                        f"{tj.get('tokens', '?')}-token launch ({tj.get('source', 'profiles/')}), scaled to this launch")
    except Exception:
        pass
    value = world * B * args.steps / (ms * 1e-3)
    e2e = world * B * args.steps / (ms_e2e * 1e-3)
    line = {
        "metric": "images/sec", "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic",
        "config": _config_block(args, world),
        "e2e": {"value": e2e, "unit": "images/s",
                "h2d_bytes_per_step": int(cond_h.numel() * 2 + masks_h.numel() * 8 + cmap_h.numel() * 2),
                "d2h_bytes_per_step": int(img_h.numel() * 4)},
        "gpu_launches": launches,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "traffic_note": traffic_note, "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6.65 TB/s",
                     "kernel": "pk_decode_kernel: persistent decode loop (per token 36 x {qkv | attention | wo | w1w3 | w2} + head + CFG/top-k sampler), one launch per generate()",
                     "algorithmic_bytes": step_bytes, "n_range": [T + 1, T + N - 1], "decode_ms": dec_ms, "ms_per_token": dec_ms / (N - 1),
                     "per_step": table},
        "clocks": clk,
    }
    if not args.no_gpu_eager and world == 1:
        # the reference's own PyTorch-eager path on this GPU (the north_star target is >= 4x this)
        ge = gpu_eager_reference(args, dev, cond_d, masks_d, cmap_d, compile_too=args.ref_compile)
        line["gpu_eager_baseline"] = ge
        if "value" in ge:
            line["vs_gpu_eager"] = {"e2e_ratio": e2e / ge["value"], "note": "ours e2e (host copies timed) / reference eager (inputs resident)"}
    if not args.no_cpu_baseline and world == 1:
        v, cores, sample = cpu_reference_images_per_sec(args, n_decode_steps=16, repeats=3)
        line["cpu_baseline"] = {"value": v, "unit": "images/s", "cores": cores, "kind": "port", "sample": sample}
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
