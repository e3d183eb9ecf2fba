"""The reference's own training step on this GPU, for comparison with scripts/bench_train.py: the UNMODIFIED reference modules
(oracle/_ref, oracle/install_ref.sh) driven like autoregressive/train/train_c2i_canny.py:190-211 — fp32 parameters,
`torch.autocast(bf16)`, `model(cond_idx, idx, targets, condition)`, `loss.backward()`, `torch.optim.AdamW(fused=True).step()` —
on the BASELINE.json config-5 shape (LlamaGen-L c2i 256 x 256, DINOv2-small canny adapter, 32 images per GPU), PyTorch eager.
--freeze-adapter stops the gradient at the control tokens, which is where controlar_b200's backward stops (like for like);
without it the reference also differentiates the DINOv2 encoder.  Prints one JSON line (CUDA-event medians)."""
import argparse
import contextlib
import io
import json
import os
import sys
import tempfile
import warnings

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--model", default="GPT-L")
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--image-size", type=int, default=256)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--freeze-adapter", action="store_true")
    ap.add_argument("--device", default="cuda")
    args = ap.parse_args()
    warnings.filterwarnings("ignore")
    dev = torch.device(args.device)
    ref_root = os.path.join(ROOT, "oracle", "_ref")
    assert os.path.isdir(os.path.join(ref_root, "autoregressive", "models")), "oracle/_ref missing: run oracle/install_ref.sh <reference checkout>"
    from transformers import Dinov2Config, Dinov2Model
    n = (args.image_size // 16) ** 2
    old_cwd = os.getcwd()
    with tempfile.TemporaryDirectory() as tmp:
        d = os.path.join(tmp, "autoregressive", "models", "dinov2-small")          # dinov2_adapter.py:13 loads it relative to CWD
        os.makedirs(d)
        Dinov2Model(Dinov2Config(hidden_size=384, num_hidden_layers=12, num_attention_heads=6, mlp_ratio=4, patch_size=14, image_size=518,
                                 layerscale_value=1.0, qkv_bias=True, layer_norm_eps=1e-6)).save_pretrained(d)
        os.chdir(tmp)
        sys.path.insert(0, ref_root)
        with contextlib.redirect_stdout(io.StringIO()):
            from autoregressive.models.gpt_t2i import GPT_models as REF_GPT
            torch.manual_seed(0)
            model = REF_GPT[args.model](vocab_size=16384, block_size=n, num_classes=1000, cls_token_num=1, model_type="c2i",
                                        condition_type="canny", adapter_size="small", token_dropout_p=0.0, resid_dropout_p=0.0,
                                        ffn_dropout_p=0.0)
        os.chdir(old_cwd)
    model.output.weight.data.normal_(0, 0.02)
    model = model.to(dev).train()
    if args.freeze_adapter:
        for p in model.adapter.parameters():
            p.requires_grad_(False)
    params = [p for p in model.parameters() if p.requires_grad]
    opt = torch.optim.AdamW(params, lr=1e-4, betas=(0.9, 0.95), weight_decay=0.05, fused=(dev.type == "cuda"))
    g = torch.Generator(device=dev).manual_seed(1)
    B = args.batch
    z = torch.randint(0, 16384, (B, n), device=dev, generator=g)
    labels = torch.randint(0, 1000, (B,), device=dev, generator=g)
    canny = (torch.rand(B, 1, args.image_size, args.image_size, device=dev, generator=g) > 0.9).float().repeat(1, 3, 1, 1) * 2 - 1
    cuda = dev.type == "cuda"
    rows = []
    import time
    for it in range(args.warmup + args.steps):
        if cuda:
            e = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
            torch.cuda.synchronize()
            mark = lambda i: e[i].record()
        else:
            ts = [0.0] * 4

            def mark(i):
                ts[i] = time.perf_counter()
        with torch.enable_grad():
            mark(0)
            with torch.autocast(dev.type, dtype=torch.bfloat16):
                _, loss = model(cond_idx=labels, idx=z[:, :-1], targets=z, condition=canny)
            mark(1)
            loss.backward()
            mark(2)
            opt.step()
            opt.zero_grad(set_to_none=True)
            mark(3)
        if cuda:
            torch.cuda.synchronize()
            t = [e[i].elapsed_time(e[i + 1]) for i in range(3)]
        else:
            t = [1000.0 * (ts[i + 1] - ts[i]) for i in range(3)]
        if it >= args.warmup:
            rows.append((*t, float(loss.detach())))
    med = lambda i: sorted(r[i] for r in rows)[len(rows) // 2]
    total = med(0) + med(1) + med(2)
    print(json.dumps({"impl": "reference modules (oracle/_ref, unmodified), PyTorch eager, bf16 autocast, torch " + torch.__version__,
                      "workload": f"{args.model} c2i {args.image_size}^2 training step, batch {B} per GPU", "adapter_frozen": args.freeze_adapter,
                      "forward_loss_ms": med(0), "backward_ms": med(1), "adamw_ms": med(2), "images_per_s": 1000.0 * B / total,
                      "loss_first": rows[0][3], "loss_last": rows[-1][3], "steps": args.steps, "warmup": args.warmup}))


if __name__ == "__main__":
    main()
