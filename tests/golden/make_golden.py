#!/usr/bin/env python
"""Generate the committed golden fixtures by running the REFERENCE ITSELF (read-only import from
/root/reference) on CPU with procedural weights (oracle/weights.py).  Run from the repo root in the build
container only:

    python tests/golden/make_golden.py [case ...]

The GPU box has no /root/reference; tests there only read tests/golden/*.pt.  Each fixture records the torch /
transformers versions it was made with.  Weights are NOT stored: tests rebuild them from (spec, seed).
"""
from __future__ import annotations

import os
import sys
import tempfile
import contextlib
import io

REPO = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
REF = "/root/reference"
OUT = os.path.join(REPO, "tests", "golden")
sys.path.insert(0, REPO)
sys.path.insert(0, REF)       # reference first: `autoregressive.*`, `tokenizer.*`, `utils.*` resolve to it

import torch
import transformers

from oracle.weights import GPTSpec, make_gpt_state_dict, make_vq_state_dict, gpt_shapes, vq_shapes
from oracle.inputs import text_inputs, class_inputs, control_map, xl_ctrl_in

torch.set_grad_enabled(False)


def math_sdpa():
    """Force the math SDPA backend — the one the reference itself forces in decode (generate.py:120) — for
    prefill too.  On CPU the default backend for bf16 is the fused flash kernel, whose internal rounding differs
    from the math path by ~1e-3 relative (and from whatever backend a GPU run would pick); pinning the oracle
    needs one defined arithmetic.  `*_defaultsdpa` fixtures keep the platform-default spread on record."""
    import warnings
    warnings.filterwarnings("ignore", category=FutureWarning)
    return torch.backends.cuda.sdp_kernel(enable_flash=False, enable_mem_efficient=False, enable_math=True)


def header():
    return {"torch": str(torch.__version__), "transformers": str(transformers.__version__), "device": "cpu",
            "generator": "tests/golden/make_golden.py"}


@contextlib.contextmanager
def fake_hf_cwd(adapter_size: str):
    """dinov2_adapter.py:13 loads 'autoregressive/models/dinov2-{size}' relative to CWD."""
    from transformers import Dinov2Config, Dinov2Model
    hidden = 384 if adapter_size == "small" else 768
    cfg = Dinov2Config(hidden_size=hidden, num_hidden_layers=12, num_attention_heads=hidden // 64, mlp_ratio=4,
                       patch_size=14, image_size=518, layerscale_value=1.0, qkv_bias=True, layer_norm_eps=1e-6)
    old = os.getcwd()
    with tempfile.TemporaryDirectory() as tmp:
        d = os.path.join(tmp, "autoregressive", "models", f"dinov2-{adapter_size}")
        os.makedirs(d)
        Dinov2Model(cfg).save_pretrained(d)
        os.chdir(tmp)
        try:
            yield
        finally:
            os.chdir(old)


def build_ref_gpt(spec: GPTSpec, seed: int, dtype, **model_kw):
    from autoregressive.models.gpt_t2i import Transformer, ModelArgs
    with fake_hf_cwd(spec.adapter_size), contextlib.redirect_stdout(io.StringIO()):
        m = Transformer(ModelArgs(dim=spec.dim, n_layer=spec.n_layer, n_head=spec.n_head,
                                  multiple_of=spec.multiple_of, vocab_size=spec.vocab_size,
                                  cls_token_num=spec.cls_token_num, block_size=spec.block_size,
                                  caption_dim=spec.caption_dim, num_classes=spec.num_classes,
                                  model_type=spec.model_type, adapter_size=spec.adapter_size,
                                  condition_type=spec.condition_type, **model_kw))
    sd = make_gpt_state_dict(spec, seed)
    ref_sd = m.state_dict()
    assert set(ref_sd.keys()) == set(sd.keys()), (set(ref_sd) ^ set(sd))
    for k in sd:
        assert tuple(ref_sd[k].shape) == tuple(sd[k].shape), k
    m.load_state_dict(sd, strict=True)
    return m.to(dtype).eval()


def ar_case(name: str, spec: GPTSpec, B: int, H: int, W: int, cfg_scale: float, cs: float, dtype, seed: int = 0,
            logit_steps=(0, 1, 2, 7), sampled: bool = True, save_all_logits: bool = True, force_math: bool = True):
    from autoregressive.models.generate import generate
    import autoregressive.models.generate as G
    m = build_ref_gpt(spec, seed, dtype)
    N = (H // 16) * (W // 16)
    if spec.model_type == "t2i":
        cond, masks = text_inputs(spec.cls_token_num, spec.caption_dim, B, seed + 1, dtype)
    else:
        cond = class_inputs(spec.num_classes, B, seed + 1)
        masks = None
    cmap = control_map(B, H, W, seed + 2, "canny" if spec.condition_type in ("canny", "seg") else "depth", dtype)

    # --- control encoder outputs (reference modules) ---
    feat = m.adapter(cmap)                 # [B, N, C]   dinov2_adapter.py:26-29
    ctrl_in = m.adapter_mlp(feat)          # [B, N, d]   generate.py:138

    # --- teacher-forced logits via instrumented decode: record fp32 logits the model returns ---
    rec = []
    orig_forward = m.forward

    def spy(*a, **k):
        lg, loss = orig_forward(*a, **k)
        rec.append(lg[:, -1].clone())
        return lg, loss
    m.forward = spy
    ctx = math_sdpa() if force_math else contextlib.nullcontext()
    with ctx:
      greedy = generate(m, cond, N, emb_masks=masks, cfg_scale=cfg_scale, condition=cmap, control_strength=cs,
                      temperature=1.0, top_k=0, top_p=1.0, sample_logits=False)
    m.forward = orig_forward
    raw = torch.stack(rec, dim=1)          # [B_eff, N, V] raw model logits along the greedy trajectory
    out = {"header": header(), "prefill_sdpa": "math" if force_math else "platform default", "spec": spec.__dict__, "seed": seed, "dtype": str(dtype), "B": B, "H": H, "W": W,
           "cfg_scale": cfg_scale, "control_strength": cs,
           "inputs": "oracle.inputs: text_inputs/class_inputs(seed+1), control_map(seed+2)",
           "emb_masks": masks, "adapter_out": feat, "ctrl_in": ctrl_in,
           "greedy_tokens": greedy.clone(),
           "logit_steps": list(logit_steps),
           "raw_logits": None if save_all_logits else raw[:, list(logit_steps)].clone(),
           "raw_logits_all": raw.to(dtype).clone() if save_all_logits else None,
           "raw_logits_absmax": raw.abs().amax(dim=-1),
           "raw_top2": torch.topk(raw, 2, dim=-1)[0]}
    if sampled:
        torch.manual_seed(1234)
        with (math_sdpa() if force_math else contextlib.nullcontext()):
          out["sampled_tokens"] = generate(m, cond, N, emb_masks=masks, cfg_scale=cfg_scale, condition=cmap,
                                         control_strength=cs, temperature=1.0, top_k=100, top_p=1.0,
                                         sample_logits=True).clone()
        out["sampled_seed"] = 1234
        out["sampled_top_k"] = 100
    torch.save(out, os.path.join(OUT, name + ".pt"))
    print(name, "greedy", tuple(greedy.shape), "raw", tuple(raw.shape), flush=True)


def sampler_case():
    import autoregressive.models.generate as G
    g = torch.Generator().manual_seed(7)
    logits = torch.randn(4, 1, 16384, generator=g) * 2.0
    logits[0, 0, 5] = logits[0, 0, 9] = logits[0].max() + 1.0        # exact tie at the top
    cases = []
    for (temp, k, p) in [(1.0, 2000, 1.0), (0.7, 50, 1.0), (1.0, 0, 0.9), (1.3, 1000, 0.8), (1.0, 1, 1.0)]:
        idx, probs = G.sample(logits.clone(), temperature=temp, top_k=k, top_p=p, sample_logits=False)
        cases.append({"temperature": temp, "top_k": k, "top_p": p, "probs": probs.clone(),
                      "kept": torch.isfinite(torch.log(probs)).sum(-1)})
    torch.manual_seed(99)
    idx_s, probs_s = G.sample(logits.clone(), temperature=1.0, top_k=2000, top_p=1.0, sample_logits=True)
    torch.save({"header": header(), "logits": logits, "cases": cases,
                "multinomial_seed": 99, "multinomial_idx": idx_s}, os.path.join(OUT, "sampler.pt"))
    print("sampler ok", flush=True)


def vq_case():
    from tokenizer.tokenizer_image.vq_model import VQ_models
    vq = VQ_models["VQ-16"](codebook_size=16384, codebook_embed_dim=8)
    sd = make_vq_state_dict(seed=3)
    ref = vq.state_dict()
    assert set(ref) == set(sd), set(ref) ^ set(sd)
    for k in sd:
        assert tuple(ref[k].shape) == tuple(sd[k].shape), k
    vq.load_state_dict(sd)
    vq.eval()
    g = torch.Generator().manual_seed(11)
    out = {"header": header(), "seed": 3}
    for tag, (h, w) in {"sq": (8, 8), "mr": (4, 6)}.items():
        codes = torch.randint(0, 16384, (2, h * w), generator=g)
        img = vq.decode_code(codes, [2, 8, h, w])
        out[f"codes_{tag}"] = codes
        out[f"image_{tag}"] = img.clone()
        quant, _, info = vq.encode(img.clamp(-1, 1))
        out[f"enc_idx_{tag}"] = info[2].clone()
        out[f"enc_quant_{tag}"] = quant.clone()
        # pre-quantisation latent, to measure near-ties in the arg-min
        z = vq.quant_conv(vq.encoder(img.clamp(-1, 1)))
        out[f"enc_z_{tag}"] = z.clone()
    torch.save(out, os.path.join(OUT, "vq16.pt"))
    print("vq ok", flush=True)


def dino_case():
    from autoregressive.models.dinov2_adapter import Dinov2_Adapter
    from oracle.weights import dinov2_shapes, _fill
    out = {"header": header(), "seed": 5}
    for size in ("small", "base"):
        hidden = 384 if size == "small" else 768
        sd = _fill(dinov2_shapes(hidden, prefix="model."), 5, 0.02)
        for ctype in ("canny", "depth"):
            with fake_hf_cwd(size), contextlib.redirect_stdout(io.StringIO()):
                ad = Dinov2_Adapter(adapter_size=size, condition_type=ctype)
            assert set(ad.state_dict()) == set(sd)
            ad.load_state_dict(sd)
            ad.eval()
            for dt in (torch.float32, torch.bfloat16):
                a = ad.to(dt)
                for (H, W) in ((64, 96),) if size == "base" else ((128, 128), (64, 96)):
                    x = control_map(2, H, W, 21, "canny" if ctype == "canny" else "depth", dt)
                    y = a(x)
                    key = f"{size}_{ctype}_{str(dt).split('.')[-1]}_{H}x{W}"
                    out[key + "_out"] = y.clone()
            ad.to(torch.float32)
    torch.save(out, os.path.join(OUT, "dinov2.pt"))
    print("dino ok", flush=True)


def vision_512_case():
    """VERDICT r1 item 5: the vision stages at the REAL size (512 x 512, one image): DINOv2-small features (1025-token attention),
    VQ decode_code of a 32 x 32 grid (1024-token AttnBlock, the 512^2 level-0 convolutions) and VQ encode indices with the
    reference's fp32 distances (top-2, to bound near-ties).  Images are stored as fp16 (quantisation 5e-4, far below the
    tolerance they are compared at)."""
    from tokenizer.tokenizer_image.vq_model import VQ_models
    from autoregressive.models.dinov2_adapter import Dinov2_Adapter
    from oracle.weights import dinov2_shapes, _fill
    out = {"header": header(), "vq_seed": 3, "dino_seed": 5}
    # --- DINOv2-small, canny (nearest resize) and depth (bicubic), bf16 like the sampling scripts
    sd = _fill(dinov2_shapes(384, prefix="model."), 5, 0.02)
    for ctype in ("canny", "depth"):
        with fake_hf_cwd("small"), contextlib.redirect_stdout(io.StringIO()):
            ad = Dinov2_Adapter(adapter_size="small", condition_type=ctype)
        ad.load_state_dict(sd)
        ad = ad.eval().to(torch.bfloat16)
        x = control_map(1, 512, 512, 31, ctype, torch.bfloat16)
        out[f"dino_small_{ctype}_bf16_512"] = ad(x).clone()
    # --- VQ-16 decode / encode at 32 x 32 latents
    vq = VQ_models["VQ-16"](codebook_size=16384, codebook_embed_dim=8)
    vq.load_state_dict(make_vq_state_dict(seed=3))
    vq.eval()
    g = torch.Generator().manual_seed(13)
    codes = torch.randint(0, 16384, (1, 1024), generator=g)
    img = vq.decode_code(codes, [1, 8, 32, 32])
    out["codes"] = codes
    out["image_absmax"] = img.abs().max().clone()
    out["image_fp16"] = img.to(torch.float16).clone()
    x = img.clamp(-1, 1)
    quant, _, info = vq.encode(x)
    out["enc_idx"] = info[2].to(torch.int32).clone()
    z = vq.quant_conv(vq.encoder(x))                                   # [1, 8, 32, 32] pre-quantisation latent
    out["enc_z"] = z.clone()
    # the reference's distance matrix (vq_model.py:222-233) and its top-2 per position: margin of the arg-min
    zf = torch.nn.functional.normalize(z.permute(0, 2, 3, 1).reshape(-1, 8), p=2, dim=-1)
    e = torch.nn.functional.normalize(vq.quantize.embedding.weight, p=2, dim=-1)
    d = torch.sum(zf ** 2, dim=1, keepdim=True) + torch.sum(e ** 2, dim=1) - 2 * torch.einsum("bd,dn->bn", zf, torch.einsum("n d -> d n", e))
    top2 = torch.topk(-d, 2, dim=1)
    assert torch.equal(top2.indices[:, 0].to(torch.int32), out["enc_idx"].view(-1))
    out["enc_second_idx"] = top2.indices[:, 1].to(torch.int32).clone()
    out["enc_margin"] = (top2.values[:, 0] - top2.values[:, 1]).clone()        # d(second) - d(best) >= 0
    torch.save(out, os.path.join(OUT, "vision_512.pt"))
    print("vision_512 ok", tuple(out["image_fp16"].shape), float(out["enc_margin"].min()), flush=True)


def canny_inputs():
    """Seeded uint8 (H, W, 3) test images for the Canny front-end: pure noise, blurred noise (natural-image-like edge chains that
    cross many 32 x 32 tiles) and a synthetic scene of ramps / discs at the real size."""
    import numpy as np
    rng = np.random.default_rng(7)
    out = {}
    out["noise_67x131"] = rng.integers(0, 256, (67, 131, 3), dtype=np.uint8)
    k = np.array([1, 4, 6, 4, 1], dtype=np.float64); k /= k.sum()
    def blur(a, times):
        a = a.astype(np.float64)
        for _ in range(times):
            a = np.apply_along_axis(lambda v: np.convolve(np.pad(v, 2, mode="edge"), k, mode="valid"), 0, a)
            a = np.apply_along_axis(lambda v: np.convolve(np.pad(v, 2, mode="edge"), k, mode="valid"), 1, a)
        return np.clip(np.rint(a), 0, 255).astype(np.uint8)
    out["blur_200x160"] = blur(rng.integers(0, 256, (200, 160, 3)), 3)
    yy, xx = np.mgrid[0:512, 0:512]
    scene = np.stack([(127 + 120 * np.sin(xx / (9.0 + c) + yy / (13.0 - c))) for c in range(3)], -1)
    scene += 60.0 * (((xx - 300) ** 2 + (yy - 200) ** 2) < 90 ** 2)[..., None]
    scene += rng.normal(0, 6, scene.shape)
    out["scene_512x512"] = np.clip(np.rint(scene), 0, 255).astype(np.uint8)
    out["gray_40x56"] = blur(rng.integers(0, 256, (40, 56, 1)), 1)
    return out


def canny_case():
    """cv2.Canny (the call of reference condition/canny.py:14) on the seeded images, with the reference's default thresholds and two
    other pairs -> tests/golden/canny.npz (inputs are regenerated from the seed by the tests)."""
    import cv2
    import numpy as np
    res = {"cv2_version": np.array(cv2.__version__)}
    for name, img in canny_inputs().items():
        for lo, hi in ((100, 200), (50, 150), (30.5, 90.7)):
            res[f"{name}_{lo}_{hi}"] = cv2.Canny(img if img.shape[2] == 3 else img[:, :, 0], lo, hi)
    np.savez_compressed(os.path.join(OUT, "canny.npz"), **res)
    print("canny ok", len(res) - 1, "maps, cv2", cv2.__version__, flush=True)


def hed_inputs():
    """Seeded (B, 3, H, W) float images in 0..255 for the HED front-end: a batch whose sides divide by 16 and an odd-sized one
    (max_pool2d floors: 70 x 90 -> 35 x 45 -> 17 x 22 -> 8 x 11 -> 4 x 5)."""
    g = torch.Generator().manual_seed(23)
    def img(B, H, W):
        base = torch.rand(B, 3, H // 4 + 2, W // 4 + 2, generator=g)
        up = torch.nn.functional.interpolate(base, size=(H, W), mode="bicubic", align_corners=False)
        return (up * 255 + torch.randn(B, 3, H, W, generator=g) * 4).clamp(0, 255).round()
    return {"b2_96x128": img(2, 96, 128), "b1_70x90": img(1, 70, 90)}


def hed_case():
    """The reference's HED detector (condition/hed.py: ControlNetHED_Apache2 + the arithmetic of HEDdetector.__call__, :69-84) in
    fp32 on procedural weights (oracle/weights.py:make_hed_state_dict; the pretrained checkpoint is a download) -> edge maps and the
    five projections."""
    import types
    from condition.hed import ControlNetHED_Apache2, HEDdetector
    from oracle.weights import make_hed_state_dict
    net = ControlNetHED_Apache2().float()
    net.load_state_dict(make_hed_state_dict(seed=4), strict=True)
    net.eval()
    out = {"header": header(), "seed": 4}
    fake = types.SimpleNamespace(netNetwork=net)
    with torch.no_grad():
        for name, x in hed_inputs().items():
            out[name + "_edge"] = HEDdetector.__call__(fake, x).clone()
            out[name + "_proj"] = [p.clone() for p in net(x)]
    torch.save(out, os.path.join(OUT, "hed.pt"))
    print("hed ok", {k: tuple(v.shape) for k, v in out.items() if k.endswith("_edge")},
          float(out["b2_96x128_edge"].min()), float(out["b2_96x128_edge"].max()), flush=True)


T5_SMALL = dict(d_model=256, d_kv=64, num_heads=4, d_ff=640, num_layers=3, vocab=512)


def t5_inputs():
    """Seeded (input_ids, attention_mask) batches: right-padded prompts like the T5 tokenizer produces (pad id 0), incl. a one-token
    prompt, and a 160-token one whose relative distances exceed relative_attention_max_distance = 128."""
    g = torch.Generator().manual_seed(31)
    out = {}
    for name, (B, L, lens) in {"b3_L24": (3, 24, [24, 9, 1]), "b2_L120": (2, 120, [120, 37]), "b1_L160": (1, 160, [160])}.items():
        ids = torch.randint(2, T5_SMALL["vocab"], (B, L), generator=g)
        mask = torch.zeros(B, L, dtype=torch.int64)
        for b, n in enumerate(lens):
            mask[b, :n] = 1
        out[name] = (ids * mask, mask)
    return out


def t5_case():
    """HF T5EncoderModel (the model behind the reference's language/t5.py:54,69-75) in bf16 on procedural weights, v1.1 / flan
    architecture at a small size -> last_hidden_state."""
    from transformers import T5Config, T5EncoderModel
    from oracle.weights import make_t5_state_dict
    c = T5_SMALL
    cfg = T5Config(vocab_size=c["vocab"], d_model=c["d_model"], d_kv=c["d_kv"], d_ff=c["d_ff"], num_layers=c["num_layers"], num_heads=c["num_heads"],
                   relative_attention_num_buckets=32, relative_attention_max_distance=128, feed_forward_proj="gated-gelu",
                   layer_norm_epsilon=1e-6, dropout_rate=0.0, tie_word_embeddings=False)
    model = T5EncoderModel(cfg)
    missing, unexpected = model.load_state_dict(make_t5_state_dict(**c, seed=6), strict=False)
    assert not unexpected and all("embed_tokens" in m or "shared" in m for m in missing), (missing, unexpected)
    model = model.to(torch.bfloat16).eval()
    assert cfg.dense_act_fn == "gelu_new" and cfg.is_gated_act
    out = {"header": header(), "seed": 6, "config": dict(c)}
    # the same bf16-rounded weights evaluated in fp32: the exact result both bf16 evaluations (HF's and the CUDA path's) approximate
    exact = T5EncoderModel(cfg)
    exact.load_state_dict({k: v.to(torch.bfloat16).float() for k, v in make_t5_state_dict(**c, seed=6).items()}, strict=False)
    exact.eval()
    with torch.no_grad():
        for name, (ids, mask) in t5_inputs().items():
            out[name] = model(input_ids=ids, attention_mask=mask)["last_hidden_state"].clone()
            out[name + "_fp32"] = exact(input_ids=ids, attention_mask=mask)["last_hidden_state"].to(torch.float16).clone()
    torch.save(out, os.path.join(OUT, "t5.pt"))
    print("t5 ok", {k: tuple(v.shape) for k, v in out.items() if hasattr(v, "shape") and not k.endswith("_fp32")}, float(out["b3_L24"].float().abs().mean()), flush=True)


@contextlib.contextmanager
def fake_vit_cwd(layers: int = 12):
    """vit_adapter.py:11 loads 'autoregressive/models/vit-small' relative to CWD (ViT-S/16: hidden 384, 6 heads, MLP 1536)."""
    from transformers import ViTConfig, ViTModel
    cfg = ViTConfig(hidden_size=384, num_hidden_layers=layers, num_attention_heads=6, intermediate_size=1536, patch_size=16,
                    image_size=224, qkv_bias=True, layer_norm_eps=1e-12, hidden_act="gelu")
    old = os.getcwd()
    with tempfile.TemporaryDirectory() as tmp:
        d = os.path.join(tmp, "autoregressive", "models", "vit-small")
        os.makedirs(d)
        ViTModel(cfg).save_pretrained(d)
        os.chdir(tmp)
        try:
            yield
        finally:
            os.chdir(old)


def vit_case():
    """ViT_Adapter (the control encoder of the legacy c2i class gpt.py): outputs for square and non-square inputs."""
    from autoregressive.models.vit_adapter import ViT_Adapter
    from oracle.weights import vit_shapes, _fill
    out = {"header": header(), "seed": 9, "layers": 4}
    sd = _fill(vit_shapes(384, layers=4, prefix="model."), 9, 0.02)
    with fake_vit_cwd(4), contextlib.redirect_stdout(io.StringIO()):
        ad = ViT_Adapter()
    assert set(ad.state_dict()) == set(sd), set(ad.state_dict()) ^ set(sd)
    ad.load_state_dict(sd)
    ad.eval()
    for dt in (torch.float32, torch.bfloat16):
        a = ad.to(dt)
        for (H, W) in ((224, 224), (64, 64), (64, 96)):
            x = control_map(2, H, W, 23, "canny", dt)
            with torch.no_grad():
                out[f"{str(dt).split('.')[-1]}_{H}x{W}_out"] = a(x).clone()
        ad.to(torch.float32)
    torch.save(out, os.path.join(OUT, "vit.pt"))
    print("vit ok", flush=True)


def gptpy_case():
    """The LEGACY c2i class autoregressive/models/gpt.py (ViT adapter, per-step condition_layers, no control_strength) run
    through the reference generate() with cfg_scale 1.0 (gpt.py + CFG raises TypeError, BASELINE.md §2), bf16 (gpt.py:427
    hard-casts the control tokens to bf16).  Pins the claim that its inference arithmetic equals the gpt_t2i class with
    model_type='c2i' given the same adapter_mlp output."""
    from autoregressive.models.gpt import Transformer, ModelArgs
    from autoregressive.models.generate import generate
    from oracle.weights import vit_shapes, _fill
    seed, B, H, W, dtype = 0, 2, 64, 64, torch.bfloat16
    spec = GPTSpec(**SMALL, cls_token_num=1, block_size=(H // 16) * (W // 16), model_type="c2i")
    with fake_vit_cwd(2), contextlib.redirect_stdout(io.StringIO()):
        m = Transformer(ModelArgs(dim=spec.dim, n_layer=spec.n_layer, n_head=spec.n_head, multiple_of=spec.multiple_of,
                                  vocab_size=spec.vocab_size, cls_token_num=1, block_size=spec.block_size,
                                  num_classes=spec.num_classes, model_type="c2i", condition_token_num=0, image_size=H))
    sd = make_gpt_state_dict(spec, seed, with_adapter=False)
    ref_sd = m.state_dict()
    extra = {k for k in ref_sd if k not in sd}
    assert all(k.startswith("adapter.model.") or k == "condition_norm.weight" for k in extra), extra
    assert all(k in ref_sd and tuple(ref_sd[k].shape) == tuple(v.shape) for k, v in sd.items()), "gpt.py key/shape mismatch"
    full = dict(sd)
    full.update(_fill(vit_shapes(384, layers=2, prefix="adapter.model."), seed, 0.02))
    full["condition_norm.weight"] = torch.ones(spec.dim)
    m.load_state_dict(full, strict=True)
    m = m.to(dtype).eval()
    N = spec.block_size
    cond = class_inputs(spec.num_classes, B, seed + 1)
    cmap = control_map(B, H, W, seed + 2, "canny", dtype)
    with torch.no_grad():
        feat = m.adapter(cmap)
        ctrl_in = m.adapter_mlp(feat)
    rec = []
    orig_forward = m.forward

    def spy(*a, **k):
        lg, loss = orig_forward(*a, **k)
        rec.append(lg[:, -1].clone())
        return lg, loss
    m.forward = spy
    with math_sdpa():
        greedy = generate(m, cond, N, cfg_scale=1.0, condition=cmap, temperature=1.0, top_k=0, top_p=1.0, sample_logits=False)
    m.forward = orig_forward
    raw = torch.stack(rec, dim=1)
    out = {"header": header(), "spec": spec.__dict__, "seed": seed, "dtype": str(dtype), "B": B, "H": H, "W": W, "cfg_scale": 1.0,
           "control_strength": 1.0, "class": "autoregressive/models/gpt.py Transformer (legacy c2i class), ViT layers = 2",
           "adapter_out": feat, "ctrl_in": ctrl_in, "greedy_tokens": greedy.clone(), "raw_logits_all": raw.to(dtype).clone(),
           "raw_logits_absmax": raw.abs().amax(dim=-1)}
    torch.save(out, os.path.join(OUT, "c2i_gptpy_bf16.pt"))
    print("gptpy greedy", tuple(greedy.shape), "raw", tuple(raw.shape), flush=True)


def train_case(name: str, spec: GPTSpec, B: int, H: int, W: int, autocast, use_mask: bool, valid, seed: int = 0,
               drop_prob: float = 0.5, rand_seed: int = 1):
    """SURVEY.md §8 row f1: the teacher-forced TRAINING forward (module in train mode, fp32 parameters, bf16 autocast like
    train_t2i_canny.py:166-167 / train_c2i_canny.py:200-201) + backward through the reference, dropout layers at p = 0 and the
    CFG drop decision recorded.  Stores logits, loss and a probe of every parameter gradient (oracle.train_oracle.grad_probe)."""
    from oracle.inputs import train_attn_mask, code_inputs
    from oracle.train_oracle import grad_probe
    torch.set_grad_enabled(True)
    m = build_ref_gpt(spec, seed, torch.float32, token_dropout_p=0.0, resid_dropout_p=0.0, ffn_dropout_p=0.0,
                      class_dropout_prob=drop_prob)
    m.train()
    N = (H // 16) * (W // 16)
    T = spec.cls_token_num
    if spec.model_type == "t2i":
        cond, masks = text_inputs(T, spec.caption_dim, B, seed + 1, torch.float32)
    else:
        cond, masks = class_inputs(spec.num_classes, B, seed + 1), None
    cmap = control_map(B, H, W, seed + 2, "canny" if spec.condition_type in ("canny", "seg") else "depth", torch.float32)
    z = code_inputs(spec.vocab_size, B, N, seed + 4)
    mask = train_attn_mask(masks, N) if (use_mask and masks is not None) else None
    vt = None if valid is None else torch.tensor(valid)
    seen = {}
    orig_drop = m.cls_embedding.token_drop

    def spy_drop(*a, **k):
        out = orig_drop(*a, **k)
        seen["drop_ids"] = out[1].clone()
        return out
    m.cls_embedding.token_drop = spy_drop
    hook = m.adapter.register_forward_hook(lambda mod, inp, out: (out.retain_grad(), seen.__setitem__("feat", out))[0])
    torch.manual_seed(rand_seed)
    ac = torch.autocast("cpu", dtype=autocast) if autocast is not None else contextlib.nullcontext()
    kw = {} if mask is None else {"mask": mask}
    if vt is not None:
        kw["valid"] = vt
    with ac, math_sdpa():
        logits, loss = m(cond_idx=cond, idx=z[:, :-1], targets=z, condition=cmap if autocast is None else cmap.to(autocast), **kw)
    loss.backward()
    hook.remove()
    grads = {k: grad_probe(k, p.grad) for k, p in m.named_parameters()
             if p.grad is not None and not k.startswith("adapter.model.")}
    no_grad = sorted(k for k, p in m.named_parameters() if p.grad is None)
    small = {k: p.grad.clone() for k, p in m.named_parameters()
             if p.grad is not None and (k.endswith("norm.weight") and ("layers.0." in k or k == "norm.weight"))}
    out = {"header": header(), "spec": spec.__dict__, "seed": seed, "B": B, "H": H, "W": W,
           "autocast": None if autocast is None else str(autocast), "sdpa": "math", "use_mask": bool(mask is not None),
           "valid": valid, "dropout": "token/resid/ffn p = 0; class_dropout_prob = %g, torch.manual_seed(%d)" % (drop_prob, rand_seed),
           "inputs": "oracle.inputs: text_inputs/class_inputs(seed+1), control_map(seed+2), code_inputs(seed+4), train_attn_mask",
           "drop_ids": seen["drop_ids"], "feat": seen["feat"].detach().clone(), "feat_grad": seen["feat"].grad.clone(),
           "logits": (logits.detach().to(autocast) if autocast is not None else logits.detach()).clone(),
           "loss": loss.detach().clone(), "grads": grads, "grads_full": small, "params_without_grad": no_grad}
    torch.save(out, os.path.join(OUT, name + ".pt"))
    torch.set_grad_enabled(False)
    print(name, "loss %.6f" % float(loss), "drop", seen["drop_ids"].tolist(), "grads", len(grads), flush=True)


def gptpy_train_case(n_cols: int = 512):
    """The LEGACY class gpt.py in train mode (fp32, the configuration its train_c2i_canny.py uses: cls_token_num = 1,
    condition_token_num = 0) -> the CFG drop decision, the adapter output, the loss and the logits at a fixed seeded set of
    `n_cols` vocabulary columns (all rows).  tests/test_train_oracle_golden.py pins oracle/train_oracle.py against it."""
    from autoregressive.models.gpt import Transformer, ModelArgs
    from oracle.weights import vit_shapes, _fill
    from oracle.inputs import code_inputs
    seed, B, H, W = 0, 4, 64, 64
    spec = GPTSpec(**SMALL, cls_token_num=1, block_size=(H // 16) * (W // 16), model_type="c2i")
    with fake_vit_cwd(2), contextlib.redirect_stdout(io.StringIO()):
        m = Transformer(ModelArgs(dim=spec.dim, n_layer=spec.n_layer, n_head=spec.n_head, multiple_of=spec.multiple_of,
                                  vocab_size=spec.vocab_size, cls_token_num=1, block_size=spec.block_size, num_classes=spec.num_classes,
                                  model_type="c2i", condition_token_num=0, image_size=H, token_dropout_p=0.0, resid_dropout_p=0.0,
                                  ffn_dropout_p=0.0, class_dropout_prob=0.5))
    full = make_gpt_state_dict(spec, seed, with_adapter=False)
    full.update(_fill(vit_shapes(384, layers=2, prefix="adapter.model."), seed, 0.02))
    full["condition_norm.weight"] = torch.ones(spec.dim)
    m.load_state_dict(full, strict=True)
    m = m.float().train()
    cond = class_inputs(spec.num_classes, B, seed + 1)
    cmap = control_map(B, H, W, seed + 2, "canny", torch.float32)
    z = code_inputs(spec.vocab_size, B, spec.block_size, seed + 4)
    seen = {}
    orig_drop = m.cls_embedding.token_drop

    def spy_drop(*a, **k):
        out = orig_drop(*a, **k)
        seen["drop_ids"] = out[1].clone()
        return out
    m.cls_embedding.token_drop = spy_drop
    hook = m.adapter.register_forward_hook(lambda mod, inp, out: seen.__setitem__("feat", out.detach().clone()))
    torch.manual_seed(1)
    with math_sdpa():
        logits, loss = m(cond_idx=cond, idx=z[:, :-1], targets=z, condition=cmap)
    hook.remove()
    cols = torch.randperm(spec.vocab_size, generator=torch.Generator().manual_seed(seed + 13))[:n_cols].sort().values
    out = {"header": header(), "spec": spec.__dict__, "seed": seed, "B": B, "H": H, "W": W, "sdpa": "math",
           "class": "autoregressive/models/gpt.py Transformer (legacy c2i class), ViT layers = 2, train mode, fp32",
           "dropout": "token/resid/ffn p = 0; class_dropout_prob = 0.5, torch.manual_seed(1)",
           "inputs": "oracle.inputs: class_inputs(seed+1), control_map(seed+2), code_inputs(seed+4)",
           "drop_ids": seen["drop_ids"], "feat": seen["feat"], "loss": loss.detach().clone(),
           "logits_shape": tuple(logits.shape), "cols": cols, "logits_cols": logits.detach()[..., cols].float().clone()}
    torch.save(out, os.path.join(OUT, "train_c2i_gptpy_fp32.pt"))
    print("gptpy train loss %.6f" % float(loss), "drop", seen["drop_ids"].tolist(), "feat", tuple(seen["feat"].shape), flush=True)


def reference_surface_case():
    """The parts of the reference's public surface the drop-in must reproduce: ModelArgs fields and defaults, the parameter
    lists of generate() / the sampling helpers / Transformer.forward, and the .py files of the packages the drop-in tree is put
    in front of (none of them has an __init__.py: all are namespace packages) -> reference_surface.json."""
    import dataclasses
    import inspect
    import json
    import autoregressive.models.gpt_t2i as t2i
    import autoregressive.models.gpt as gpt
    import autoregressive.models.generate as gen

    def params(fn):
        return list(inspect.signature(fn).parameters)
    tree = []
    for d in ("autoregressive", "autoregressive/models", "autoregressive/serve", "tokenizer", "tokenizer/tokenizer_image",
              "condition", "utils", "dataset"):
        tree += sorted(f"{d}/{f}" for f in os.listdir(os.path.join(REF, d)) if f.endswith(".py"))
    out = {"generator": "tests/golden/make_golden.py reference_surface",
           "model_args": {name: {f.name: f.default for f in dataclasses.fields(mod.ModelArgs)}
                          for name, mod in (("gpt_t2i", t2i), ("gpt", gpt))},
           "signatures": {"generate": params(gen.generate), "sample": params(gen.sample),
                          "top_k_top_p_filtering": params(gen.top_k_top_p_filtering), "logits_to_probs": params(gen.logits_to_probs),
                          "gpt_t2i.Transformer.forward": params(t2i.Transformer.forward),
                          "gpt.Transformer.forward": params(gpt.Transformer.forward)},
           "tree": tree}
    with open(os.path.join(OUT, "reference_surface.json"), "w") as fh:
        json.dump(out, fh, indent=1)
        fh.write("\n")
    print("reference surface ok", len(tree), "files", flush=True)


XL = dict(dim=1280, n_layer=36, n_head=20, vocab_size=16384)


def xl_forced_case(name: str, B: int, n_tokens: int, full_steps, col_stride_after: int = 8, seed: int = 0,
                   cfg_scale: float = 4.0, cs: float = 0.6, threads: int = 0):
    """VERDICT r1 item 1: the reference's generate() at GPT-XL shape (dim 1280 / H 20 / F 3584 / V 16384 / L 36, block_size 1024,
    T 120) in bf16 with CFG, left-padded masks and control_strength != 1, TEACHER-FORCED along a fixed random token grid:
    generate.py's `sample` is replaced by a function that returns the forced token, every other line of generate()/prefill/
    decode_one_token/Transformer.forward runs unmodified.  Stored (bf16-exact, the reference's logits are bf16 values):
    full logits rows at `full_steps`, a 256-column probe at every step < 64 and every `col_stride_after`-th step after, and per
    step the CFG-combined arg-max + top-2 margin + |logit| max."""
    import autoregressive.models.generate as G
    if threads:
        torch.set_num_threads(threads)
    dtype = torch.bfloat16
    spec = GPTSpec(**XL, cls_token_num=120, block_size=1024, model_type="t2i")
    m = build_ref_gpt(spec, seed, dtype)
    m.adapter = torch.nn.Identity()          # generate.py:137-138 then pass the procedural control tokens through
    m.adapter_mlp = torch.nn.Identity()
    N_img = 1024
    cond, masks = text_inputs(spec.cls_token_num, spec.caption_dim, B, seed + 1, dtype)
    ctrl_in = xl_ctrl_in(B, N_img, spec.dim, seed + 7, dtype)
    g = torch.Generator().manual_seed(seed + 11)
    forced = torch.randint(0, spec.vocab_size, (B, n_tokens), generator=g, dtype=torch.int64)
    cols = torch.randperm(spec.vocab_size, generator=g)[:256].sort().values
    full_steps = [s for s in full_steps if s < n_tokens]
    col_steps = [s for s in range(n_tokens) if s < 64 or s % col_stride_after == 0 or s == n_tokens - 1]
    rec = {"full": {}, "cols": {}, "argmax": [], "margin": [], "absmax": []}
    state = {"i": 0}
    orig_forward = m.forward

    def spy(*a, **k):
        lg, loss = orig_forward(*a, **k)
        raw = lg[:, -1].float()                       # [B_eff, V] fp32 carrier of bf16 values (gpt_t2i.py:470)
        i = state["i"]
        if i in full_steps:
            rec["full"][i] = raw.to(dtype).clone()
        if i in col_steps:
            rec["cols"][i] = raw[:, cols].to(dtype).clone()
        c, u = raw[:B], raw[B:]
        z = u + (c - u) * cfg_scale
        t2 = torch.topk(z, 2, dim=-1)
        rec["argmax"].append(t2.indices[:, 0].clone())
        rec["margin"].append((t2.values[:, 0] - t2.values[:, 1]).clone())
        rec["absmax"].append(raw.abs().max().clone())
        return lg, loss

    def forced_sample(logits, **kw):
        i = state["i"]
        state["i"] = i + 1
        if i % 32 == 0:
            print(f"  {name}: step {i}/{n_tokens}", flush=True)
        return forced[:, i:i + 1].clone(), torch.zeros(1)

    m.forward = spy
    orig_sample = G.sample
    G.sample = forced_sample
    try:
        with math_sdpa():
            out_tokens = G.generate(m, cond, n_tokens, emb_masks=masks, cfg_scale=cfg_scale, condition=ctrl_in,
                                    control_strength=cs, temperature=1.0, top_k=0, top_p=1.0, sample_logits=False)
    finally:
        G.sample = orig_sample
        m.forward = orig_forward
    assert torch.equal(out_tokens.long(), forced)
    out = {"header": header(), "spec": spec.__dict__, "seed": seed, "dtype": str(dtype), "B": B, "n_tokens": n_tokens,
           "N_img": N_img, "cfg_scale": cfg_scale, "control_strength": cs, "prefill_sdpa": "math",
           "inputs": "oracle.inputs.text_inputs(seed+1); ctrl_in = randn(B,1024,1280, seed+7)*0.5 (bf16) fed as adapter_mlp output; "
                     "forced tokens randint(seed+11)",
           "emb_masks": masks, "forced_tokens": forced.to(torch.int32), "cols": cols,
           "full_steps": full_steps, "full_logits": torch.stack([rec["full"][s] for s in full_steps], dim=1),
           "col_steps": col_steps, "col_logits": torch.stack([rec["cols"][s] for s in col_steps], dim=1),
           "argmax_cfg": torch.stack(rec["argmax"], dim=1).to(torch.int32), "margin_cfg": torch.stack(rec["margin"], dim=1),
           "raw_absmax": torch.stack(rec["absmax"])}
    torch.save(out, os.path.join(OUT, name + ".pt"))
    print(name, "done", tuple(out["full_logits"].shape), tuple(out["col_logits"].shape), flush=True)


SMALL = dict(dim=256, n_layer=6, n_head=4, vocab_size=2048)

CASES = {
    "t2i_small_bf16": lambda: ar_case("t2i_small_bf16", GPTSpec(**SMALL, cls_token_num=120, block_size=64,
                                                                model_type="t2i"),
                                      B=2, H=128, W=128, cfg_scale=4.0, cs=0.6, dtype=torch.bfloat16),
    "t2i_small_fp32": lambda: ar_case("t2i_small_fp32", GPTSpec(**SMALL, cls_token_num=120, block_size=64,
                                                                model_type="t2i"),
                                      B=2, H=128, W=128, cfg_scale=4.0, cs=0.6, dtype=torch.float32),
    "t2i_mr_bf16": lambda: ar_case("t2i_mr_bf16", GPTSpec(**SMALL, cls_token_num=120, block_size=144,
                                                          model_type="t2i", condition_type="depth"),
                                   B=1, H=128, W=192, cfg_scale=4.0, cs=1.0, dtype=torch.bfloat16),
    "t2i_mr_tall_bf16": lambda: ar_case("t2i_mr_tall_bf16", GPTSpec(**SMALL, cls_token_num=120, block_size=144,
                                                                    model_type="t2i", condition_type="depth"),
                                        B=1, H=192, W=128, cfg_scale=1.0, cs=1.0, dtype=torch.bfloat16,
                                        sampled=False),
    "c2i_small_bf16": lambda: ar_case("c2i_small_bf16", GPTSpec(**SMALL, cls_token_num=1, block_size=64,
                                                                model_type="c2i"),
                                      B=2, H=128, W=128, cfg_scale=4.0, cs=1.0, dtype=torch.bfloat16),
    "c2i_small_fp32": lambda: ar_case("c2i_small_fp32", GPTSpec(**SMALL, cls_token_num=1, block_size=64,
                                                                model_type="c2i"),
                                      B=2, H=128, W=128, cfg_scale=1.0, cs=1.0, dtype=torch.float32,
                                      sampled=False),
    "t2i_B_bf16": lambda: ar_case("t2i_B_bf16", GPTSpec(dim=768, n_layer=12, n_head=12, vocab_size=16384,
                                                        cls_token_num=120, block_size=64, model_type="t2i"),
                                  B=1, H=128, W=128, cfg_scale=4.0, cs=1.0, dtype=torch.bfloat16,
                                  logit_steps=(0, 5), sampled=False, save_all_logits=False),
    "t2i_small_bf16_defaultsdpa": lambda: ar_case("t2i_small_bf16_defaultsdpa",
                                                  GPTSpec(**SMALL, cls_token_num=120, block_size=64, model_type="t2i"),
                                                  B=2, H=128, W=128, cfg_scale=4.0, cs=0.6, dtype=torch.bfloat16,
                                                  sampled=False, save_all_logits=False, force_math=False),
    "sampler": sampler_case,
    "vq16": vq_case,
    "dinov2": dino_case,
    "vit": vit_case,
    "vision_512": vision_512_case,
    "canny": canny_case,
    "hed": hed_case,
    "t5": t5_case,
    "c2i_gptpy_bf16": gptpy_case,
    "train_c2i_gptpy_fp32": gptpy_train_case,
    "reference_surface": reference_surface_case,
    "train_t2i_small_ac": lambda: train_case("train_t2i_small_ac", GPTSpec(**SMALL, cls_token_num=120, block_size=64, model_type="t2i"),
                                             B=3, H=128, W=128, autocast=torch.bfloat16, use_mask=True, valid=[1, 0, 1]),
    "train_t2i_small_fp32": lambda: train_case("train_t2i_small_fp32", GPTSpec(**SMALL, cls_token_num=120, block_size=64, model_type="t2i"),
                                               B=3, H=128, W=128, autocast=None, use_mask=True, valid=[1, 1, 1]),
    "train_c2i_small_ac": lambda: train_case("train_c2i_small_ac", GPTSpec(**SMALL, cls_token_num=1, block_size=64, model_type="c2i"),
                                             B=4, H=128, W=128, autocast=torch.bfloat16, use_mask=False, valid=None),
    "xl_b1_long": lambda: xl_forced_case("xl_b1_long", B=1, n_tokens=1024, full_steps=(0, 1, 2, 391, 392, 777, 1022, 1023)),
    "xl_b8_short": lambda: xl_forced_case("xl_b8_short", B=8, n_tokens=49, full_steps=(0, 1, 2, 7, 23, 48)),
    "xl_b8_long": lambda: xl_forced_case("xl_b8_long", B=8, n_tokens=1024, full_steps=(0, 1, 65, 391, 1023)),
    "train_t2i_mr_ac": lambda: train_case("train_t2i_mr_ac", GPTSpec(**SMALL, cls_token_num=120, block_size=144, model_type="t2i",
                                                                     condition_type="depth"),
                                          B=2, H=128, W=192, autocast=torch.bfloat16, use_mask=True, valid=[1, 1]),
}

if __name__ == "__main__":
    todo = sys.argv[1:] or [c for c in CASES if not c.startswith('xl_')]   # XL cases: minutes to ~40 min of CPU, on request
    for c in todo:
        CASES[c]()
