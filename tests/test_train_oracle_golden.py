"""CPU: oracle/train_oracle.py (SURVEY.md §8 row f1, the teacher-forced training forward + loss, gradients by autograd over the
restatement) against fixtures produced by the reference itself in train mode (tests/golden/make_golden.py::train_case).
This pins the checker the round-2 CUDA training path will be compared with; no product code is involved."""
import pytest
import torch

from oracle.weights import GPTSpec, make_gpt_state_dict
from oracle.train_oracle import TrainOracle, grad_probe
from oracle.inputs import text_inputs, class_inputs, train_attn_mask, code_inputs
from tests.helpers import load_golden, rel_l2

CASES = ["train_t2i_small_ac", "train_t2i_small_fp32", "train_c2i_small_ac", "train_t2i_mr_ac"]


def _run(g):
    spec = GPTSpec(**g["spec"])
    ac = {None: None, "torch.bfloat16": torch.bfloat16}[g["autocast"]]
    orc = TrainOracle(spec, make_gpt_state_dict(spec, g["seed"]), ac)
    B, N = g["B"], (g["H"] // 16) * (g["W"] // 16)
    if spec.model_type == "t2i":
        cond, masks = text_inputs(spec.cls_token_num, spec.caption_dim, B, g["seed"] + 1, torch.float32)
    else:
        cond, masks = class_inputs(spec.num_classes, B, g["seed"] + 1), None
    z = code_inputs(spec.vocab_size, B, N, g["seed"] + 4)
    mask = train_attn_mask(masks, N) if g["use_mask"] else None
    valid = None if g["valid"] is None else torch.tensor(g["valid"])
    feat = g["feat"].clone().requires_grad_(True)
    with torch.enable_grad():
        logits, loss = orc.forward(z[:, :-1], cond, feat, g["drop_ids"], mask, z, valid)
        loss.backward()
    return orc, feat, logits.detach(), loss.detach()


@pytest.mark.parametrize("name", CASES)
def test_train_forward_loss_and_logits(name):
    g = load_golden(name)
    assert g["drop_ids"].any() and not g["drop_ids"].all(), "fixture must mix dropped and kept samples"
    orc, feat, logits, loss = _run(g)
    ref = g["logits"].float()
    assert logits.shape == ref.shape and logits.dtype == torch.float32
    if g["autocast"] is None:
        assert rel_l2(logits, ref) < 2e-6
        assert abs(float(loss) - float(g["loss"])) < 2e-6 * float(g["loss"])
    else:
        # bf16 autocast: same casts at the same places -> differences are single bf16 roundings of near-identical fp32 values
        assert rel_l2(logits, ref) < 4e-3
        assert (logits - ref).abs().max() <= 2.0 ** -7 * ref.abs().max()
        assert abs(float(loss) - float(g["loss"])) < 2e-5 * float(g["loss"])


@pytest.mark.parametrize("name", CASES)
def test_train_gradients(name):
    """Every parameter the reference gives a gradient gets the same one from the restatement (norm + 256 probed entries per
    tensor, the first block's norm weights in full), and so does the control-encoder output (the hand-over to its backward)."""
    g = load_golden(name)
    orc, feat, _, _ = _run(g)
    tol_n, tol_v = (1e-5, 2e-5) if g["autocast"] is None else (5e-3, 3e-2)   # measured: 2e-7 / 1e-6 and 9e-4 / 8e-3
    ref_keys = set(g["grads"])
    mine = {k for k, p in orc.p.items() if p.grad is not None}
    assert mine == ref_keys, (sorted(mine ^ ref_keys))
    assert set(g["params_without_grad"]) >= {"condition_embeddings.weight"}
    for k in sorted(ref_keys):
        pr = g["grads"][k]
        pm = grad_probe(k, orc.p[k].grad)
        assert torch.equal(pm["pos"], pr["pos"])
        nr = float(pr["norm"])
        assert abs(float(pm["norm"]) - nr) <= tol_n * nr + 1e-12, (k, float(pm["norm"]), nr)
        scale = nr / max(orc.p[k].numel(), 1) ** 0.5           # RMS of the gradient tensor
        assert float((pm["val"] - pr["val"]).norm()) <= tol_v * (float(pr["val"].norm()) + scale * 16), k
    for k, full in g["grads_full"].items():
        assert rel_l2(orc.p[k].grad, full) < tol_v, k
    assert rel_l2(feat.grad, g["feat_grad"]) < tol_v


def test_train_mask_and_valid_semantics():
    """Properties the CUDA path must keep: a sample with valid = 0 contributes nothing (loss and gradients), and the padded
    text columns are never attended (changing the padded caption rows changes nothing)."""
    g = load_golden("train_t2i_small_ac")
    spec = GPTSpec(**g["spec"])
    sd = make_gpt_state_dict(spec, g["seed"])
    B, N = g["B"], 64
    cond, masks = text_inputs(spec.cls_token_num, spec.caption_dim, B, g["seed"] + 1, torch.float32)
    z = code_inputs(spec.vocab_size, B, N, g["seed"] + 4)
    mask = train_attn_mask(masks, N)
    valid = torch.tensor(g["valid"])
    assert int(valid[1]) == 0
    drop = torch.zeros(B, dtype=torch.bool)

    def run(cond_, z_):
        o = TrainOracle(spec, sd, torch.bfloat16)
        with torch.enable_grad():
            lg, loss = o.forward(z_[:, :-1], cond_, g["feat"], drop, mask, z_, valid)
            loss.backward()
        return lg.detach(), float(loss.detach()), o.p["layers.0.attention.wqkv.weight"].grad.clone()
    lg0, l0, g0 = run(cond, z)
    z2 = z.clone(); z2[1] = (z2[1] + 7) % spec.vocab_size           # only the invalid sample changes
    lg1, l1, g1 = run(cond, z2)
    assert l0 == l1 and torch.equal(g0, g1) and torch.equal(lg0[0], lg1[0]) and torch.equal(lg0[2], lg1[2])
    cond3 = cond.clone()
    cond3[masks == 0] = 5.0                                           # garbage in the padded caption rows
    lg2, l2, _ = run(cond3, z)
    # image-token rows never see padded columns; their logits are unchanged
    assert torch.equal(lg0, lg2) and l0 == l2


@pytest.mark.parametrize("shape", [(64, 96, 48, 80), (50, 70, 64, 64), (96, 96, 24, 40), (33, 47, 33, 100), (128, 128, 96, 160)])
def test_resize_oracle_matches_torch(shape):
    """Row f2 checker: oracle/resize_oracle.py against the call the reference makes (train_t2i_depth_multiscale.py:52-54),
    `F.interpolate(..., mode='bilinear', align_corners=False, antialias=True)`, on 0..255 image data; fp32 summation-order noise only."""
    import torch.nn.functional as F
    from oracle.resize_oracle import bilinear_aa_resize
    h, w, oh, ow = shape
    x = torch.rand(2, 3, h, w, generator=torch.Generator().manual_seed(h * 1000 + w)) * 255
    ref = F.interpolate(x, size=(oh, ow), mode="bilinear", align_corners=False, antialias=True)
    got = bilinear_aa_resize(x, (oh, ow))
    assert got.shape == ref.shape
    assert float((got - ref).abs().max()) < 1e-4           # 4e-7 of full scale


def test_legacy_gptpy_train_branch_is_the_same_arithmetic():
    """The LEGACY class autoregressive/models/gpt.py (imported by train_c2i_canny.py) has its own copy of the training branch
    (gpt.py:410-421,440-449).  With the only configuration its scripts use (cls_token_num = 1, condition_token_num = 0) it is the
    gpt_t2i branch: control tokens added to every row, logits from row 0 on.  Pinned here by running the reference's gpt.py in
    train mode (fp32) against the oracle on the same weights — which is why controlar_b200's gpt.py shell inherits the training
    forward / backward of gpt_t2i unchanged.  The reference's side (its CFG drop decision, adapter output, loss and logits at 512
    seeded vocabulary columns) is stored by tests/golden/make_golden.py::gptpy_train_case."""
    g = load_golden("train_c2i_gptpy_fp32")
    spec = GPTSpec(**g["spec"])
    seed, B = g["seed"], g["B"]
    sd = make_gpt_state_dict(spec, seed, with_adapter=False)
    cond = class_inputs(spec.num_classes, B, seed + 1)
    z = code_inputs(spec.vocab_size, B, spec.block_size, seed + 4)
    drop_ids, feat, cols, logits, loss = g["drop_ids"], g["feat"], g["cols"], g["logits_cols"], g["loss"]
    assert drop_ids.any() and not drop_ids.all()
    # one difference: gpt.py's ConditionEmbedder.token_drop gives dropped samples literal zeros (gpt.py:118-119), gpt_t2i's gives
    # them the `uncond_embedding` buffer (gpt_t2i.py:120) — identical for released checkpoints (the buffer is zero), not for the
    # procedural weights used here.  controlar_b200's gpt.py shell therefore passes no buffer (cond_uncond = NULL => zeros).
    sd0 = dict(sd)
    sd0["condition_mlp.uncond_embedding"] = torch.zeros_like(sd["condition_mlp.uncond_embedding"])
    orc = TrainOracle(spec, sd0, None)
    with torch.no_grad():
        lo, ls = orc.forward(z[:, :-1], cond, feat, drop_ids, None, z, None)
        lb, _ = TrainOracle(spec, sd, None).forward(z[:, :-1], cond, feat, drop_ids, None, z, None)
    assert tuple(lo.shape) == tuple(g["logits_shape"])
    assert rel_l2(lo[..., cols], logits) < 5e-6
    assert abs(float(ls) - float(loss)) < 5e-6 * float(loss)
    assert rel_l2(lb[..., cols], logits) > 1e-3       # with the buffer's rows instead of zeros the result is visibly different
