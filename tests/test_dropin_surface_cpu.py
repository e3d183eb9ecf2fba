"""CPU: the drop-in surface (SURVEY.md §8b) — constructor fields, function signatures, registry keys and state-dict keys of
the product shells against the reference.  The state-dict key sets come from oracle/weights.py, which
tests/golden/make_golden.py asserts equal to the reference modules' own ``state_dict()``; the dataclass fields and signatures
are compared with the reference's as recorded from its source by make_golden.py (tests/golden/reference_surface.json)."""
import dataclasses
import inspect
import json
import os

import torch

from oracle.weights import GPTSpec, gpt_shapes, vit_shapes, vq_shapes

with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_surface.json")) as _fh:
    REF = json.load(_fh)


def test_state_dict_keys_t2i_and_c2i():
    from controlar_b200.autoregressive.models.gpt_t2i import Transformer, ModelArgs
    for spec in (GPTSpec(dim=256, n_layer=6, n_head=4, vocab_size=2048, cls_token_num=120, block_size=64, model_type="t2i"),
                 GPTSpec(dim=256, n_layer=6, n_head=4, vocab_size=2048, cls_token_num=1, block_size=64, model_type="c2i",
                         adapter_size="base")):
        m = Transformer(ModelArgs(dim=spec.dim, n_layer=spec.n_layer, n_head=spec.n_head, vocab_size=spec.vocab_size,
                                  cls_token_num=spec.cls_token_num, block_size=spec.block_size, model_type=spec.model_type,
                                  adapter_size=spec.adapter_size))
        want = gpt_shapes(spec)
        got = {k: tuple(v.shape) for k, v in m.state_dict().items()}
        assert got == want


def test_state_dict_keys_legacy_gpt_and_vq():
    from controlar_b200.autoregressive.models.gpt import Transformer, ModelArgs
    from controlar_b200.tokenizer.tokenizer_image.vq_model import VQ_models
    spec = GPTSpec(dim=256, n_layer=6, n_head=4, vocab_size=2048, cls_token_num=1, block_size=16, model_type="c2i")
    m = Transformer(ModelArgs(dim=256, n_layer=6, n_head=4, vocab_size=2048, cls_token_num=1, block_size=16, model_type="c2i",
                              condition_token_num=0, image_size=64))
    want = gpt_shapes(spec, with_adapter=False)
    want.update(vit_shapes(384, layers=12, prefix="adapter.model."))
    want["condition_norm.weight"] = (256,)
    assert {k: tuple(v.shape) for k, v in m.state_dict().items()} == want
    vq = VQ_models["VQ-16"](codebook_size=16384, codebook_embed_dim=8)
    assert {k: tuple(v.shape) for k, v in vq.state_dict().items()} == vq_shapes()


def test_model_registries_and_public_attributes():
    from controlar_b200.autoregressive.models import gpt_t2i, gpt
    names = {"GPT-B", "GPT-L", "GPT-XL", "GPT-XXL", "GPT-XXXL", "GPT-1B", "GPT-3B", "GPT-7B"}
    assert set(gpt_t2i.GPT_models) == names and set(gpt.GPT_models) == names
    m = gpt_t2i.GPT_models["GPT-B"](vocab_size=64, block_size=16, cls_token_num=120, model_type="t2i")
    for attr in ("adapter", "adapter_mlp", "model_type", "num_classes", "cls_embedding", "tok_embeddings", "setup_caches",
                 "forward", "get_fsdp_wrap_module_list", "layers", "output", "norm", "freqs_cis"):
        assert hasattr(m, attr), attr
    assert m.cls_embedding.uncond_embedding.shape == (120, 2048)
    assert len(m.get_fsdp_wrap_module_list()) == 12


def test_model_args_fields_match_reference():
    ours_t2i = {f.name: f.default for f in dataclasses.fields(__import__(
        "controlar_b200.autoregressive.models.gpt_t2i", fromlist=["ModelArgs"]).ModelArgs)}
    ours_gpt = {f.name: f.default for f in dataclasses.fields(__import__(
        "controlar_b200.autoregressive.models.gpt", fromlist=["ModelArgs"]).ModelArgs)}
    assert ours_t2i == REF["model_args"]["gpt_t2i"]
    assert ours_gpt == REF["model_args"]["gpt"]


def test_generate_and_forward_signatures_cover_the_reference():
    from controlar_b200.autoregressive.models import generate as og, gpt_t2i as ot, gpt as ol
    sig = REF["signatures"]
    ref_params = sig["generate"]
    our_params = list(inspect.signature(og.generate).parameters)
    assert [p for p in our_params if p in ref_params] == ref_params                       # same names, same order
    assert set(our_params) - set(ref_params) <= {"noise", "seed"}                         # keyword-only extras
    for name in ("sample", "top_k_top_p_filtering", "logits_to_probs"):
        rp, op = sig[name], inspect.signature(getattr(og, name)).parameters
        assert list(rp)[:2] == list(op)[:2], name
    rf = sig["gpt_t2i.Transformer.forward"]
    assert list(inspect.signature(ot.Transformer.forward).parameters) == rf
    rl = sig["gpt.Transformer.forward"]
    assert list(inspect.signature(ol.Transformer.forward).parameters)[:len(rl)] == rl     # + control_strength (must stay 1)


def test_modules_with_live_library_handles_can_be_deep_copied():
    """`ema = deepcopy(model)` (train_c2i_canny.py:117) and `torch.save(model)` must work after the model has been used: library
    handles are dropped from the copy (which rebuilds them lazily) instead of failing in ctypes' pickling."""
    import copy
    import ctypes as C
    import pickle
    from controlar_b200 import engine, vision
    from controlar_b200.autoregressive.models.gpt_t2i import Transformer, ModelArgs

    def fake(cls):
        class F(cls):
            def __init__(self):
                self.handle = C.c_void_p(0)            # null: close() / __del__ have nothing to destroy

            def close(self):
                pass
        return F()
    m = Transformer(ModelArgs(dim=128, n_layer=3, n_head=2, vocab_size=64, cls_token_num=1, block_size=16, num_classes=10, model_type="c2i"))
    m._car_model, m._car_state, m._car_train = fake(engine.ARModelHandle), fake(engine.ARStateHandle), fake(engine.ARTrainHandle)
    object.__setattr__(m.adapter, "_car_dino", fake(vision.DinoHandle))
    for clone in (copy.deepcopy(m), pickle.loads(pickle.dumps(m))):
        assert clone._car_model is None and clone._car_state is None and clone._car_train is None and clone.adapter._car_dino is None
        assert all(torch.equal(a, b) for a, b in zip(m.state_dict().values(), clone.state_dict().values()))
    assert m._car_model is not None                    # the original keeps its handles
