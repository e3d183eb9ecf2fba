"""Row b (drop-in boundary): the PYTHONPATH configuration INTEGRATION.md documents must make the reference's own import lines
(autoregressive/sample/sample_t2i.py:15-19, sample_c2i.py:19) resolve to this repository's modules — checked in a fresh interpreter,
from a foreign working directory.  Behind it, the modules this repository does NOT replace must still resolve to the reference
tree: checked against a stand-in tree with the reference's package layout (tests/golden/reference_surface.json)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

CODE = r"""
import os, sys
from tokenizer.tokenizer_image.vq_model import VQ_models            # sample_t2i.py:15
from autoregressive.models.gpt_t2i import GPT_models                # sample_t2i.py:17-18
from autoregressive.models.generate import generate                 # sample_t2i.py:19
from autoregressive.models.gpt import GPT_models as GPT_models_c2i  # sample_c2i.py:19
import autoregressive.models.gpt_t2i as m, autoregressive.models.generate as g, tokenizer.tokenizer_image.vq_model as v
import autoregressive.models.dinov2_adapter as da, autoregressive.models.vit_adapter as va
root = sys.argv[1]
for mod in (m, g, v, da, va):
    assert mod.__file__.startswith(os.path.join(root, "dropin")), mod.__file__
import controlar_b200.autoregressive.models.gpt_t2i as impl
assert GPT_models is impl.GPT_models and m.Transformer is impl.Transformer and m.ModelArgs is impl.ModelArgs
assert callable(generate) and "VQ-16" in VQ_models and "GPT-XL" in GPT_models and "GPT-B" in GPT_models_c2i
assert callable(g.sample) and callable(g.top_k_top_p_filtering) and callable(m.precompute_freqs_cis_2d) and callable(m.find_multiple)
if len(sys.argv) > 2:
    import utils.drop_path as dp, dataset.augmentation as aug
    assert dp.__file__.startswith(sys.argv[2]) and aug.__file__.startswith(sys.argv[2]), (dp.__file__, aug.__file__)
print("OK")
"""


def _run(extra_path, extra_args, tmp_path):
    env = dict(os.environ)
    env["PYTHONPATH"] = os.pathsep.join([os.path.join(ROOT, "dropin"), ROOT] + extra_path)
    r = subprocess.run([sys.executable, "-c", CODE, ROOT] + extra_args, cwd=str(tmp_path), env=env, capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0 and r.stdout.strip().endswith("OK"), r.stdout + r.stderr


def test_dropin_imports_resolve_to_this_repo(tmp_path):
    _run([], [], tmp_path)


def _reference_tree(dst):
    """Placeholder modules at the reference's .py paths, without __init__.py files like the reference: which directory a module
    resolves from depends only on that layout."""
    with open(os.path.join(ROOT, "tests", "golden", "reference_surface.json")) as fh:
        files = json.load(fh)["tree"]
    for rel in files:
        path = os.path.join(dst, *rel.split("/"))
        os.makedirs(os.path.dirname(path), exist_ok=True)
        with open(path, "w") as fh:
            fh.write(f'"""Stand-in for the reference\'s {rel}."""\n')
    return str(dst)


def test_dropin_in_front_of_the_reference_tree(tmp_path):
    ref = _reference_tree(tmp_path / "reference")
    work = tmp_path / "work"
    work.mkdir()
    _run([ref], [ref], work)
