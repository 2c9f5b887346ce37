"""The drop-in boundary, proven with the reference's own call sequence (SURVEY.md section 8b).

CPU part (this file, ``-m "not gpu"``): every test runs in a fresh interpreter, because ``install()``
edits ``sys.modules``.
  * stand-alone install (no reference on sys.path): the two submodule names resolve to the mirror;
  * next to a package tree laid out like the reference's (its ``generators`` / ``siren`` packages, the
    modules of them that the rest of the reference imports, a ``curriculums`` naming the classes of its
    three curricula): after ``install()`` ``curriculums`` imports (curriculums.py:1 needs the reference's
    own ``generators.neural_rendering``), the reference-only submodules stay reachable, and the train
    script's class lookups (train_double_latent_semantic.py:20-22, 116, 142) find the mirror classes;
  * a generator built from the REFERENCE classes and saved with ``torch.save(generator)``
    (train_double_latent_semantic.py:128-150 / render_multiview_images_double_semantic.py:58; stored by
    ``tests/golden/make_goldens.py --pickles``) loads under the mirror with an identical state_dict and the
    same parameter order, so torch_ema's positional ``copy_to`` / ``restore`` (``param.data.copy_``) lands
    on the right tensors;
  * a generator saved under the mirror pickles exactly like the reference's own checkpoint: the same
    module classes by module path, attribute names and parameters.
GPU part: tests/test_gpu_parity.py::test_render_script_call_sequence replays
render_multiview_images_double_semantic.py:43-65 against a golden.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")


def _run(code, *args, timeout=600):
    env = dict(os.environ, PYTHONDONTWRITEBYTECODE="1")
    r = subprocess.run([sys.executable, "-c", code, ROOT] + list(args), capture_output=True, text=True,
                       timeout=timeout, env=env)
    assert r.returncode == 0, "child failed:\n%s\n%s" % (r.stdout[-3000:], r.stderr[-3000:])
    return r.stdout


#: the reference tree as install() meets it: its own `generators` / `siren` packages, whose two mirrored
#: submodules must never be imported once install() ran, the modules of those packages that the rest of the
#: reference imports (curriculums.py:1, prepare_segmaps.py:9, generators/networks.py:18), and a `curriculums`
#: naming the model / generator classes of the reference's three curricula (curriculums.py:66-68, 111-112, 159-160)
_REFERENCE_LAYOUT = {
    "generators/__init__.py": "",
    "generators/generators.py": "raise AssertionError('the reference module was imported instead of the mirror')\n",
    "generators/neural_rendering.py": "class NeuralRenderer:\n    pass\n",
    "generators/BiSeNet.py": "",
    "siren/__init__.py": "",
    "siren/siren.py": "raise AssertionError('the reference module was imported instead of the mirror')\n",
    "siren/op/__init__.py": "",
    "curriculums.py": ("from generators.neural_rendering import NeuralRenderer\n"
                       "CelebA = {'model': 'SPATIALSIRENBASELINE', 'generator': 'ImplicitGenerator3d'}\n"
                       "CelebA_double_semantic = {'model': 'SIRENBASELINESEMANTICDISENTANGLE', "
                       "'generator': 'DoubleImplicitGenerator3d'}\n"
                       "CelebA_double_semantic_texture_embedding_256_dim_96 = {"
                       "'model': 'TextureEmbeddingPiGAN256SEMANTICDISENTANGLE_DIM_96', "
                       "'generator': 'DoubleImplicitGenerator3d'}\n"),
}


def _reference_like_tree(tmp_path):
    root = tmp_path / "reference"
    for rel, text in _REFERENCE_LAYOUT.items():
        (root / rel).parent.mkdir(parents=True, exist_ok=True)
        (root / rel).write_text(text)
    return str(root)


def test_standalone_install_resolves_the_two_submodules():
    out = _run(r'''
import sys
sys.path.insert(0, sys.argv[1])
import fenerf_b200
g, s = fenerf_b200.install()
from generators import generators
from siren import siren
assert generators is g and siren is s
import generators.generators as gg, siren.siren as ss
assert gg is g and ss is s
cls = getattr(generators, "DoubleImplicitGenerator3d")
assert cls.__module__ == "generators.generators", cls.__module__
assert hasattr(siren, "TextureEmbeddingPiGAN256SEMANTICDISENTANGLE_DIM_96") and hasattr(siren, "TALLSIREN")
fenerf_b200.install()      # idempotent
print("ok")
''')
    assert "ok" in out


def test_install_keeps_the_reference_packages_importable(tmp_path):
    out = _run(r'''
import sys
sys.path.insert(0, sys.argv[2]); sys.path.insert(0, sys.argv[1])
import fenerf_b200
fenerf_b200.install()
import curriculums                                    # curriculums.py:1 -> generators.neural_rendering (reference's)
import generators.neural_rendering as nr
assert nr.__file__.startswith(sys.argv[2]), nr.__file__
from generators import generators                     # train_double_latent_semantic.py:20
from siren import siren                               # :22
assert generators.__name__ == "fenerf_b200.generators.generators", generators.__name__
assert siren.__name__ == "fenerf_b200.siren.siren"
import importlib.util                                 # reference-only subpackages still reachable (networks.py:18)
assert importlib.util.find_spec("siren.op") is not None and importlib.util.find_spec("generators.BiSeNet") is not None
md = curriculums.CelebA_double_semantic_texture_embedding_256_dim_96
SIREN = getattr(siren, md['model'])                   # :116
gen_cls = getattr(generators, md['generator'])        # :142
assert gen_cls.__module__ == "generators.generators" and SIREN.__module__ == "siren.siren"
md2 = curriculums.CelebA
assert hasattr(siren, md2['model']) and hasattr(generators, md2['generator'])
md3 = curriculums.CelebA_double_semantic
assert hasattr(siren, md3['model']) and hasattr(generators, md3['generator'])
print("ok", md['model'], md['generator'])
''', _reference_like_tree(tmp_path))
    assert "ok TextureEmbeddingPiGAN256SEMANTICDISENTANGLE_DIM_96 DoubleImplicitGenerator3d" in out


def _reference_checkpoint(tmp_path, model):
    """The reference's own torch.save(generator) of `model` (and its {names, state}), written to tmp_path."""
    gold = np.load(os.path.join(GOLDEN_DIR, "ref_pickle_%s.npz" % model))
    path = tmp_path / ("reference_%s.pth" % model)
    path.write_bytes(gold["checkpoint"].tobytes())
    (tmp_path / ("reference_%s.pth.meta" % model)).write_bytes(gold["meta"].tobytes())
    return str(path)


_LOAD_WITH_MIRROR = r'''
import sys
sys.path.insert(0, sys.argv[1])
import torch, fenerf_b200
fenerf_b200.install()
gen = torch.load(sys.argv[2], map_location="cpu", weights_only=False)   # render_multiview_images_double_semantic.py:58
meta = torch.load(sys.argv[2] + ".meta", map_location="cpu", weights_only=False)
assert type(gen).__module__ == "generators.generators", type(gen).__module__
assert type(gen).__mro__[1].__name__ == "_RenderSkeleton", "not the mirror class"
assert gen.step == 1234 and gen.epoch == 7 and gen.device == "cpu"
# parameter registration order (torch_ema is positional) and state_dict equality
assert [n for n, _ in gen.named_parameters()] == meta["names"]
sd = gen.state_dict()
assert list(sd.keys()) == list(meta["state"].keys())
for k, v in meta["state"].items():
    assert torch.equal(sd[k], v), k
# what ExponentialMovingAverage.copy_to does: param.data.copy_(shadow) in parameters() order
shadow = [p.detach().clone() + 0.125 for p in gen.parameters()]
for s_param, param in zip(shadow, gen.parameters()):
    param.data.copy_(s_param.data)
for (n, p), s in zip(gen.named_parameters(), shadow):
    assert torch.equal(p, s), n
# the sequence of render_multiview_images_double_semantic.py:59-65 up to the render call
gen.softmax_label = False
gen.neural_renderer_img = None
gen.neural_renderer_seg = None
gen.set_device("cpu")            # runs generate_avg_frequencies with the mapping network on the CPU
gen.eval()
assert hasattr(gen, "avg_frequencies") or hasattr(gen, "avg_frequencies_geo")
# and a checkpoint saved under the mirror carries the reference's module paths
import io, pickletools
buf = io.BytesIO(); torch.save(gen, buf)
assert b"generators.generators" in buf.getvalue() and b"fenerf_b200" not in buf.getvalue()
print("ok")
'''


@pytest.mark.parametrize("model", ["A", "D"])
def test_reference_pickle_loads_under_the_mirror(tmp_path, model):
    out = _run(_LOAD_WITH_MIRROR, _reference_checkpoint(tmp_path, model))
    assert "ok" in out


def test_mirror_pickle_loads_under_the_reference(tmp_path):
    """The other direction: a whole-module checkpoint written under this library is a valid
    reference checkpoint -- unpickled with every class of the reference's packages replaced by an empty
    stand-in named by its module path (so nothing of this library takes part), it has the same module
    classes, attribute names and types, parameter order and state_dict as the reference's own checkpoint,
    and carries the values it was saved with."""
    path = str(tmp_path / "generator.pth")
    _run(r'''
import sys
sys.path.insert(0, sys.argv[1])
import torch, fenerf_b200
g, s = fenerf_b200.install()
torch.manual_seed(0)
gen = g.ImplicitGenerator3d(s.TALLSIREN, 256, 4)
gen.set_device("cpu")
gen.step, gen.epoch = 1234, 7                        # as the reference's checkpoint (train_double_latent_semantic.py)
torch.save(gen, sys.argv[2])
torch.save(gen.state_dict(), sys.argv[2] + ".sd")
''', path)
    out = _run(r'''
import pickle, sys, types
import torch

class _StandInUnpickler(pickle.Unpickler):
    stand_ins = {}

    def find_class(self, module, name):
        if module.split(".")[0] in ("generators", "siren"):
            key = module + "." + name
            if key not in self.stand_ins:
                self.stand_ins[key] = type(name, (torch.nn.Module,), {"__module__": module})
            return self.stand_ins[key]
        return super().find_class(module, name)

stand_in_pickle = types.ModuleType("stand_in_pickle")
stand_in_pickle.Unpickler = _StandInUnpickler

def structure(path):
    gen = torch.load(path, map_location="cpu", pickle_module=stand_in_pickle, weights_only=False)
    mods = [(n, type(m).__module__ + "." + type(m).__name__,
             sorted((k, type(v).__name__) for k, v in vars(m).items() if not k.startswith("_")))
            for n, m in gen.named_modules()]
    params = [n for n, _ in gen.named_parameters()]
    state = [(k, tuple(v.shape), v.dtype) for k, v in gen.state_dict().items()]
    return gen, mods, params, state

gen, mods, params, state = structure(sys.argv[2])
_, ref_mods, ref_params, ref_state = structure(sys.argv[3])
assert type(gen).__module__ == "generators.generators" and type(gen).__name__ == "ImplicitGenerator3d"
assert "fenerf_b200" not in sys.modules
for mine, ref in zip(mods, ref_mods):
    assert mine == ref, (mine, ref)
assert len(mods) == len(ref_mods) and params == ref_params and state == ref_state
sd = torch.load(sys.argv[2] + ".sd", map_location="cpu")
for k, v in gen.state_dict().items():
    assert torch.equal(v, sd[k]), k
print("ok")
''', path, _reference_checkpoint(tmp_path, "A"))
    assert "ok" in out
