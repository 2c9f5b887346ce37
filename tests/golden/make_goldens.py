"""Generates tests/golden/*.npz by running the UNMODIFIED reference (needs /root/reference).

    python tests/golden/make_goldens.py

The reference holds no golden vectors for the render path (SURVEY.md section 4), so the pin of the
oracle is the reference's own forward on fixed seeds, captured here.  Run in the build container
only; the .npz files travel with the repo, /root/reference does not.

Seed protocol (shared with tests/_cases.py):
  torch.manual_seed(0)            -> construct the generator (reference init order)
  generator.set_device('cpu')     -> consumes the generate_avg_frequencies draws
  [case-specific weight edits, e.g. final_layer.bias += 0.5]
  torch.manual_seed(1000 + i)     -> latent i = randn(1, 256)    (geo, then app for model B)
  torch.manual_seed(case.seed)    -> the forward under test  (+ random.seed(case.seed): the 'hybrid' camera
                                     mode flips Python's global coin, volumetric_rendering.py:199)
"""
import hashlib
import os
import random
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from oracle import ref_shim  # noqa: E402
import _cases  # noqa: E402


def state_digest(module):
    h = hashlib.sha256()
    for k, v in module.state_dict().items():
        h.update(k.encode())
        h.update(v.detach().cpu().numpy().tobytes())
    return h.hexdigest()


def build_reference(case, ref_generators, ref_siren):
    torch.manual_seed(0)
    gen = _cases.construct(ref_generators, ref_siren, case.model, case.cfg.get("softmax_label", False))
    gen.set_device("cpu")      # (draws the avg-frequency latents for the Implicit / Double wrappers; nothing for Style)
    gen.eval()
    digest = state_digest(gen)
    _cases.apply_weight_edits(gen, case)
    return gen, digest


def main():
    ref_generators, ref_siren, _ = ref_shim.load()
    out_dir = os.path.dirname(os.path.abspath(__file__))
    only = set(sys.argv[1:])                       # optional: case names to (re)generate
    torch.set_num_threads(_cases.GOLDEN_THREADS)
    for case in _cases.CASES:
        if only and case.name not in only:
            continue
        gen, digest = build_reference(case, ref_generators, ref_siren)
        latents = _cases.make_latents(case)
        kw = _cases.reference_kwargs(case)
        torch.manual_seed(case.seed)
        random.seed(case.seed)
        with torch.no_grad():
            if case.method == "forward":
                pixels, poses = gen(*latents, **kw)
                extra = {"poses": poses.numpy()}
            elif case.method == "staged_forward":
                res = gen.staged_forward(*latents, **kw)
                pixels = res[0]
                extra = {"depth_map": res[1].numpy()}
                if len(res) > 2:
                    extra["third"] = res[2].numpy()
            else:
                raise ValueError(case.method)
        path = os.path.join(out_dir, case.name + ".npz")
        np.savez_compressed(path, pixels=pixels.cpu().numpy(), state_digest=np.array(digest), **extra)
        print("%-28s pixels %s  mean|x| %.6f  -> %s (%.1f KB)" % (
            case.name, tuple(pixels.shape), float(pixels.abs().mean()), os.path.basename(path), os.path.getsize(path) / 1024))


# ---- gradients of the differentiable call (the reference's G step / inversion path) -----------------
GRAD_CASES = ("a_small", "d_small", "b_small", "d_staged_softmax", "a_hier_softplus")
#: parameters whose gradients are stored (a cross-section of trunk, heads, colour branch, mapping network)
GRAD_PARAMS = {
    "A": ["siren.network.0.layer.weight", "siren.network.7.layer.bias", "siren.final_layer.weight",
          "siren.color_layer_sine.layer.bias", "siren.color_layer_linear.0.weight",
          "siren.mapping_network.network.8.bias"],
    "D": ["siren.network.0.layer.weight", "siren.network.7.layer.bias", "siren.final_layer.weight",
          "siren.color_layer_sine.2.layer.bias", "siren.color_layer_linear.0.weight",
          "siren.label_layer_linear.1.weight", "siren.geo_mapping_network.network.8.bias",
          "siren.app_mapping_network.network.8.bias"],
    "B": ["siren.network.0.layer.weight", "siren.network.3.layer.weight", "siren.network.7.layer.bias",
          "siren.final_layer.weight", "siren.final_layer.bias", "siren.color_layer_sine.0.layer.weight",
          "siren.color_layer_sine.2.layer.bias", "siren.color_layer_linear.0.weight", "siren.color_layer_linear.0.bias",
          "siren.label_layer_linear.0.weight", "siren.label_layer_linear.1.bias", "siren.label_layer_linear.2.weight",
          "siren.geo_mapping_network.network.8.bias", "siren.app_mapping_network.network.8.bias"],
}
#: model B's grid gradient is 113 MB: stored as a fixed random projection (and its abs-sum)
GRID_PROBE = 4096


def grad_goldens():
    """tests/golden/grad_<case>.npz: d L / d (latents, selected parameters) of the reference's forward with
    autograd on, same seed protocol (and therefore the same random draws) as the forward goldens."""
    ref_generators, ref_siren, _ = ref_shim.load()
    out_dir = os.path.dirname(os.path.abspath(__file__))
    for name in GRAD_CASES:
        case = _cases.CASE_BY_NAME[name]
        gen, _ = build_reference(case, ref_generators, ref_siren)
        latents = tuple(z.clone().requires_grad_(True) for z in _cases.make_latents(case))
        torch.manual_seed(case.seed)
        kw = {k: v for k, v in case.cfg.items() if k != "fill_mode"}      # forward() of a staged case: same config
        pixels, _ = gen(*latents, **kw)
        loss = (pixels * _cases.loss_weights(pixels.shape)).sum()
        loss.backward()
        params = dict(gen.named_parameters())
        out = {"loss": np.array(loss.item())}
        for i, z in enumerate(latents):
            out["latent%d" % i] = z.grad.numpy()
        for k in GRAD_PARAMS[case.model]:
            out[k] = params[k].grad.numpy()
        if "siren.spatial_embeddings" in params:
            g = params["siren.spatial_embeddings"].grad.reshape(-1)
            idx = _cases.grid_probe_index(g.numel(), GRID_PROBE)
            out["grid_probe"] = g[idx].numpy()
            out["grid_abs_sum"] = np.array(g.abs().sum().item())
        path = os.path.join(out_dir, "grad_%s.npz" % name)
        np.savez_compressed(path, **out)
        print("%-28s loss %.6f  %d gradient tensors -> %s (%.1f KB)" % (
            name, loss.item(), len(out) - 1, os.path.basename(path), os.path.getsize(path) / 1024))


def frequency_grad_goldens():
    """tests/golden/gradfreq_a_small.npz: the inversion call -- d L / d (frequencies, phase_shifts) through
    forward_with_frequencies (inverse_render_double_semantic.py:385-407, generators.py:353-431)."""
    ref_generators, ref_siren, _ = ref_shim.load()
    out_dir = os.path.dirname(os.path.abspath(__file__))
    for name in ("a_small", "d_small"):
        case = _cases.CASE_BY_NAME[name]
        gen, _ = build_reference(case, ref_generators, ref_siren)
        latents = _cases.make_latents(case)
        with torch.no_grad():
            if case.model == "A":
                fp = list(gen.siren.mapping_network(latents[0]))
            else:
                fg, pg = gen.siren.geo_mapping_network(latents[0])
                fa, pa = gen.siren.app_mapping_network(latents[1])
                fp = [fg, fa, pg, pa]
        fp = [t.clone().requires_grad_(True) for t in fp]
        torch.manual_seed(case.seed)
        pixels, _ = gen.forward_with_frequencies(*fp, **case.cfg)
        loss = (pixels * _cases.loss_weights(pixels.shape)).sum()
        loss.backward()
        out = {"loss": np.array(loss.item())}
        for i, t in enumerate(fp):
            out["arg%d" % i] = t.grad.numpy()
        path = os.path.join(out_dir, "gradfreq_%s.npz" % name)
        np.savez_compressed(path, **out)
        print("%-28s loss %.6f -> %s (%.1f KB)" % (name, loss.item(), os.path.basename(path), os.path.getsize(path) / 1024))


class _RecordDraws:
    """Records every torch.rand / randn / randperm made while the reference runs (part_forward draws per ray subset,
    which the oracle does not restate): the GPU test replays them through ReplayRng."""

    def __enter__(self):
        self.log = []
        self.saved = (torch.rand, torch.randn, torch.randperm)

        def wrap(kind, fn):
            def inner(*a, **k):
                t = fn(*a, **k)
                self.log.append((kind, t.clone()))
                return t
            return inner
        torch.rand, torch.randn, torch.randperm = (wrap(k, f) for k, f in zip(("rand", "randn", "randperm"), self.saved))
        return self

    def __exit__(self, *exc):
        torch.rand, torch.randn, torch.randperm = self.saved


def part_forward_goldens():
    """tests/golden/part_d_small.npz: ray-subset training (generators.py:858-910) -- frames, recorded draws and
    gradients of DoubleImplicitGenerator3d.forward(..., grad_points=G)."""
    ref_generators, ref_siren, _ = ref_shim.load()
    out_dir = os.path.dirname(os.path.abspath(__file__))
    case = _cases.CASE_BY_NAME["d_small"]
    gen, _ = build_reference(case, ref_generators, ref_siren)
    latents = tuple(z.clone().requires_grad_(True) for z in _cases.make_latents(case))
    n_rays = case.cfg["img_size"] ** 2
    kw = dict(case.cfg, grad_points=n_rays * 3 // 8)
    torch.manual_seed(case.seed)
    with _RecordDraws() as rec:
        pixels, poses = gen(*latents, **kw)
    loss = (pixels * _cases.loss_weights(pixels.shape)).sum()
    loss.backward()
    params = dict(gen.named_parameters())
    out = {"loss": np.array(loss.item()), "pixels": pixels.detach().numpy(), "poses": poses.detach().numpy(),
           "grad_points": np.array(kw["grad_points"]), "n_draws": np.array(len(rec.log))}
    for i, (kind, t) in enumerate(rec.log):
        out["draw%d_%s" % (i, kind)] = t.numpy()
    for i, z in enumerate(latents):
        out["g_latent%d" % i] = z.grad.numpy()
    for k in GRAD_PARAMS[case.model]:
        out["g_" + k] = params[k].grad.numpy()
    path = os.path.join(out_dir, "part_d_small.npz")
    np.savez_compressed(path, **out)
    print("%-28s loss %.6f  %d draws -> %s (%.1f KB)" % ("part_d_small", loss.item(), len(rec.log), os.path.basename(path),
                                                        os.path.getsize(path) / 1024))


def pickle_goldens():
    """tests/golden/ref_pickle_<A|D>.npz: whole-module checkpoints written by the reference's own classes
    (train_double_latent_semantic.py:523 style) for tests/test_dropin.py.  What those tests check is the pickle's
    structure (module paths, attribute names, parameter order) and that every state_dict entry lands on the right
    tensor, so each state_dict tensor is first filled with its own constant (index + 1) / 64: the file then deflates
    from ~10 MB to ~50 KB.  `checkpoint` holds the torch.save bytes, `meta` those of {names, state}."""
    import io
    ref_generators, ref_siren, _ = ref_shim.load()
    out_dir = os.path.dirname(os.path.abspath(__file__))
    for model in ("A", "D"):
        torch.manual_seed(0)
        if model == "A":
            gen = ref_generators.ImplicitGenerator3d(ref_siren.TALLSIREN, 256, 4)
        else:
            gen = ref_generators.DoubleImplicitGenerator3d(ref_siren.SIRENBASELINESEMANTICDISENTANGLE, 256, 256, 22)
        gen.set_device("cpu")
        gen.step, gen.epoch = 1234, 7
        with torch.no_grad():
            for i, t in enumerate(gen.state_dict().values()):
                t.fill_((i + 1) / 64)
        ckpt, meta = io.BytesIO(), io.BytesIO()
        torch.save(gen, ckpt)
        torch.save({"names": [n for n, _ in gen.named_parameters()], "state": gen.state_dict()}, meta)
        path = os.path.join(out_dir, "ref_pickle_%s.npz" % model)
        np.savez_compressed(path, checkpoint=np.frombuffer(ckpt.getvalue(), np.uint8),
                            meta=np.frombuffer(meta.getvalue(), np.uint8))
        print("%-28s %d + %d bytes -> %s (%.1f KB)" % ("ref_pickle_" + model, len(ckpt.getvalue()), len(meta.getvalue()),
                                                       os.path.basename(path), os.path.getsize(path) / 1024))


if __name__ == "__main__":
    if sys.argv[1:2] == ["--part"]:
        part_forward_goldens()
    elif sys.argv[1:2] == ["--pickles"]:
        pickle_goldens()
    elif sys.argv[1:2] == ["--grads"]:
        grad_goldens()
        frequency_grad_goldens()
    else:
        main()
