"""Parity cases shared by the golden generator, the oracle tests and the GPU parity tests."""
import math
import os
import sys
from dataclasses import dataclass, field
from functools import lru_cache

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# constants of the named curricula (curriculums.py:139-146, 164)
BASE = dict(fov=12, ray_start=0.88, ray_end=1.12, h_mean=math.pi * 0.5, v_mean=math.pi * 0.5, clamp_mode='relu',
            last_back=False, hierarchical_sample=True, sample_dist='gaussian')


#: model letter -> (generator class, SIREN class, number of latent codes, output_dim); A / B are the two
#: benchmarked fields, C / D the networks of the reference's other two curricula (curriculums.py:66, 111)
MODELS = {
    "A": ("ImplicitGenerator3d", "TALLSIREN", 1, 4),
    "B": ("DoubleImplicitGenerator3d", "TextureEmbeddingPiGAN256SEMANTICDISENTANGLE_DIM_96", 2, 22),
    "C": ("ImplicitGenerator3d", "SPATIALSIRENBASELINE", 1, 4),
    "D": ("DoubleImplicitGenerator3d", "SIRENBASELINESEMANTICDISENTANGLE", 2, 22),
    # D with 19 label channels: the only width at which the reference's 'debug' / 'weight_debug' fill modes run at
    # all -- they assign a hard-coded 22-vector to the (C-1)-channel pixels (volumetric_rendering.py:54, 66)
    "E": ("DoubleImplicitGenerator3d", "SIRENBASELINESEMANTICDISENTANGLE", 2, 23),
    # the third wrapper type of generators.py (:914-1294): no avg-frequency table, no psi truncation
    "S": ("StyleGenerator3d", "TALLSIREN", 1, 4),
    # three more of siren.py's variants through the same kernels (FieldSpec table): single latent + semantic head,
    # double latent without one, and the 8 + 8 layer deep-appearance network
    "F": ("ImplicitGenerator3d", "SPATIALSIRENBASELINESEMANTIC", 1, 23),
    "G": ("DoubleImplicitGenerator3d", "SPATIALSIRENDISENTANGLE", 2, 4),
    "H": ("DoubleImplicitGenerator3d", "SPATIALSIRENSEMANTICDISENTANGLE", 2, 22),
}


def n_latents(model):
    return MODELS[model][2]


def construct(generators_mod, siren_mod, model, softmax_label=False):
    """Generator of `model` from a (generators, siren) module pair -- the reference's or the mirror's."""
    gen_name, siren_name, n_lat, out_dim = MODELS[model]
    gen_cls, siren_cls = getattr(generators_mod, gen_name), getattr(siren_mod, siren_name)
    if n_lat == 1:
        return gen_cls(siren_cls, 256, out_dim, softmax_label=softmax_label)
    return gen_cls(siren_cls, 256, 256, out_dim, softmax_label=softmax_label)


@dataclass(frozen=True)
class Case:
    name: str
    model: str                     # key of MODELS
    batch: int
    seed: int
    cfg: dict = field(default_factory=dict)
    method: str = "forward"        # or "staged_forward"
    sigma_bias_shift: float = 0.0  # final_layer.bias += shift (opaque-regime fixture, SURVEY.md 7.1)
    psi: float = 1.0


def _cfg(**kw):
    d = dict(BASE)
    d.update(kw)
    return d


CASES = [
    # parity runs keep the camera at the mean pose unless stated (BASELINE.md section 3)
    Case("a_small", "A", 2, 11, _cfg(img_size=16, num_steps=12, h_stddev=0.3, v_stddev=0.155, nerf_noise=0.0)),
    Case("a_small_noise", "A", 2, 12, _cfg(img_size=16, num_steps=12, h_stddev=0.0, v_stddev=0.0, nerf_noise=0.4)),
    Case("a_small_opaque", "A", 1, 13, _cfg(img_size=16, num_steps=12, h_stddev=0.0, v_stddev=0.0, nerf_noise=0.0,
                                            white_back=True), sigma_bias_shift=0.5),
    Case("a_nohier_softplus", "A", 1, 14, _cfg(img_size=16, num_steps=8, h_stddev=0.0, v_stddev=0.0, nerf_noise=0.0,
                                               hierarchical_sample=False, clamp_mode='softplus', last_back=True)),
    Case("a_lockview_uniform", "A", 1, 15, _cfg(img_size=12, num_steps=9, h_stddev=0.2, v_stddev=0.1, nerf_noise=0.0,
                                                sample_dist='uniform', lock_view_dependence=True, black_back=True)),
    Case("a_cfg1", "A", 1, 16, _cfg(img_size=64, num_steps=12, h_stddev=0.0, v_stddev=0.0, nerf_noise=0.0)),
    Case("a_staged_white", "A", 1, 17, _cfg(img_size=16, num_steps=12, h_stddev=0.0, v_stddev=0.0, nerf_noise=0.0,
                                            fill_mode='eval_white_back'), method="staged_forward", psi=0.7),
    Case("b_small", "B", 1, 21, _cfg(img_size=16, num_steps=12, h_stddev=0.3, v_stddev=0.155, nerf_noise=0.0)),
    Case("b_small_opaque", "B", 1, 22, _cfg(img_size=12, num_steps=10, h_stddev=0.0, v_stddev=0.0, nerf_noise=0.0),
         sigma_bias_shift=0.5),
    Case("b_staged_segpad", "B", 1, 23, _cfg(img_size=16, num_steps=12, h_stddev=0.0, v_stddev=0.0, nerf_noise=0.0,
                                             fill_mode='seg_padding_background', fill_color='grey'),
         method="staged_forward", psi=0.7),
    Case("c_small", "C", 2, 31, _cfg(img_size=16, num_steps=12, h_stddev=0.3, v_stddev=0.155, nerf_noise=0.0)),
    Case("d_small", "D", 1, 32, _cfg(img_size=16, num_steps=12, h_stddev=0.3, v_stddev=0.155, nerf_noise=0.0)),
    Case("d_staged_softmax", "D", 1, 33, _cfg(img_size=12, num_steps=10, h_stddev=0.0, v_stddev=0.0, nerf_noise=0.0,
                                              softmax_label=True, fill_mode='weight'), method="staged_forward", psi=0.7),
    # ---- round 2: the branches round 1 left untested (VERDICT r1 "What's weak" 3) ----
    # fill modes of fancy_integration (volumetric_rendering.py:53-102).  A random-init field has sigma ~ +-0.03, so
    # weights_sum is ~1 where the far sample's sigma is positive (its interval is 1e10 wide) and ~0.01 elsewhere:
    # both sides of the `weights_sum < 0.9` test occur in every image
    Case("e_staged_debug", "E", 1, 41, _cfg(img_size=12, num_steps=10, h_stddev=0.0, v_stddev=0.0, nerf_noise=0.0,
                                            fill_mode='debug'), method="staged_forward", psi=0.7),
    Case("e_staged_weight_debug", "E", 2, 42, _cfg(img_size=12, num_steps=10, h_stddev=0.0, v_stddev=0.0, nerf_noise=0.0,
                                                   fill_mode='weight_debug'), method="staged_forward", psi=0.7),
    Case("b_staged_evalsegpad_white", "B", 1, 43, _cfg(img_size=12, num_steps=10, h_stddev=0.0, v_stddev=0.0,
                                                       nerf_noise=0.0, fill_mode='eval_seg_padding_background',
                                                       fill_color='white'), method="staged_forward", psi=0.7),
    Case("d_staged_segpad_lightgrey", "D", 1, 44, _cfg(img_size=12, num_steps=10, h_stddev=0.0, v_stddev=0.0,
                                                       nerf_noise=0.0, fill_mode='seg_padding_background',
                                                       fill_color='light_grey'), method="staged_forward", psi=0.7),
    Case("a_hier_softplus", "A", 1, 45, _cfg(img_size=16, num_steps=12, h_stddev=0.0, v_stddev=0.0, nerf_noise=0.0,
                                             clamp_mode='softplus')),
    Case("b_noise_b2", "B", 2, 46, _cfg(img_size=12, num_steps=10, h_stddev=0.3, v_stddev=0.155, nerf_noise=0.3)),
    Case("d_b2", "D", 2, 47, _cfg(img_size=12, num_steps=10, h_stddev=0.3, v_stddev=0.155, nerf_noise=0.0)),
    # the three rare sample_dist modes (volumetric_rendering.py:198-219)
    Case("a_cam_hybrid", "A", 2, 48, _cfg(img_size=12, num_steps=9, h_stddev=0.3, v_stddev=0.155, nerf_noise=0.0,
                                          sample_dist='hybrid')),
    Case("a_cam_hybrid2", "A", 2, 51, _cfg(img_size=12, num_steps=9, h_stddev=0.3, v_stddev=0.155, nerf_noise=0.0,
                                           sample_dist='hybrid')),
    Case("a_cam_truncgauss", "A", 3, 49, _cfg(img_size=12, num_steps=9, h_stddev=0.3, v_stddev=0.155, nerf_noise=0.0,
                                              sample_dist='truncated_gaussian')),
    Case("a_cam_spherical", "A", 2, 50, _cfg(img_size=12, num_steps=9, h_stddev=0.3, v_stddev=0.155, nerf_noise=0.0,
                                             sample_dist='spherical_uniform')),
    Case("s_small", "S", 2, 53, _cfg(img_size=12, num_steps=9, h_stddev=0.3, v_stddev=0.155, nerf_noise=0.0)),
    Case("s_staged_weight", "S", 1, 54, _cfg(img_size=12, num_steps=9, h_stddev=0.0, v_stddev=0.0, nerf_noise=0.0,
                                             fill_mode='weight'), method="staged_forward", psi=0.7),
    Case("f_small", "F", 1, 55, _cfg(img_size=12, num_steps=9, h_stddev=0.3, v_stddev=0.155, nerf_noise=0.0)),
    Case("g_small", "G", 2, 56, _cfg(img_size=12, num_steps=9, h_stddev=0.3, v_stddev=0.155, nerf_noise=0.0)),
    Case("h_small", "H", 1, 57, _cfg(img_size=12, num_steps=9, h_stddev=0.3, v_stddev=0.155, nerf_noise=0.0)),
    # ---- the benchmarked shapes themselves (BASELINE.json configs[1] and the configs[4] shape), one face each ----
    Case("a_cfg2", "A", 1, 61, _cfg(img_size=128, num_steps=24, h_stddev=0.3, v_stddev=0.155, nerf_noise=0.0)),
    Case("b_cfg2", "B", 1, 62, _cfg(img_size=128, num_steps=24, h_stddev=0.3, v_stddev=0.155, nerf_noise=0.0)),
    Case("a_cfg5", "A", 1, 63, _cfg(img_size=256, num_steps=48, h_stddev=0.3, v_stddev=0.155, nerf_noise=0.0)),
]
#: cases whose CPU oracle run takes tens of seconds: the CPU suite (-m "not gpu") checks them only with
#: FENERF_SLOW_TESTS=1; the GPU suite always runs them
BIG_CASES = ("b_cfg2", "a_cfg5")
CASE_BY_NAME = {c.name: c for c in CASES}
GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
#: intra-op CPU threads the forward goldens were computed with: torch's CPU reductions split their work by thread count,
#: so the oracle reproduces the reference's stored outputs bit for bit only under the same count
GOLDEN_THREADS = 8


def golden_path(case):
    return os.path.join(GOLDEN_DIR, case.name + ".npz")


def apply_weight_edits(gen, case):
    if case.sigma_bias_shift:
        with torch.no_grad():
            gen.siren.final_layer.bias += case.sigma_bias_shift


def make_latents(case):
    """latent i of the batch = randn(1, 256) under manual_seed(1000 + i); model B: geo then app."""
    zs = []
    for i in range(case.batch):
        torch.manual_seed(1000 + i)
        zs.append([torch.randn(1, 256) for _ in range(n_latents(case.model))])
    return tuple(torch.cat([z[j] for z in zs], 0) for j in range(len(zs[0])))


def reference_kwargs(case):
    kw = dict(case.cfg)
    if case.method == "staged_forward":
        kw["psi"] = case.psi
        kw["max_batch_size"] = 2400000
    return kw


@lru_cache(maxsize=8)
def _mirror_generator_cached(model, softmax_label):
    from fenerf_b200.generators import generators as g
    from fenerf_b200.siren import siren as s
    torch.manual_seed(0)
    gen = construct(g, s, model, softmax_label)
    gen.eval()
    return gen


def build_mirror(case, device="cpu"):
    """Our mirror classes, constructed under the same seed protocol as the reference; returns a fresh
    deep copy so that weight edits and device moves do not leak between tests."""
    import copy
    gen = copy.deepcopy(_mirror_generator_cached(case.model, bool(case.cfg.get("softmax_label", False))))
    apply_weight_edits(gen, case)
    gen.to(device)
    gen.device = device
    gen.siren.device = device
    return gen


def has_avg_frequencies(case):
    """StyleGenerator3d has no average-frequency table: its staged_forward neither draws nor truncates."""
    return MODELS[case.model][0] != "StyleGenerator3d"


def avg_film_draws(case):
    """The generate_avg_frequencies draws a staged_forward makes first (generators.py:142, 554)."""
    return [torch.randn(10000, 256) for _ in range(n_latents(case.model))]


def loss_weights(shape):
    """Fixed projection of rendered frames to a scalar for the gradient goldens: L = sum(pixels * W)."""
    g = torch.Generator().manual_seed(99)
    return torch.randn(shape, generator=g)


def grid_probe_index(numel, n):
    """Fixed pseudo-random flat indices into the feature grid (the gradient goldens store only these entries)."""
    g = torch.Generator().manual_seed(7)
    return torch.randint(0, numel, (n,), generator=g)
