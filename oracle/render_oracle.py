"""CPU oracle of the FENeRF render hot path.  TEST INFRASTRUCTURE -- not product code.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
import this package, and only as the checker or as the timed CPU baseline.  The product path
(fenerf_b200/) never imports it and fails loudly when its CUDA library is missing.

What it is: a restatement, as a plain functional pipeline over fp32 CPU tensors, of the algorithm
the reference runs inside ``*Generator3d.forward`` -- same ATen ops in the same order, so that on
the same host it reproduces the reference's output bit for bit.  Each function cites the
reference span it follows (paths relative to the reference root).

How it is pinned: the reference holds no tests or golden vectors for this path (SURVEY.md
section 4), so the pin is the unmodified reference itself, imported in the build container:
``tests/golden/make_goldens.py`` (committed) runs it on fixed seeds and stores its outputs under
``tests/golden/``; ``tests/test_oracle.py`` checks this oracle against those files within a
cross-host tolerance, and ``tests/test_oracle_vs_reference.py`` checks bit-equality with them.

RNG: every random draw goes through a ``Draws`` object so that a run can be recorded on the CPU
and replayed, tensor for tensor, into the CUDA path (CPU and CUDA generators differ).
"""
import math

import numpy as np
import torch
import torch.nn.functional as F


# --------------------------------------------------------------------------------------------
# RNG recording
# --------------------------------------------------------------------------------------------
class Draws:
    """Draws from torch's global CPU generator and keeps a log [(kind, tensor), ...]."""

    def __init__(self):
        self.log = []

    def rand(self, *shape):
        t = torch.rand(shape)
        self.log.append(("rand", t))
        return t

    def randn(self, *shape):
        t = torch.randn(shape)
        self.log.append(("randn", t))
        return t

    def coin(self):
        """Python's global `random.random()` ('hybrid' camera mode, volumetric_rendering.py:199)."""
        import random
        v = random.random()
        self.log.append(("coin", torch.tensor(v, dtype=torch.float64)))
        return v


# --------------------------------------------------------------------------------------------
# camera + rays        generators/volumetric_rendering.py:109-248
# --------------------------------------------------------------------------------------------
def unit(v):
    # math_utils_torch.py:16-20
    return v / (torch.norm(v, dim=-1, keepdim=True))


def camera_rays(n_img, img_size, num_steps, fov, ray_start, ray_end):
    """Camera-space sample points, depths and directions (get_initial_rays_trig, :109-131)."""
    gx, gy = torch.meshgrid(torch.linspace(-1, 1, img_size), torch.linspace(1, -1, img_size), indexing="ij")
    gx = gx.T.flatten()
    gy = gy.T.flatten()
    gz = -torch.ones_like(gx) / np.tan((2 * math.pi * fov / 360) / 2)
    dirs = unit(torch.stack([gx, gy, gz], -1))
    z = torch.linspace(ray_start, ray_end, num_steps).reshape(1, num_steps, 1).repeat(img_size * img_size, 1, 1)
    pts = dirs.unsqueeze(1).repeat(1, num_steps, 1) * z
    return torch.stack(n_img * [pts]), torch.stack(n_img * [z]), torch.stack(n_img * [dirs])


def jitter(points, z_vals, dirs, draws):
    """Stratified perturbation (perturb_points, :133-139): draw #1."""
    spacing = z_vals[:, :, 1:2, :] - z_vals[:, :, 0:1, :]
    offset = (draws.rand(*z_vals.shape) - 0.5) * spacing
    return points + offset * dirs.unsqueeze(2), z_vals + offset


def _first_inside_pm2(draws, n):
    """truncated_normal_ (:170-177) with mean 0 / std 1: of four normal draws per entry, the first one inside
    (-2, 2) (the first of the four if none is)."""
    tmp = draws.randn(n, 1, 4)
    valid = (tmp < 2) & (tmp > -2)
    ind = valid.max(-1, keepdim=True)[1]
    return tmp.gather(-1, ind).squeeze(-1) * 1 + 0


def camera_pose(n, h_stddev, v_stddev, h_mean, v_mean, mode, draws):
    """theta (yaw), phi (pitch) and the unit-sphere origin (sample_camera_positions, :179-228)."""
    if mode == 'uniform':
        theta = (draws.rand(n, 1) - 0.5) * 2 * h_stddev + h_mean
        phi = (draws.rand(n, 1) - 0.5) * 2 * v_stddev + v_mean
    elif mode in ('normal', 'gaussian'):
        theta = draws.randn(n, 1) * h_stddev + h_mean
        phi = draws.randn(n, 1) * v_stddev + v_mean
    elif mode == 'hybrid':
        if draws.coin() < 0.5:
            theta = (draws.rand(n, 1) - 0.5) * 2 * h_stddev * 2 + h_mean
            phi = (draws.rand(n, 1) - 0.5) * 2 * v_stddev * 2 + v_mean
        else:
            theta = draws.randn(n, 1) * h_stddev + h_mean
            phi = draws.randn(n, 1) * v_stddev + v_mean
    elif mode == 'truncated_gaussian':
        theta = _first_inside_pm2(draws, n) * h_stddev + h_mean
        phi = _first_inside_pm2(draws, n) * v_stddev + v_mean
    elif mode == 'spherical_uniform':
        theta = (draws.rand(n, 1) - .5) * 2 * h_stddev + h_mean
        v_std, v_mu = v_stddev / math.pi, v_mean / math.pi
        v = torch.clamp((draws.rand(n, 1) - .5) * 2 * v_std + v_mu, 1e-5, 1 - 1e-5)
        phi = torch.arccos(1 - 2 * v)
    else:
        theta = torch.ones((n, 1), dtype=torch.float) * h_mean
        phi = torch.ones((n, 1), dtype=torch.float) * v_mean
    phi = torch.clamp(phi, 1e-5, math.pi - 1e-5)
    origin = torch.zeros((n, 3))
    origin[:, 0:1] = 1 * torch.sin(phi) * torch.cos(theta)
    origin[:, 2:3] = 1 * torch.sin(phi) * torch.sin(theta)
    origin[:, 1:2] = 1 * torch.cos(phi)
    return origin, phi, theta


def look_at(forward, origin):
    """4x4 camera-to-world (create_cam2world_matrix, :230-248)."""
    forward = unit(forward)
    up = torch.tensor([0, 1, 0], dtype=torch.float).expand_as(forward)
    left = unit(torch.cross(up, forward, dim=-1))
    up = unit(torch.cross(forward, left, dim=-1))
    rot = torch.eye(4).unsqueeze(0).repeat(forward.shape[0], 1, 1)
    rot[:, :3, :3] = torch.stack((-left, up, -forward), axis=-1)
    trans = torch.eye(4).unsqueeze(0).repeat(forward.shape[0], 1, 1)
    trans[:, :3, 3] = origin
    return trans @ rot


def to_world(points, z_vals, dirs, cam2world):
    """Homogeneous pad + the three bmm (transform_sampled_points, :155-168)."""
    n, n_rays, n_steps, _ = points.shape
    hom = torch.ones((n, n_rays, n_steps, 4))
    hom[:, :, :, :3] = points
    pts_w = torch.bmm(cam2world, hom.reshape(n, -1, 4).permute(0, 2, 1)).permute(0, 2, 1).reshape(n, n_rays, n_steps, 4)
    dirs_w = torch.bmm(cam2world[..., :3, :3], dirs.reshape(n, -1, 3).permute(0, 2, 1)).permute(0, 2, 1).reshape(n, n_rays, 3)
    org = torch.zeros((n, 4, n_rays))
    org[:, 3, :] = 1
    org_w = torch.bmm(cam2world, org).permute(0, 2, 1).reshape(n, n_rays, 4)[..., :3]
    return pts_w[..., :3], dirs_w, org_w


# --------------------------------------------------------------------------------------------
# point network        siren/siren.py:113-123, 164-178, 314-330, 1509-1530
# --------------------------------------------------------------------------------------------
def _film(linear, x, freq, phase):
    x = linear(x)
    freq = freq.unsqueeze(1).expand_as(x)
    phase = phase.unsqueeze(1).expand_as(x)
    return torch.sin(freq * x + phase)


def grid_lookup(coords, grid):
    # sample_from_3dgrid, siren.py:314-330
    b, n, d = coords.shape
    s = F.grid_sample(grid.float().expand(b, -1, -1, -1, -1), coords.float().reshape(b, 1, 1, -1, d), mode='bilinear',
                      padding_mode='zeros', align_corners=True)
    nn_, c, h, w, dd = s.shape
    return s.permute(0, 4, 3, 2, 1).reshape(nn_, h * w * dd, c)


def field_eval(field, points, film, dirs):
    """(B,P,3), (B,L,2,256) [15f+30, phase], (B,P,3) -> (B,P,C).  `field` is any module with the
    reference's attribute names (network, final_layer, color_layer_sine, ...)."""
    has_grid = hasattr(field, 'spatial_embeddings')
    has_labels = hasattr(field, 'label_layer_linear')
    x = points
    if hasattr(field, 'gridwarper'):
        x = x * (2 / 0.24)                      # UniformBoxWarp(0.24), siren.py:218, 1203, 1501, 1513
    if has_grid:
        feats = grid_lookup(x, field.spatial_embeddings)
    h = x
    n_trunk = len(field.network)
    for i, layer in enumerate(field.network):
        h = _film(layer.layer, h, film[:, i, 0], film[:, i, 1])
    sigma = field.final_layer(h)
    c = torch.cat([dirs, feats, h], dim=-1) if has_grid else torch.cat([dirs, h], dim=-1)
    if has_labels:
        labels = field.label_layer_linear(h)
    color = field.color_layer_sine
    color = list(color) if isinstance(color, torch.nn.ModuleList) else [color]
    for j, layer in enumerate(color):
        c = _film(layer.layer, c, film[:, n_trunk + j, 0], film[:, n_trunk + j, 1])
    rgb = torch.sigmoid(field.color_layer_linear[0](c))
    return torch.cat([labels, rgb, sigma], dim=-1) if has_labels else torch.cat([rgb, sigma], dim=-1)


# --------------------------------------------------------------------------------------------
# compositing + resampling       generators/volumetric_rendering.py:18-106, 259-300
# --------------------------------------------------------------------------------------------
_FILL_VALUE = {'white': 1.0, 'black': 0.0, 'grey': 0.5, 'light_grey': 0.81}


def alpha_composite(raw, z_vals, draws, noise_std, clamp_mode, last_back=False, white_back=False, black_back=False,
                    fill_mode=None, fill_color='black'):
    """fancy_integration (:18-106).  Returns (values, depth, weights, weights_sum)."""
    values, sigmas = raw[..., :-1], raw[..., -1:]
    deltas = z_vals[:, :, 1:] - z_vals[:, :, :-1]
    deltas = torch.cat([deltas, 1e10 * torch.ones_like(deltas[:, :, :1])], -2)
    noise = draws.randn(*sigmas.shape) * noise_std
    if clamp_mode == 'softplus':
        alphas = 1 - torch.exp(-deltas * (F.softplus(sigmas + noise)))
    elif clamp_mode == 'relu':
        alphas = 1 - torch.exp(-deltas * (F.relu(sigmas + noise)))
    else:
        raise TypeError("exceptions must derive from BaseException")
    shifted = torch.cat([torch.ones_like(alphas[:, :, :1]), 1 - alphas + 1e-10], -2)
    weights = alphas * torch.cumprod(shifted, -2)[:, :, :-1]
    weights_sum = weights.sum(2)
    if last_back:
        weights[:, :, -1] += (1 - weights_sum)
    out = torch.sum(weights * values, -2)
    depth = torch.sum(weights * z_vals, -2)
    if white_back:
        out = out + 1 - weights_sum
    if black_back:
        out = out + (1 - weights_sum) * -1
    empty = weights_sum.squeeze(-1) < 0.9
    n_ch = out.shape[-1]
    if fill_mode in ('debug', 'weight_debug'):
        out[empty] = torch.tensor([1.] + [0.] * (n_ch - 1))
    elif fill_mode in ('seg_padding_background', 'eval_seg_padding_background'):
        out = torch.cat([torch.zeros((out.shape[0], out.shape[1], 1)), out], dim=-1)
        if fill_color in _FILL_VALUE:
            out[empty] = torch.tensor([1.] + [_FILL_VALUE[fill_color]] * n_ch)
    elif fill_mode == 'eval_white_back':
        out[empty] = torch.tensor([1., 1., 1.])
    return out, depth, weights, weights_sum


def inverse_cdf_sample(bins, weights, n_samples, draws, eps=1e-5):
    """sample_pdf (:259-300), det=False.  Returns (samples, inds)."""
    n_rays, n_w = weights.shape
    weights = weights + eps
    pdf = weights / torch.sum(weights, -1, keepdim=True)
    cdf = torch.cumsum(pdf, -1)
    cdf = torch.cat([torch.zeros_like(cdf[:, :1]), cdf], -1)
    u = draws.rand(n_rays, n_samples).contiguous()
    inds = torch.searchsorted(cdf, u)
    below = torch.clamp_min(inds - 1, 0)
    above = torch.clamp_max(inds, n_w)
    pair = torch.stack([below, above], -1).view(n_rays, 2 * n_samples)
    cdf_g = torch.gather(cdf, 1, pair).view(n_rays, n_samples, 2)
    bins_g = torch.gather(bins, 1, pair).view(n_rays, n_samples, 2)
    denom = cdf_g[..., 1] - cdf_g[..., 0]
    denom[denom < eps] = 1
    return bins_g[..., 0] + (u - cdf_g[..., 0]) / denom * (bins_g[..., 1] - bins_g[..., 0]), inds


# --------------------------------------------------------------------------------------------
# the render skeleton       generators/generators.py:32-104, 452-527 (+ staged :132-233, 546-646)
# --------------------------------------------------------------------------------------------
def render(field, film, cfg, draws=None, keep_stages=False):
    """One forward of the hot path on the CPU.

    cfg keys: img_size fov ray_start ray_end num_steps h_stddev v_stddev h_mean v_mean
              hierarchical_sample sample_dist lock_view_dependence clamp_mode nerf_noise
              [last_back white_back black_back fill_mode fill_color softmax_label]
    Returns a dict: pixels (B,C_img,R,R) in [-1,1], depth (B,N,1), weights_sum (B,N,1), poses (B,2),
    and, with keep_stages, every intermediate the stage-level parity tests compare.
    """
    draws = draws or Draws()
    b = film.shape[0]
    r, s = cfg['img_size'], cfg['num_steps']
    n = r * r
    st = {}
    with torch.no_grad():
        pts_cam, z_vals, dirs_cam = camera_rays(b, r, s, cfg['fov'], cfg['ray_start'], cfg['ray_end'])
        pts_cam, z_vals = jitter(pts_cam, z_vals, dirs_cam, draws)                       # draw 1
        origin, pitch, yaw = camera_pose(b, cfg['h_stddev'], cfg['v_stddev'], cfg['h_mean'], cfg['v_mean'],
                                         cfg.get('sample_dist'), draws)                  # draws 2, 3
        cam2world = look_at(unit(-origin), origin)
        pts, dirs, origins = to_world(pts_cam, z_vals, dirs_cam, cam2world)
        dirs_pp = dirs.unsqueeze(-2).expand(-1, -1, s, -1).reshape(b, n * s, 3)
        pts = pts.reshape(b, n * s, 3)
        if cfg.get('lock_view_dependence', False):
            dirs_pp = torch.zeros_like(dirs_pp)
            dirs_pp[..., -1] = -1
        coarse = field_eval(field, pts, film, dirs_pp).reshape(b, n, s, -1)
        st.update(points_coarse=pts.reshape(b, n, s, 3), z_coarse=z_vals, dirs=dirs, origins=origins[:, 0, :],
                  cam2world=cam2world, raw_coarse=coarse)
        if cfg['hierarchical_sample']:
            _, _, w, _ = alpha_composite(coarse, z_vals, draws, cfg['nerf_noise'], cfg['clamp_mode'])   # draw 4
            w = w.reshape(b * n, s) + 1e-5
            zf = z_vals.reshape(b * n, s)
            z_mid = 0.5 * (zf[:, :-1] + zf[:, 1:])
            z_fine, inds = inverse_cdf_sample(z_mid, w[:, 1:-1], s, draws)                              # draw 5
            z_fine = z_fine.reshape(b, n, s, 1)
            pts_f = origins.unsqueeze(2).contiguous() + dirs.unsqueeze(2).contiguous() * z_fine.expand(-1, -1, -1, 3).contiguous()
            fine = field_eval(field, pts_f.reshape(b, n * s, 3), film, dirs_pp).reshape(b, n, s, -1)
            all_raw = torch.cat([fine, coarse], dim=-2)
            all_z = torch.cat([z_fine, z_vals], dim=-2)
            _, order = torch.sort(all_z, dim=-2)
            all_z = torch.gather(all_z, -2, order)
            all_raw = torch.gather(all_raw, -2, order.expand(-1, -1, -1, all_raw.shape[-1]))
            st.update(coarse_weights=w, inds=inds, z_fine=z_fine, points_fine=pts_f, raw_fine=fine, sort_order=order)
        else:
            all_raw, all_z = coarse, z_vals
        px, depth, weights, wsum = alpha_composite(
            all_raw, all_z, draws, cfg['nerf_noise'], cfg['clamp_mode'], last_back=cfg.get('last_back', False),
            white_back=cfg.get('white_back', False), black_back=cfg.get('black_back', False),
            fill_mode=cfg.get('fill_mode'), fill_color=cfg.get('fill_color', 'black'))                  # draw 6
        if cfg.get('softmax_label', False):
            px = torch.cat([torch.nn.Softmax(dim=-1)(px[..., :-3]), px[..., -3:]], dim=-1)
        px = px.reshape((b, r, r, -1)).permute(0, 3, 1, 2).contiguous() * 2 - 1
        st.update(all_raw=all_raw, all_z=all_z, weights=weights)
    out = dict(pixels=px, depth=depth, weights_sum=wsum, poses=torch.cat([pitch, yaw], -1), draws=draws.log)
    if keep_stages:
        out['stages'] = st
    return out


def film_from_latents(field, latents):
    """Mapping network(s) + the 15 f + 30 affine (siren.py:161, 165, 1505-1511) -> (B, L, 2, 256)."""
    with torch.no_grad():
        if len(latents) == 1:
            f, p = field.mapping_network(latents[0])
            f = f * 15 + 30
        else:
            f_geo, p_geo = field.geo_mapping_network(latents[0])
            f_app, p_app = field.app_mapping_network(latents[1])
            f = torch.cat([f_geo * 15 + 30, f_app * 15 + 30], -1)
            p = torch.cat([p_geo, p_app], -1)
        b = f.shape[0]
        return torch.stack([f.reshape(b, -1, 256), p.reshape(b, -1, 256)], dim=2).contiguous()


# --------------------------------------------------------------------------------------------
# frame consumers        train_double_latent_semantic.py:36-55, 66-72; fid_evaluation.py:146-151
# --------------------------------------------------------------------------------------------
COLOR_MAP = {0: [0, 0, 0], 1: [204, 0, 0], 2: [76, 153, 0], 3: [204, 204, 0], 4: [51, 51, 255], 5: [204, 0, 204],
             6: [0, 255, 255], 7: [255, 204, 204], 8: [102, 51, 0], 9: [255, 0, 0], 10: [102, 204, 0], 11: [255, 255, 0],
             12: [0, 0, 153], 13: [0, 0, 204], 14: [255, 51, 153], 15: [0, 204, 204], 16: [0, 51, 0], 17: [255, 153, 51],
             18: [0, 204, 0]}


def mask2color(masks):
    """train_double_latent_semantic.py:66-72."""
    masks = torch.argmax(masks, dim=1).float()
    sample_mask = torch.zeros((masks.shape[0], masks.shape[1], masks.shape[2], 3), dtype=torch.float)
    for key in COLOR_MAP:
        sample_mask[masks == key] = torch.tensor(COLOR_MAP[key], dtype=torch.float)
    return sample_mask.permute(0, 3, 1, 2)


def save_image_bytes(img):
    """The uint8 HWC array torchvision.utils.save_image(img, normalize=True, range=(-1, 1)) hands to PIL
    (fid_evaluation.py:149; torchvision 0.x utils.py:84-90 norm_ip: clamp to the range, sub low, div max(high - low, 1e-5);
    then save_image's mul(255).add_(0.5).clamp_(0, 255).to(uint8))."""
    x = img.clone().float().clamp_(min=-1, max=1)
    x = (x - (-1)) / max(1 - (-1), 1e-5)
    return x.mul(255).add_(0.5).clamp_(0, 255).permute(1, 2, 0).to(torch.uint8)
