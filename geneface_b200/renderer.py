"""B200-native drop-in for modules/radnerfs/{renderer,radnerf,radnerf_torso}.py (reference @ 15ff4e5c).

Same classes, constructor (`hparams` dict), parameter/buffer names (reference checkpoints load with
`load_state_dict`) and the same `render(rays_o, rays_d, cond, bg_coords, poses, index=0, dt_gamma=0,
bg_color=None, perturb=False, force_all_rays=False, max_steps=1024, T_thresh=1e-4, **kwargs) -> dict`
boundary (renderer.py:263, radnerf_torso.py:86), `**hparams` splat tolerated.

Eval mode has two implementations of the same semantics:
  * fused (default): one call into libgfrender `gf_render_frame` -- no host loop, no device sync;
  * reference_loop=True (or perturb=True, which needs torch's RNG stream): the reference's host-driven
    march / field / composite loop (renderer.py:314-351) on our fine-grained ops, for parity testing.
Training mode runs the reference's training branch (renderer.py:296-313) on our ops with autograd.
There is no CPU path: tensors must be CUDA and libgfrender.so must load.
"""
import ctypes
import math
import os
import random

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _lib, raymarching
from ._lib import c_f32, c_u32, c_vp, check, ptr, stream_ptr
from .cond_encoder import MLP, AudioAttNet, AudioNet
from .encoders import get_encoder
from .utils import convert_poses, custom_meshgrid, get_audio_features, trunc_exp


# ------------------------------------------------------------------------- C structs (include/gfrender.h)
class GfModelDesc(ctypes.Structure):
    _fields_ = [
        ("bound", c_f32), ("cascade", c_u32), ("grid_size", c_u32), ("min_near", c_f32), ("aabb", c_f32 * 6),
        ("gridtype", c_u32), ("interp", c_u32), ("hidden_dim", c_u32), ("cond_dim", c_u32), ("ind_dim", c_u32),
        ("density_bitfield", c_vp),
        ("pos_embeddings", c_vp), ("pos_offsets", c_vp), ("pos_S", c_f32), ("pos_H", c_u32),
        ("amb_embeddings", c_vp), ("amb_offsets", c_vp), ("amb_S", c_f32), ("amb_H", c_u32),
        ("ambient_w0", c_vp), ("ambient_w1", c_vp), ("ambient_w2", c_vp),
        ("sigma_w0", c_vp), ("sigma_w1", c_vp), ("sigma_w2", c_vp),
        ("color_w0", c_vp), ("color_w1", c_vp),
        ("geo_feat_dim", c_u32), ("ind_code", c_vp),
        ("has_torso", c_u32), ("density_grid_torso", c_vp), ("density_thresh_torso", c_f32), ("torso_shrink", c_f32),
        ("torso_embeddings", c_vp), ("torso_offsets", c_vp), ("torso_S", c_f32), ("torso_H", c_u32),
        ("torso_deform_w0", c_vp), ("torso_deform_w1", c_vp), ("torso_deform_w2", c_vp),
        ("torso_canon_w0", c_vp), ("torso_canon_w1", c_vp), ("torso_canon_w2", c_vp),
        ("torso_ind_dim", c_u32), ("torso_ind_code", c_vp),
    ]


class GfFrame(ctypes.Structure):
    _fields_ = [
        ("H", c_u32), ("W", c_u32), ("rays_o", c_vp), ("rays_d", c_vp), ("pose", c_f32 * 12), ("intrinsics", c_f32 * 4),
        ("cond_feat", c_vp), ("bg_color", c_vp), ("bg_coords", c_vp), ("torso_pose", c_f32 * 6), ("dt_gamma", c_f32),
        ("max_steps", c_u32), ("T_thresh", c_f32), ("precision", c_u32), ("dyn", c_vp),
    ]


class GfOut(ctypes.Structure):
    _fields_ = [
        ("rgb_map", c_vp), ("depth_map", c_vp), ("weights_sum", c_vp), ("torso_alpha_map", c_vp), ("torso_rgb_map", c_vp),
        ("n_samples", c_vp), ("rgb8", c_vp), ("counters", c_vp), ("term_hist", c_vp), ("term_slot", c_vp),
    ]


def _dp(t):
    return None if t is None else t.data_ptr()


PRECISIONS = {'fp32': 0, 'fp16': 1}


class NeRFRenderer(nn.Module):
    """renderer.py:63-367"""

    def __init__(self, hparams):
        super().__init__()
        self.bound = hparams['bound']
        self.cascade = 1 + math.ceil(math.log2(hparams['bound']))
        self.grid_size = hparams['grid_size']
        self.density_scale = 1
        self.min_near = hparams['min_near']
        self.density_thresh = hparams['density_thresh']
        self.cuda_ray = hparams.get('cuda_ray', True)
        b = self.bound
        aabb = torch.FloatTensor([-b, -b / 2, -b, b, b / 2, b])      # renderer.py:78
        self.register_buffer('aabb_train', aabb)
        self.register_buffer('aabb_infer', aabb.clone())
        self.individual_embedding_num = hparams['individual_embedding_num']
        self.individual_embedding_dim = hparams['individual_embedding_dim']
        if self.individual_embedding_dim > 0:
            self.individual_embeddings = nn.Parameter(torch.randn(self.individual_embedding_num, self.individual_embedding_dim) * 0.1)
        self.register_buffer('density_grid', torch.zeros([self.cascade, self.grid_size ** 3]))
        self.register_buffer('density_bitfield', torch.zeros(self.cascade * self.grid_size ** 3 // 8, dtype=torch.uint8))
        self.mean_density = 0
        self.iter_density = 0
        self.register_buffer('step_counter', torch.zeros(16, 2, dtype=torch.int32))
        self.mean_count = 0
        self.local_step = 0
        # fused-path state
        self.precision = hparams.get('render_precision', 'fp32')
        self._gf_model = None
        self._gf_key = None
        self._ws = None
        self.last_counters = None

    # -- to be provided by the field ------------------------------------------------------------------
    def cal_cond_feat(self, cond):
        raise NotImplementedError()

    def forward(self, x, d, cond_feat, individual_code):
        raise NotImplementedError()

    def density(self, x, cond_feat):
        raise NotImplementedError()

    def _model_desc(self):
        raise NotImplementedError()

    def reset_extra_state(self):
        if not self.cuda_ray:
            return
        self.density_grid.zero_()
        self.mean_density = 0
        self.iter_density = 0
        self.step_counter.zero_()
        self.mean_count = 0
        self.local_step = 0

    # -- density grid maintenance (renderer.py:128-260), on our morton3D / dilation / packbits ops -----------
    # The reference walks the H^3 grid in S^3 blocks with three nested Python loops; a B200 holds the whole grid's coordinate
    # list (H^3 x 3 int32 = 25 MB at H=128) and evaluates a cascade in one field call, so both routines work on the full
    # cell list at once: `_cells()` returns (integer coords [H^3,3], morton index [H^3], centre in [-1,1]^3).
    def _cells(self):
        G, dev = self.grid_size, self.density_bitfield.device
        ar = torch.arange(G, dtype=torch.int32, device=dev)
        coords = torch.stack(torch.meshgrid(ar, ar, ar, indexing='ij'), dim=-1).view(-1, 3).contiguous()
        return coords, raymarching.morton3D(coords).long(), coords.float() * (2.0 / (G - 1)) - 1.0

    def _cascade_extent(self, cas):
        bound = min(2 ** cas, self.bound)
        return bound, bound / self.grid_size                 # (half extent of the cascade, half a cell)

    @torch.no_grad()
    def mark_untrained_grid(self, poses, intrinsic, S=64):
        """Cells no training camera ever sees get density -1 (never sampled, never updated).  S = camera batch."""
        if not self.cuda_ray:
            return
        if isinstance(poses, np.ndarray):
            poses = torch.from_numpy(poses)
        fx, fy, cx, cy = intrinsic
        poses = poses.to(self.density_bitfield.device).float()
        _, morton, centre = self._cells()
        seen = torch.zeros_like(self.density_grid)
        for cas in range(self.cascade):
            bound, half_cell = self._cascade_extent(cas)
            world = centre * (bound - half_cell)                                        # [H^3, 3]
            hits = torch.zeros(world.shape[0], device=world.device)
            for k in range(0, poses.shape[0], S):
                R, t = poses[k:k + S, :3, :3], poses[k:k + S, :3, 3]
                cam = (world[None] - t[:, None]) @ R                                    # [b, H^3, 3] camera frame (z forward)
                z = cam[..., 2]
                inside = (z > 0) & (cam[..., 0].abs() < cx / fx * z + 2 * half_cell) & (cam[..., 1].abs() < cy / fy * z + 2 * half_cell)
                hits += inside.sum(0)
            seen[cas, morton] = hits
        self.density_grid[seen == 0] = -1

    @torch.no_grad()
    def update_extra_state(self, decay=0.95, S=128, precision=None):
        """EMA-max update of the occupancy grid from the current field at one jittered point per cell, dilation, bitfield repack.
        The C * H^3 density queries -- the whole cost of the routine -- go through the packed model's field kernels (`gf_field_forward`,
        sigma-only: no colour net) when the configuration is inside the fused envelope, in `precision` (default: the model's render precision)."""
        if not self.cuda_ray:
            return
        dev = self.density_bitfield.device
        rand_idx = random.randint(0, self.conds.shape[0] - 1)
        enc_a = self.cal_cond_feat(get_audio_features(self.conds, 2, rand_idx, self.smo_win_size).to(dev))
        _, morton, centre = self._cells()
        fresh = torch.zeros_like(self.density_grid)
        for cas in range(self.cascade):
            bound, half_cell = self._cascade_extent(cas)
            pts = centre * (bound - half_cell)
            pts = pts + (torch.rand_like(pts) * 2 - 1) * half_cell
            if self._fused_supported():
                sigma = self.field_forward(pts, None, enc_a, precision=precision, sigma_only=True)[0]
            else:
                sigma = self.density(pts, enc_a)['sigma'].reshape(-1).detach()
            fresh[cas, morton] = sigma.to(fresh.dtype) * self.density_scale
        fresh = raymarching.morton3D_dilation(fresh)
        live = (self.density_grid >= 0) & (fresh >= 0)
        self.density_grid[live] = torch.maximum(self.density_grid[live] * decay, fresh[live])
        self.mean_density = torch.mean(self.density_grid.clamp(min=0)).item()
        self.iter_density += 1
        self.density_bitfield = raymarching.packbits(self.density_grid, min(self.mean_density, self.density_thresh), self.density_bitfield)
        steps = min(16, self.local_step)
        if steps > 0:
            self.mean_count = int(self.step_counter[:steps, 0].sum().item() / steps)
        self.local_step = 0
        self.invalidate_fused()   # bitfield changed -> rebuild fused model lazily

    # -- fused path plumbing ----------------------------------------------------------------------------------
    def _fused_supported(self):
        return False

    def _tensors_key(self):
        return tuple((p.data_ptr(), p._version) for p in list(self.parameters()) + list(self.buffers()))

    def invalidate_fused(self):
        """Drop the packed GfModel (and every captured frame graph): the next fused call re-packs from the live tensors.
        Called automatically by load_state_dict / train() / eval() / _apply (.to, .cuda, .half) and by the grid-maintenance
        routines; call it yourself after in-place edits that bypass autograd's version counter (`p.data.copy_`, EMA weight
        surgery, optimizers writing through .data).  That includes edits of the position and ambient grid tables: the packed model
        reads padded copies of them, made when it is built."""
        self._gf_key = None
        self._gf_epoch = getattr(self, '_gf_epoch', 0) + 1

    def load_state_dict(self, *a, **k):
        r = super().load_state_dict(*a, **k)
        self.invalidate_fused()
        return r

    def train(self, mode=True):
        self.invalidate_fused()
        return super().train(mode)

    def _apply(self, fn, *a, **k):
        self.invalidate_fused()
        return super()._apply(fn, *a, **k)

    def gf_model(self, verify=True):
        """Build (or reuse) the packed GfModel for the current weights.  verify=True walks every parameter / buffer
        (data_ptr, version) to detect in-place updates (~0.2 ms of host time); the sequence / graph paths pass verify=False
        and rely on invalidate_fused()."""
        _lib.require_cuda()
        if self._gf_model is not None and self._gf_key is not None and not verify:
            return self._gf_model
        key = self._tensors_key()
        if self._gf_model is not None and key == self._gf_key:
            return self._gf_model
        self.free_gf_model()
        desc, keep = self._model_desc()
        handle = c_vp()
        check(_lib.lib().gf_model_create(ctypes.byref(desc), ctypes.byref(handle), stream_ptr()), "gf_model_create")
        torch.cuda.current_stream().synchronize()
        self._gf_model, self._gf_key, self._gf_keep = handle, key, keep
        self._gf_epoch = getattr(self, '_gf_epoch', 0) + 1          # captured frame graphs hold the old handle: they re-capture
        return handle

    def free_gf_model(self):
        if self._gf_model is not None:
            _lib.lib().gf_model_destroy(self._gf_model)
            self._gf_model = None

    def __del__(self):
        try:
            self.free_gf_model()
        except Exception:  # noqa: BLE001
            pass

    def _workspace(self, N, device):
        need = _lib.lib().gf_render_workspace_bytes(N)
        if self._ws is None or self._ws.numel() < need or self._ws.device != device:
            self._ws = torch.empty(need, dtype=torch.uint8, device=device)
        return self._ws, need

    def field_forward(self, xyzs, dirs, cond_feat, precision=None, sigma_only=False):
        """sigma, rgb, ambient for raw samples through the packed model (== self(...) of the reference loop).
        sigma_only=True (dirs may be None): the density query of the grid maintenance (radnerf.py:107-127); the colour net is skipped
        and rgb is returned as None."""
        model = self.gf_model()
        xyzs = xyzs.float().contiguous()
        dirs = None if (dirs is None or sigma_only) else dirs.float().contiguous()
        M = xyzs.shape[0]
        sig = torch.empty(M, dtype=torch.float32, device=xyzs.device)
        rgb = None if sigma_only else torch.empty(M, 3, dtype=torch.float32, device=xyzs.device)
        amb = torch.empty(M, 2, dtype=torch.float32, device=xyzs.device)
        cf = cond_feat.float().contiguous().view(-1)
        prec = PRECISIONS[precision or self.precision]
        need = _lib.lib().gf_field_workspace_bytes(M, prec)
        ws = torch.empty(need, dtype=torch.uint8, device=xyzs.device)          # caller-owned scratch (the library never allocates)
        check(_lib.lib().gf_field_forward(model, ptr(xyzs), ptr(dirs), ptr(cf), M, ptr(sig), ptr(rgb), ptr(amb), prec, ptr(ws), need,
                                          stream_ptr()), "gf_field_forward")
        return sig, rgb, amb

    def render_fused(self, cond_feat, H, W, *, rays_o=None, rays_d=None, pose=None, intrinsics=None, bg_color=None, bg_coords=None,
                     torso_pose=None, dt_gamma=0.0, max_steps=1024, T_thresh=1e-4, precision=None, want=('weights_sum',), out=None,
                     dyn=None, check_weights=True):
        """One `gf_render_frame` call.  Rays come from rays_o/rays_d [N,3], or from pose [3|4,4] + intrinsics (by value), or from
        `dyn` = DEVICE float[22] (pose[12] | intrinsics[4] | torso_pose[6]) read at execution time -- the CUDA-graph form: no host
        conversion, nothing frame-specific in the launch arguments.  Returns dict of tensors."""
        model = self.gf_model(verify=check_weights)
        dev = cond_feat.device
        N = H * W
        fr = GfFrame()
        fr.H, fr.W = H, W
        if rays_o is not None:
            rays_o = rays_o.float().contiguous().view(-1, 3)
            rays_d = rays_d.float().contiguous().view(-1, 3)
            assert rays_o.shape[0] == N
            fr.rays_o, fr.rays_d = rays_o.data_ptr(), rays_d.data_ptr()
        elif dyn is not None:
            assert dyn.is_cuda and dyn.dtype == torch.float32 and dyn.numel() == 22 and dyn.is_contiguous()
            fr.dyn = dyn.data_ptr()
        else:
            p = np.asarray(pose.detach().cpu() if torch.is_tensor(pose) else pose, dtype=np.float32).reshape(-1, 4)[:3]
            fr.pose = (c_f32 * 12)(*p.reshape(-1).tolist())
            fr.intrinsics = (c_f32 * 4)(*[float(v) for v in intrinsics])
        cf = cond_feat.float().contiguous().view(-1)
        fr.cond_feat = cf.data_ptr()
        if bg_color is not None and torch.is_tensor(bg_color):
            bg_color = bg_color.float().expand(1, N, 3).contiguous().view(-1, 3) if bg_color.dim() == 3 else bg_color.float().contiguous().view(-1, 3)
            fr.bg_color = bg_color.data_ptr()
        elif bg_color is not None and float(bg_color) != 1.0:
            bg_color = torch.full((N, 3), float(bg_color), dtype=torch.float32, device=dev)
            fr.bg_color = bg_color.data_ptr()
        if bg_coords is not None:
            bg_coords = bg_coords.float().contiguous().view(-1, 2)
            fr.bg_coords = bg_coords.data_ptr()
        if torso_pose is not None and dyn is None:
            tp = torso_pose.detach().float().cpu().view(-1).tolist() if torch.is_tensor(torso_pose) else list(torso_pose)
            fr.torso_pose = (c_f32 * 6)(*tp)
        fr.dt_gamma, fr.max_steps, fr.T_thresh = float(dt_gamma), int(max_steps), float(T_thresh)
        fr.precision = PRECISIONS[precision or self.precision]
        res = out if out is not None else {}
        o = GfOut()
        if 'rgb_map' not in res:
            res['rgb_map'] = torch.empty(N, 3, dtype=torch.float32, device=dev)
        if 'depth_map' not in res:
            res['depth_map'] = torch.empty(N, dtype=torch.float32, device=dev)
        o.rgb_map, o.depth_map = res['rgb_map'].data_ptr(), res['depth_map'].data_ptr()
        shapes = {'weights_sum': ((N,), torch.float32), 'torso_alpha_map': ((N,), torch.float32), 'torso_rgb_map': ((N, 3), torch.float32),
                  'n_samples': ((N,), torch.int32), 'rgb8': ((N, 3), torch.uint8), 'counters': ((4,), torch.int64),
                  'term_hist': ((int(max_steps) + 1,), torch.int32), 'term_slot': ((N,), torch.int32)}
        for name in want:
            if name not in res:
                shp, dt = shapes[name]
                res[name] = torch.empty(*shp, dtype=dt, device=dev)
            setattr(o, name, res[name].data_ptr())
        ws, need = self._workspace(N, dev)
        check(_lib.lib().gf_render_frame(model, ctypes.byref(fr), ctypes.byref(o), ptr(ws), need, stream_ptr()), "gf_render_frame")
        # keep temporaries alive until the stream has consumed them
        res['_keep'] = (rays_o, rays_d, cf, bg_color, bg_coords, dyn)
        return res

    # -- the reference boundary ------------------------------------------------------------------------------------
    def _ind_code(self, index):
        if self.individual_embedding_dim > 0:
            return self.individual_embeddings[index] if self.training else self.individual_embeddings[0]
        return None

    def _render_head_loop(self, rays_o, rays_d, nears, fars, cond_feat, ind_code, dt_gamma, max_steps, T_thresh, perturb, field='torch'):
        """renderer.py:314-351 on our ops.  field='torch' evaluates self(...) (torch MLPs + our encoders);
        field='fp32'/'fp16' evaluates through the packed model (gf_field_forward)."""
        N = rays_o.shape[0]
        dev = rays_o.device
        weights_sum = torch.zeros(N, dtype=torch.float32, device=dev)
        depth = torch.zeros(N, dtype=torch.float32, device=dev)
        image = torch.zeros(N, 3, dtype=torch.float32, device=dev)
        rays_alive = torch.arange(N, dtype=torch.int32, device=dev)
        rays_t = nears.clone()
        step = 0
        trace = []
        while step < max_steps:
            n_alive = rays_alive.shape[0]
            if n_alive <= 0:
                break
            n_step = max(min(N // n_alive, 8), 1)
            xyzs, dirs, deltas = raymarching.march_rays(n_alive, n_step, rays_alive, rays_t, rays_o, rays_d, self.bound,
                                                        self.density_bitfield, self.cascade, self.grid_size, nears, fars, 128,
                                                        perturb if step == 0 else False, dt_gamma, max_steps)
            if field == 'torch':
                sigmas, rgbs, _ = self(xyzs, dirs, cond_feat, ind_code)
            else:
                sigmas, rgbs, _ = self.field_forward(xyzs, dirs, cond_feat, precision=field)
            sigmas = self.density_scale * sigmas
            raymarching.composite_rays(n_alive, n_step, rays_alive, rays_t, sigmas, rgbs, deltas, weights_sum, depth, image, T_thresh)
            rays_alive = rays_alive[rays_alive >= 0]
            trace.append((n_alive, n_step))
            step += n_step
        self.last_loop_trace = trace
        return weights_sum, depth, image

    def render(self, rays_o, rays_d, cond, bg_coords, poses, index=0, dt_gamma=0, bg_color=None, perturb=False, force_all_rays=False,
               max_steps=1024, T_thresh=1e-4, **kwargs):
        prefix = rays_o.shape[:-1]
        rays_o = rays_o.contiguous().view(-1, 3)
        rays_d = rays_d.contiguous().view(-1, 3)
        N = rays_o.shape[0]
        results = {}
        cond_feat = self.cal_cond_feat(cond)
        ind_code = self._ind_code(index)
        use_loop = self.training or perturb or kwargs.get('reference_loop', False) or not self._fused_supported()
        if not use_loop:
            out = self.render_fused(cond_feat.detach(), 1, N, rays_o=rays_o, rays_d=rays_d, bg_color=bg_color, dt_gamma=dt_gamma,
                                    max_steps=max_steps, T_thresh=T_thresh, precision=kwargs.get('precision'),
                                    want=('weights_sum', 'n_samples', 'counters', 'term_hist', 'term_slot'))
            results['depth_map'] = out['depth_map'].view(*prefix)
            results['rgb_map'] = out['rgb_map'].view(*prefix, 3)
            results['weights_sum_eval'] = out['weights_sum']
            results['n_samples'] = out['n_samples']
            results['term_hist'] = out['term_hist']
            results['term_slot'] = out['term_slot']
            self.last_counters = out['counters']
            return results
        nears, fars = raymarching.near_far_from_aabb(rays_o, rays_d, self.aabb_train if self.training else self.aabb_infer, self.min_near)
        nears, fars = nears.detach(), fars.detach()
        if self.training:
            counter = self.step_counter[self.local_step % 16]
            counter.zero_()
            self.local_step += 1
            xyzs, dirs, deltas, rays = raymarching.march_rays_train(rays_o, rays_d, self.bound, self.density_bitfield, self.cascade,
                                                                    self.grid_size, nears, fars, counter, self.mean_count, perturb, 128,
                                                                    force_all_rays, dt_gamma, max_steps)
            sigmas, rgbs, ambient = self(xyzs, dirs, cond_feat, ind_code)
            sigmas = self.density_scale * sigmas
            weights_sum, ambient_sum, depth, image = raymarching.composite_rays_train(sigmas, rgbs, ambient.abs().sum(-1), deltas, rays)
            results['weights_sum'] = weights_sum
            results['ambient'] = ambient_sum
        else:
            weights_sum, depth, image = self._render_head_loop(rays_o, rays_d, nears, fars, cond_feat, ind_code, dt_gamma, max_steps,
                                                               T_thresh, perturb, field=kwargs.get('loop_field', 'torch'))
        if bg_color is None:
            bg_color = 1
        image = image + (1 - weights_sum).unsqueeze(-1) * bg_color
        image = image.view(*prefix, 3).clamp(0, 1)
        depth = torch.clamp(depth - nears, min=0) / (fars - nears)
        results['depth_map'] = depth.view(*prefix)
        results['rgb_map'] = image
        return results


class RADNeRF(NeRFRenderer):
    """radnerf.py:11-130"""

    def __init__(self, hparams):
        super().__init__(hparams)
        self.hparams = hparams
        self.cond_in_dim = {'esperanto': 44, 'deepspeech': 29, 'idexp_lm3d_normalized': 68 * 3}.get(hparams['cond_type'])
        if self.cond_in_dim is None:
            raise NotImplementedError()
        self.cond_out_dim = hparams['cond_out_dim']
        self.cond_win_size = hparams['cond_win_size']
        self.smo_win_size = hparams['smo_win_size']
        self.cond_prenet = AudioNet(self.cond_in_dim, self.cond_out_dim, win_size=self.cond_win_size)
        self.with_att = hparams['with_att']
        if self.with_att:
            self.cond_att_net = AudioAttNet(self.cond_out_dim, seq_len=self.smo_win_size)
        self.grid_type = hparams['grid_type']
        self.grid_interpolation_type = hparams['grid_interpolation_type']
        self.position_embedder, self.position_embedding_dim = get_encoder(
            self.grid_type, input_dim=3, num_levels=16, level_dim=2, base_resolution=16, log2_hashmap_size=hparams['log2_hashmap_size'],
            desired_resolution=hparams['desired_resolution'] * self.bound, interpolation=self.grid_interpolation_type)
        self.num_layers_ambient = hparams['num_layers_ambient']
        self.hidden_dim_ambient = hparams['hidden_dim_ambient']
        self.ambient_out_dim = hparams['ambient_out_dim']
        self.ambient_net = MLP(self.position_embedding_dim + self.cond_out_dim, self.ambient_out_dim, self.hidden_dim_ambient, self.num_layers_ambient)
        self.ambient_embedder, self.ambient_embedding_dim = get_encoder(
            self.grid_type, input_dim=hparams['ambient_out_dim'], num_levels=16, level_dim=2, base_resolution=16,
            log2_hashmap_size=hparams['log2_hashmap_size'], desired_resolution=hparams['desired_resolution'], interpolation=self.grid_interpolation_type)
        self.num_layers_sigma = hparams['num_layers_sigma']
        self.hidden_dim_sigma = hparams['hidden_dim_sigma']
        self.geo_feat_dim = hparams['geo_feat_dim']
        self.sigma_net = MLP(self.position_embedding_dim + self.ambient_embedding_dim, 1 + self.geo_feat_dim, self.hidden_dim_sigma, self.num_layers_sigma)
        self.num_layers_color = hparams['num_layers_color']
        self.hidden_dim_color = hparams['hidden_dim_color']
        self.direction_embedder, self.direction_embedding_dim = get_encoder('spherical_harmonics')
        self.color_net = MLP(self.direction_embedding_dim + self.geo_feat_dim + self.individual_embedding_dim, 3, self.hidden_dim_color, self.num_layers_color)
        # training-time MLP backend (cond_encoder.MLP.backend): 'tc' = the gf_tl_* tcgen05 operators, 'torch' = library GEMMs under autograd
        backend = hparams.get('train_mlp_backend', os.environ.get('GF_TRAIN_MLP', 'torch'))
        for net in (self.ambient_net, self.sigma_net, self.color_net):
            net.backend = backend

    def cal_cond_feat(self, cond):
        cond_feat = self.cond_prenet(cond)
        if self.with_att:
            cond_feat = self.cond_att_net(cond_feat)
        return cond_feat

    def _trunk(self, position, cond_feat):
        # the MLPs take the pieces of their concatenated inputs (radnerf.py:79,90,99 build them with repeat + cat); the library backend concatenates,
        # the tensor-core backend packs the pieces straight into its tile layout and keeps the per-frame rows as broadcasts
        cond_feat = cond_feat.view(1, -1).expand(position.shape[0], -1)
        pos_feat = self.position_embedder(position, bound=self.bound)
        ambient_logit = self.ambient_net([pos_feat, cond_feat]).float()
        ambient_pos = torch.tanh(ambient_logit)
        ambient_feat = self.ambient_embedder(ambient_pos, bound=1)
        h = self.sigma_net([pos_feat, ambient_feat])
        return trunc_exp(h[..., 0]), h[..., 1:], ambient_pos

    def forward(self, position, direction, cond_feat, individual_code):
        sigma, geo_feat, ambient_pos = self._trunk(position, cond_feat)
        parts = [self.direction_embedder(direction), geo_feat]
        if individual_code is not None:
            parts.append(individual_code.view(1, -1).expand(position.shape[0], -1))
        color = torch.sigmoid(self.color_net(parts))
        return sigma, color, ambient_pos

    def density(self, position, cond_feat, e=None):
        sigma, geo_feat, _ = self._trunk(position, cond_feat)
        return {'sigma': sigma, 'geo_feat': geo_feat}

    def _fused_supported(self):
        h = self.hidden_dim_ambient
        return (self.num_layers_ambient == 3 and self.num_layers_sigma == 3 and self.num_layers_color == 2 and
                h == self.hidden_dim_sigma == self.hidden_dim_color and h in (64, 128) and self.ambient_out_dim == 2 and
                self.geo_feat_dim % 8 == 0 and 8 <= self.geo_feat_dim <= 128 and self.density_scale == 1)

    def _model_desc(self, torso=False):
        if not self._fused_supported():
            raise RuntimeError("this RADNeRF configuration is outside the fused renderer's envelope (use reference_loop=True)")
        d = GfModelDesc()
        keep = []

        def dev(t, dtype=torch.float32):
            t = t.detach()
            if t.dtype != dtype or not t.is_contiguous():
                t = t.to(dtype).contiguous()
            keep.append(t)
            return t.data_ptr()

        d.bound, d.cascade, d.grid_size, d.min_near = float(self.bound), self.cascade, self.grid_size, float(self.min_near)
        d.aabb = (c_f32 * 6)(*self.aabb_infer.detach().cpu().tolist())
        pe, ae = self.position_embedder, self.ambient_embedder
        d.gridtype, d.interp = pe.gridtype_id, pe.interp_id
        d.hidden_dim, d.cond_dim, d.ind_dim = self.hidden_dim_ambient, self.cond_out_dim, self.individual_embedding_dim
        d.density_bitfield = dev(self.density_bitfield, torch.uint8)
        d.pos_embeddings, d.pos_offsets = dev(pe.embeddings), dev(pe.offsets, torch.int32)
        d.pos_S, d.pos_H = float(np.log2(pe.per_level_scale)), pe.base_resolution
        d.amb_embeddings, d.amb_offsets = dev(ae.embeddings), dev(ae.offsets, torch.int32)
        d.amb_S, d.amb_H = float(np.log2(ae.per_level_scale)), ae.base_resolution
        d.ambient_w0, d.ambient_w1, d.ambient_w2 = [dev(l.weight) for l in self.ambient_net.net]
        d.sigma_w0, d.sigma_w1, d.sigma_w2 = [dev(l.weight) for l in self.sigma_net.net]
        d.color_w0, d.color_w1 = [dev(l.weight) for l in self.color_net.net]
        d.geo_feat_dim = self.geo_feat_dim
        if self.individual_embedding_dim > 0:
            d.ind_code = dev(self.individual_embeddings[0])
        return d, keep


class RADNeRFTorso(RADNeRF):
    """radnerf_torso.py:17-241"""

    def __init__(self, hparams):
        super().__init__(hparams)
        self.register_buffer('density_grid_torso', torch.zeros([self.grid_size ** 2]))
        self.mean_density_torso = 0
        self.density_thresh_torso = hparams['density_thresh_torso']
        self.torso_shrink = hparams.get('torso_shrink', 0.8)
        self.torso_head_aware = hparams.get('torso_head_aware', False)
        self.torso_individual_embedding_num = hparams['individual_embedding_num']
        self.torso_individual_embedding_dim = hparams['torso_individual_embedding_dim']
        if self.torso_individual_embedding_dim > 0:
            self.torso_individual_codes = nn.Parameter(torch.randn(self.torso_individual_embedding_num, self.torso_individual_embedding_dim) * 0.1)
        self.torso_pose_embedder, self.pose_embedding_dim = get_encoder('frequency', input_dim=6, multires=4)
        self.torso_deform_pos_embedder, self.torso_deform_pos_dim = get_encoder('frequency', input_dim=2, multires=10)
        self.torso_embedder, self.torso_in_dim = get_encoder('tiledgrid', input_dim=2, num_levels=16, level_dim=2, base_resolution=16,
                                                             log2_hashmap_size=16, desired_resolution=2048)
        deform_in = self.torso_deform_pos_dim + self.pose_embedding_dim + self.torso_individual_embedding_dim
        canon_in = self.torso_in_dim + deform_in
        if self.torso_head_aware:
            self.head_color_weights_encoder = nn.Sequential(nn.Linear(4, 16), nn.LeakyReLU(0.02, True), nn.Linear(16, 32),
                                                            nn.LeakyReLU(0.02, True), nn.Linear(32, 16))
            deform_in += 16
            canon_in += 16
        self.torso_deform_net = MLP(deform_in, 2, 64, 3)
        self.torso_canonicial_net = MLP(canon_in, 4, 32, 3)

    def forward_torso(self, x, poses, c=None, image=None, weights_sum=None):
        """radnerf_torso.py:51-84"""
        x = x * self.torso_shrink
        enc_pose = self.torso_pose_embedder(poses)
        enc_x = self.torso_deform_pos_embedder(x)
        parts = [enc_x, enc_pose.repeat(x.shape[0], 1)]
        if c is not None:
            parts.append(c.view(1, -1).repeat(x.shape[0], 1))
        h = torch.cat(parts, dim=-1)
        if self.torso_head_aware:
            if image is None:
                image = torch.zeros([x.shape[0], 3], dtype=h.dtype, device=h.device)
                weights_sum = torch.zeros([x.shape[0], 1], dtype=h.dtype, device=h.device)
            h = torch.cat([h, self.head_color_weights_encoder(torch.cat([image, weights_sum], dim=-1))], dim=-1)
        dx = self.torso_deform_net(h)
        x = (x + dx).clamp(-1, 1).float()
        x = self.torso_embedder(x, bound=1)
        h = self.torso_canonicial_net(torch.cat([x, h], dim=-1))
        return torch.sigmoid(h[..., :1]), torch.sigmoid(h[..., 1:]), dx

    def _fused_supported(self):
        return super()._fused_supported() and not self.torso_head_aware and self.torso_individual_embedding_dim <= 10

    def _model_desc(self):
        d, keep = super()._model_desc()

        def dev(t, dtype=torch.float32):
            t = t.detach()
            if t.dtype != dtype or not t.is_contiguous():
                t = t.to(dtype).contiguous()
            keep.append(t)
            return t.data_ptr()

        te = self.torso_embedder
        d.has_torso = 1
        d.density_grid_torso = dev(self.density_grid_torso)
        d.density_thresh_torso = float(min(self.density_thresh_torso, self.mean_density_torso))    # radnerf_torso.py:166
        d.torso_shrink = float(self.torso_shrink)
        d.torso_embeddings, d.torso_offsets = dev(te.embeddings), dev(te.offsets, torch.int32)
        d.torso_S, d.torso_H = float(np.log2(te.per_level_scale)), te.base_resolution
        d.torso_deform_w0, d.torso_deform_w1, d.torso_deform_w2 = [dev(l.weight) for l in self.torso_deform_net.net]
        d.torso_canon_w0, d.torso_canon_w1, d.torso_canon_w2 = [dev(l.weight) for l in self.torso_canonicial_net.net]
        d.torso_ind_dim = self.torso_individual_embedding_dim
        if self.torso_individual_embedding_dim > 0:
            d.torso_ind_code = dev(self.torso_individual_codes[0])
        return d, keep

    def _tensors_key(self):
        return super()._tensors_key() + (float(self.mean_density_torso),)

    def render(self, rays_o, rays_d, cond, bg_coords, poses, index=0, dt_gamma=0, bg_color=None, perturb=False, force_all_rays=False,
               max_steps=1024, T_thresh=1e-4, **kwargs):
        prefix = rays_o.shape[:-1]
        rays_o = rays_o.contiguous().view(-1, 3)
        rays_d = rays_d.contiguous().view(-1, 3)
        bg_coords = bg_coords.contiguous().view(-1, 2)
        N = rays_o.shape[0]
        dev = rays_o.device
        results = {}
        use_loop = self.training or perturb or kwargs.get('reference_loop', False) or not self._fused_supported()
        if not use_loop:
            with torch.no_grad():
                cond_feat = self.cal_cond_feat(cond)
            out = self.render_fused(cond_feat, 1, N, rays_o=rays_o, rays_d=rays_d, bg_color=bg_color, bg_coords=bg_coords,
                                    torso_pose=poses, dt_gamma=dt_gamma, max_steps=max_steps, T_thresh=T_thresh,
                                    precision=kwargs.get('precision'),
                                    want=('weights_sum', 'torso_alpha_map', 'torso_rgb_map', 'n_samples', 'counters', 'term_hist', 'term_slot'))
            results['torso_alpha_map'] = out['torso_alpha_map'].view(N, 1)
            results['torso_rgb_map'] = out['torso_rgb_map'].view(1, N, 3) if len(prefix) == 2 else out['torso_rgb_map']
            results['depth_map'] = out['depth_map'].view(*prefix)
            results['rgb_map'] = out['rgb_map'].view(*prefix, 3)
            results['weights_sum_eval'] = out['weights_sum']
            results['n_samples'] = out['n_samples']
            results['term_hist'] = out['term_hist']
            results['term_slot'] = out['term_slot']
            self.last_counters = out['counters']
            return results
        # ---- reference structure (radnerf_torso.py:92-196) on our ops ----
        with torch.no_grad():
            nears, fars = raymarching.near_far_from_aabb(rays_o, rays_d, self.aabb_train if self.training else self.aabb_infer, self.min_near)
            cond_feat = self.cal_cond_feat(cond)
            ind_code = self._ind_code(index)
            if self.training:
                counter = self.step_counter[self.local_step % 16]
                counter.zero_()
                self.local_step += 1
                xyzs, dirs, deltas, rays = raymarching.march_rays_train(rays_o, rays_d, self.bound, self.density_bitfield, self.cascade,
                                                                        self.grid_size, nears, fars, counter, self.mean_count, perturb,
                                                                        128, force_all_rays, dt_gamma, max_steps)
                sigmas, rgbs, ambient = self(xyzs, dirs, cond_feat, ind_code)
                weights_sum, ambient_sum, depth, image = raymarching.composite_rays_train(self.density_scale * sigmas, rgbs,
                                                                                          ambient.abs().sum(-1), deltas, rays)
                results['weights_sum'] = weights_sum
                results['ambient'] = ambient_sum
            else:
                weights_sum, depth, image = self._render_head_loop(rays_o, rays_d, nears, fars, cond_feat, ind_code, dt_gamma, max_steps,
                                                                   T_thresh, perturb, field=kwargs.get('loop_field', 'torch'))
            if bg_color is None:
                bg_color = 1
        if self.torso_individual_embedding_dim > 0:
            code = self.torso_individual_codes[index] if self.training else self.torso_individual_codes[0]
        else:
            code = None
        thresh = min(self.density_thresh_torso, self.mean_density_torso)
        occupancy = F.grid_sample(self.density_grid_torso.view(1, 1, self.grid_size, self.grid_size), bg_coords.view(1, -1, 1, 2),
                                  align_corners=True).view(-1)
        mask = occupancy > thresh
        torso_alpha = torch.zeros([N, 1], device=dev)
        torso_color = torch.zeros([N, 3], device=dev)
        if mask.any():
            if self.torso_head_aware and random.random() < 0.5:
                a, c, deform = self.forward_torso(bg_coords[mask], poses, code, image[mask], weights_sum.unsqueeze(-1)[mask])
            else:
                a, c, deform = self.forward_torso(bg_coords[mask], poses, code)
            torso_alpha[mask] = a.float()
            torso_color[mask] = c.float()
            results['deform'] = deform
        bg_color = torso_color * torso_alpha + bg_color * (1 - torso_alpha)
        results['torso_alpha_map'] = torso_alpha
        results['torso_rgb_map'] = bg_color
        image = image + (1 - weights_sum).unsqueeze(-1) * bg_color
        results['rgb_map'] = image.view(*prefix, 3).clamp(0, 1)
        results['depth_map'] = (torch.clamp(depth - nears, min=0) / (fars - nears)).view(*prefix)
        return results

    @torch.no_grad()
    def update_extra_state(self, decay=0.95, S=128):
        """radnerf_torso.py:200-241 (torso 2D occupancy grid only): alpha of the torso field at one jittered point per cell of the
        H x H image-plane grid, 5x5 max-dilation, EMA-max.  The whole grid (16 K cells) is one field call."""
        G, dev = self.grid_size, self.density_bitfield.device
        rand_idx = random.randint(0, self.poses.shape[0] - 1)
        pose = convert_poses(self.poses[[rand_idx]]).to(dev)
        code = self.torso_individual_codes[[rand_idx]] if self.torso_individual_embedding_dim > 0 else None
        ar = torch.arange(G, dtype=torch.int32, device=dev)
        cell = torch.stack(torch.meshgrid(ar, ar, indexing='ij'), dim=-1).view(-1, 2)
        half_cell = 1 / G
        xys = (cell.float() * (2.0 / (G - 1)) - 1.0) * (1 - half_cell)
        xys = xys + (torch.rand_like(xys) * 2 - 1) * half_cell
        alphas, _, _ = self.forward_torso(xys, pose, code)
        fresh = torch.zeros_like(self.density_grid_torso)
        fresh[(cell[:, 1] * G + cell[:, 0]).long()] = alphas.squeeze(1).float()          # x/y transposed, as the reference stores it
        fresh = F.max_pool2d(fresh.view(1, 1, G, G), kernel_size=5, stride=1, padding=2).view(-1)
        self.density_grid_torso = torch.maximum(self.density_grid_torso * decay, fresh)
        self.mean_density_torso = torch.mean(self.density_grid_torso).item()
        self.invalidate_fused()
