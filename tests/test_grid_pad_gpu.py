"""Padded grid images of the fused renderer (GridLevels::pad).

gf_model_create copies the position and ambient tables into images in which a wrapping tiled level (the reference's
corner index `(x + y*sy + z*sz) % hsize` changes some index) is followed by a copy of its first 1 + sy + sz entries, so the
field kernels read a cell's corners as rows of adjacent entries from the masked base index.  These tests check, on the
headline model (bound 4), the May model (bound 1) and a hash-grid model, that sampled points really read the pads, that the
gathers still return the reference's corner values, and that an in-place grid edit reaches a rebuilt image.
"""
import numpy as np
import pytest
import torch

import scenes

pytestmark = pytest.mark.gpu

HASH_P1, HASH_P2 = 2654435761, 805459861     # gridencoder.cu:54
M = 1 << 20

MODELS = {
    "headline": dict(torso=False, bitfield='F', seed=0, sigma_scale=0.25, bound=4),
    "may": dict(torso=False, bitfield='S', seed=0),
    "hash": dict(torso=False, bitfield='S', seed=2, grid_type='hashgrid'),
}


@pytest.fixture(scope="module", params=sorted(MODELS))
def model(request):
    from geneface_b200 import synthetic
    m, hp = synthetic.build_model(**MODELS[request.param])
    return request.param, m


def levels(enc, D, dev):
    """Per-level geometry of a grid as gf_model_create derives it (scale with the device's exp2, stride loop of get_grid_index)."""
    off = enc.offsets.cpu().numpy().astype(np.int64)
    S = np.float32(np.log2(enc.per_level_scale))
    e2 = torch.exp2(torch.tensor([np.float32(l) * S for l in range(16)], dtype=torch.float32, device=dev)).cpu().double()
    out = []
    for l in range(16):
        scale = float(np.float32(float(e2[l]) * enc.base_resolution - 1.0))        # one rounding, as __fmaf_rn
        res = int(np.ceil(scale)) + 1
        hs = int(off[l + 1] - off[l])
        R, stride, sy, sz = res + 1, res + 1, 0, 0
        if stride <= hs:
            sy, stride = stride, stride * R
        if D == 3 and stride <= hs:
            sz, stride = stride, stride * R
        hashed = enc.gridtype_id == 0 and stride > hs
        wraps = not hashed and res * (1 + sy + sz) >= hs
        out.append(dict(scale=scale, hs=hs, off=int(off[l]), sy=sy, sz=sz, hashed=hashed, pad=1 + sy + sz if wraps else 0))
    return out


def ref_level(emb64, lv, u, D):
    """One level's 2 channels at unit coordinates u [M, D] (float32), trilinear / bilinear in float64 with the reference's index rule.
    Also returns, per sample, whether the masked base index plus the largest corner offset reaches past hsize (the sample reads the pad)."""
    pos = (u.double() * lv['scale'] + 0.5).float()            # exact product + 0.5, rounded once: ffma
    g = torch.floor(pos)
    f = (pos - g).double()
    g = g.long()
    hs = lv['hs']
    strides = [1, lv['sy'], lv['sz']][:D]
    acc = torch.zeros(u.shape[0], 2, dtype=torch.float64, device=u.device)
    for c in range(1 << D):
        bit = [(c >> d) & 1 for d in range(D)]
        pc = [g[:, d] + bit[d] for d in range(D)]
        if lv['hashed']:
            idx = pc[0] & 0xFFFFFFFF
            for d, p in zip(range(1, D), (HASH_P1, HASH_P2)):
                idx = idx ^ ((pc[d] * p) & 0xFFFFFFFF)
        else:
            idx = sum(pc[d] * strides[d] for d in range(D))
        idx = idx % hs
        w = torch.ones_like(f[:, 0])
        for d in range(D):
            w = w * (f[:, d] if bit[d] else 1.0 - f[:, d])
        acc += w[:, None] * emb64[lv['off'] + idx]
    base = sum(g[:, d] * strides[d] for d in range(D)) % hs if not lv['hashed'] else None
    reads_pad = (base + 1 + lv['sy'] + lv['sz'] >= hs) if lv['pad'] else torch.zeros_like(g[:, 0], dtype=torch.bool)
    return acc, reads_pad


def test_pads_are_read_and_gathers_match_the_reference_index(model):
    from geneface_b200 import _lib
    name, m = model
    dev = torch.device('cuda')
    bound = float(m.bound)
    gen = torch.Generator().manual_seed(11)
    xyz = ((torch.rand(M, 3, generator=gen) * 2 - 1) * bound).to(dev)
    amb = (torch.rand(M, 2, generator=gen) * 2 - 1).to(dev)
    out = torch.empty(M, 2, device=dev)
    L = _lib.lib()
    _lib.check(L.gf_gather_probe(m.gf_model(), _lib.ptr(xyz), _lib.ptr(amb), M, _lib.ptr(out), _lib.stream_ptr()))
    torch.cuda.synchronize()

    inv2b = np.float32(np.float32(0.5) / np.float32(bound))
    u3 = (xyz + np.float32(bound)) * float(inv2b)             # float32 ops, as the probe
    u2 = (amb + 1.0) * 0.5
    ref = torch.zeros(M, 2, dtype=torch.float64, device=dev)
    mag = torch.zeros(M, dtype=torch.float64, device=dev)
    wrapping = 0
    for enc, D, u in ((m.position_embedder, 3, u3), (m.ambient_embedder, 2, u2)):
        emb64 = enc.embeddings.detach().double()
        for l, lv in enumerate(levels(enc, D, dev)):
            f, reads_pad = ref_level(emb64, lv, u, D)
            ref += f
            mag += f.abs().sum(1)
            if lv['pad']:
                wrapping += 1
                frac = reads_pad.double().mean().item()
                print(f"{name} D={D} level {l}: pad {lv['pad']}, {100 * frac:.2f} % of the points read it")
                assert frac > 0, f"{name} D={D} level {l} wraps but no sampled point reads its pad"
    if name == "hash":
        assert wrapping == 0, "a hash grid has only never-wrapping dense levels and hashed levels"
    else:
        assert wrapping > 0, "a tiled model is expected to have wrapping levels"
    err = (out.double() - ref).abs().max(1).values
    tol = 1e-5 * torch.clamp(mag, min=1.0)
    worst = (err / tol).max().item()
    print(f"{name}: gather probe vs float64 reference, worst err / tol {worst:.3f}")
    assert bool((err <= tol).all()), f"{name}: {(err > tol).sum().item()} samples differ from the reference's corner values"


def test_tensor_core_field_matches_fp32_field(model):
    name, m = model
    bound = float(m.bound)
    xyz, d = scenes.field_samples(20000, seed=25, bound=bound)
    xyz, d = torch.from_numpy(xyz).cuda(), torch.from_numpy(d).cuda()
    cond_feat = torch.randn(64, generator=torch.Generator().manual_seed(3)).cuda()
    s32, c32, _ = m.field_forward(xyz, d, cond_feat, precision='fp32')
    s16, c16, _ = m.field_forward(xyz, d, cond_feat, precision='fp16')
    rel_sigma = ((s16 - s32).abs() / s32).cpu().numpy()
    print(f"{name}: tc sigma rel err p99 {np.percentile(rel_sigma, 99):.2e}; rgb abs max {(c16 - c32).abs().max().item():.2e}")
    assert np.percentile(rel_sigma, 99) < 2e-2 and (c16 - c32).abs().max().item() < 5e-3


def test_in_place_grid_edit_reaches_the_rebuilt_model():
    """An edit of both grid tables under no_grad bumps their version: render_fused(check_weights=True) rebuilds the model and with it the
    padded images, so the frame equals a freshly built model's frame bit for bit."""
    from geneface_b200 import synthetic
    Himg = 64

    def frame(m, hp):
        fi = synthetic.frame_inputs(Himg, Himg)
        with torch.no_grad():
            cf = m.cal_cond_feat(fi['cond'])
        o = m.render_fused(cf, Himg, Himg, pose=fi['pose'][0], intrinsics=fi['intrinsics'], bg_color=fi['bg_color'], dt_gamma=hp['dt_gamma'],
                           max_steps=hp['max_steps'], precision='fp16', want=('weights_sum', 'n_samples'))
        return {k: v.clone() for k, v in o.items() if torch.is_tensor(v)}

    def edit(m):
        g = torch.Generator().manual_seed(5)
        with torch.no_grad():
            for enc in (m.position_embedder, m.ambient_embedder):
                enc.embeddings.add_((torch.rand(enc.embeddings.shape, generator=g) - 0.5).to(enc.embeddings.device))

    m, hp = synthetic.build_model(**MODELS["may"])
    before = frame(m, hp)
    edit(m)
    after = frame(m, hp)
    fresh_m, _ = synthetic.build_model(**MODELS["may"])
    edit(fresh_m)
    fresh = frame(fresh_m, hp)
    assert not torch.equal(before['rgb_map'], after['rgb_map']), "the grid edit did not change the frame"
    for k in fresh:
        assert torch.equal(after[k], fresh[k]), f"{k}: the edited model's frame differs from a freshly built model's"
