"""Frame-level parity against the REFERENCE ITSELF (SURVEY.md section 8c): the unmodified `RADNeRF(Torso).render()` of
modules/radnerfs, imported from the byte-for-byte mirror oracle/_ref/pyref on the compiled unmodified extensions.

  * tests/golden/frame_{may,may_torso,b4}.npz were written by oracle/gen_golden_frames.py on a B200 (reference eval / fp32);
  * CPU  : the numpy/C oracle (oracle/field.py + oracle/gf_oracle.c) must reproduce them  -> pins the oracle at MODEL level;
  * GPU  : `gf_render_frame` (fp32 and fp16 tensor-core precision) must reproduce them, and the benchmark configuration itself
           (bound 4, 3 cascades, 128 steps, fp16) is compared with the reference's render() on identical rays at 128x128 and 512x64:
           live where oracle/_ref is built, else against its outputs recorded under tests/golden/reference/ (tests/refgold.py).

Bars (north_star): rgb / depth / weights within 1e-3 relative per pixel (abs floor 1e-5), per-ray sample counts and the host
loop's (n_alive, n_step) sequence exact.
"""
import os

import numpy as np
import pytest
import torch

import refgold

REL, ABS = 1e-3, 1e-5
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
NAMES = ("may", "may_torso", "b4")


@pytest.fixture(autouse=True)
def fp32_without_tf32():
    """The reference computes in plain fp32 (oracle/ref_model.py turns TF32 off when it loads it); our side of every comparison
    runs under the same arithmetic whether the reference's outputs are live or recorded."""
    saved = torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
    yield
    torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = saved


def scaled_err(a, b, abs_=ABS):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    both_nan = np.isnan(a) & np.isnan(b)
    return np.where(both_nan, 0.0, np.abs(a - b) / (abs_ + np.abs(b)))


def assert_close(a, b, rel=REL, what="", allow_frac=0.0):
    e = scaled_err(a, b)
    # |a-b| <= abs + rel*|b|  <=>  e <= (abs + rel|b|)/(abs+|b|); use the looser-but-simple e <= rel*(1+abs/(abs+|b|)) form exactly:
    b64 = np.abs(np.asarray(b, np.float64))
    ok = e * (ABS + b64) <= ABS + rel * b64
    bad = (~ok).mean()
    assert bad <= allow_frac, f"{what}: {int((~ok).sum())} of {ok.size} outside tolerance, worst scaled err {np.nanmax(e):.3e}"
    return float(np.nanmax(e))


def load_golden(name):
    p = os.path.join(GOLDEN, f"frame_{name}.npz")
    if not os.path.exists(p):
        pytest.fail(f"{p} missing: generate it with oracle/gen_golden_frames.py on the GPU box")
    g = dict(np.load(p))
    N = int(g["H"]) ** 2
    if g["rays_o"].shape[0] == 1:
        g["rays_o"] = np.ascontiguousarray(np.broadcast_to(g["rays_o"], (N, 3)))
    return g


def scene(name, device):
    from oracle import gen_golden_frames as G
    model, hp, fi, cfg = G.scene_model(name, device=device)
    return model, hp, fi, cfg, G.state_checksum(model.state_dict())


def term_iter_of(term_slot, trace):
    """Host-loop iteration in which the reference marks a ray with termination slot k dead: the iteration whose offered slots
    (S_i, S_i + n_step_i] contain k; -1 for k == 0 (alive) or k > S_total (the loop ended before it could notice)."""
    ends = np.cumsum([s for _, s in trace])                       # slots offered after each iteration
    k = np.asarray(term_slot, np.int64)
    it = np.searchsorted(ends, k, side="left")                    # first i with ends[i] >= k
    return np.where((k <= 0) | (k > (ends[-1] if len(ends) else 0)), -1, it).astype(np.int32)


def replay_schedule(hist, N, max_steps):
    """The reference host loop's (n_alive, n_step) sequence from the fused path's termination histogram (DESIGN.md section 3)."""
    terminated_by = np.concatenate([[0], np.cumsum(hist[1:])])
    trace, step, offered = [], 0, 0
    while step < max_steps:
        n_alive = N - int(terminated_by[min(offered, len(terminated_by) - 1)])
        if n_alive <= 0:
            break
        n_step = max(min(N // n_alive, 8), 1)
        trace.append((n_alive, n_step))
        offered += n_step
        step += n_step
    return trace


# ------------------------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("name", NAMES)
def test_cpu_oracle_reproduces_the_reference_frames(name):
    """oracle/field.py (numpy field + host loop + torso) on oracle/gf_oracle.c (march / composite / encoders) vs the golden
    frames rendered by the reference's own render()."""
    from geneface_b200 import synthetic
    from oracle import field as OF
    g = load_golden(name)
    model, hp, fi, cfg, csum = scene(name, "cpu")
    assert abs(csum - float(g["state_checksum"])) <= 1e-9 * abs(csum), "synthetic weights differ from the ones the golden was rendered with"
    sd = synthetic.state_to_numpy(model)
    fo = OF.FieldOracle(sd, bound=float(cfg["bound"]))
    cf = OF.cal_cond_feat(sd, fi["cond"].numpy())
    trace = []
    term_iter = np.full(g["rays_d"].shape[0], -1, np.int32)
    ws, depth, img, nears, fars, ns = OF.render_head(fo, sd, g["rays_o"], g["rays_d"], cf, sd["density_bitfield"], model.cascade, 128,
                                                    sd["aabb_infer"], hp["min_near"], float(g["dt_gamma"]), int(g["max_steps"]), trace=trace,
                                                    term_iter=term_iter)
    bg = fi["bg_color"][0].numpy()
    if cfg["torso"]:
        bg, t_alpha, _, mask = OF.render_torso_mix(OF.TorsoOracle(sd), sd, g["bg_coords"], g["poses6"][0], bg, img, ws)
        assert_close(t_alpha[:, 0], g["torso_alpha_map"], what="torso_alpha_map")
        assert_close(bg, g["torso_rgb_map"], what="torso_rgb_map")
    img_f, depth_f = OF.finish(img, ws, depth, nears, fars, bg)
    # integer outputs: per-ray termination iteration and the loop schedule.  expf (libm) vs __expf (MUFU.EX2) can move a ray
    # across the T < 1e-4 threshold by one sample; the schedule is compared only when no ray did.
    mism = term_iter != g["term_iter"]
    assert mism.mean() <= 2e-3, f"{int(mism.sum())} rays differ in termination iteration"
    if not mism.any():
        assert [tuple(t) for t in g["trace"].tolist()] == trace
    good = ~mism
    assert_close(ws[good], g["weights_sum"][good], what="weights_sum")
    assert_close(img_f[good], g["rgb_map"][good], what="rgb_map")
    assert_close(depth_f[good], g["depth_map"][good], what="depth_map")


def test_reference_mirror_is_importable_and_unmodified():
    """oracle/_ref/pyref holds the reference's Python byte for byte (checked where the reference tree exists) and imports with the
    six documented stubs; the model constructs and strictly loads our synthetic state_dict (same parameter / buffer names).  From a
    clean checkout our state_dict is compared with the reference model's recorded inventory."""
    from oracle import build_ref, ref_model
    from geneface_b200 import synthetic
    model, hp = synthetic.build_model(torso=True, bitfield='S', seed=0, device='cpu')
    R = refgold.Reference("mirror_inventory", ref_model.available())
    if R.live:
        if os.path.isdir(build_ref.REF):
            for rel in build_ref.PY_FILES:
                a = open(os.path.join(build_ref.REF, rel), "rb").read()
                b = open(os.path.join(build_ref.OUT, "pyref", rel), "rb").read()
                assert a == b, f"{rel} differs from the reference"
        ref = ref_model.build(model.state_dict(), hp, torso=True, device='cpu')
        assert type(ref).__module__ == "modules.radnerfs.radnerf_torso"
        R.put("inventory", np.array(sorted(f"{k}{tuple(v.shape)}" for k, v in ref.state_dict().items())))
        R.put("n_params", np.int64(sum(p.numel() for p in ref.parameters())))
    assert np.array_equal(np.array(sorted(f"{k}{tuple(v.shape)}" for k, v in model.state_dict().items())), R["inventory"])
    assert int(R["n_params"]) == 4344011 == sum(p.numel() for p in model.parameters())


# ------------------------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "fp16"])
@pytest.mark.parametrize("name", NAMES)
def test_fused_frame_reproduces_the_reference_frames(name, precision):
    """gf_render_frame through the drop-in render() boundary on the golden's rays, both precisions."""
    g = load_golden(name)
    model, hp, fi, cfg, csum = scene(name, "cuda")
    assert abs(csum - float(g["state_checksum"])) <= 1e-9 * abs(csum)
    N = int(g["H"]) ** 2
    ro, rd = torch.from_numpy(g["rays_o"]).cuda().view(1, N, 3), torch.from_numpy(g["rays_d"]).cuda().view(1, N, 3)
    bgc = torch.from_numpy(g["bg_coords"]).cuda().view(1, N, 2)
    poses6 = torch.from_numpy(g["poses6"]).cuda()
    with torch.no_grad():
        res = model.render(ro, rd, fi["cond"], bgc, poses6, bg_color=fi["bg_color"], dt_gamma=float(g["dt_gamma"]), max_steps=int(g["max_steps"]),
                           precision=precision)
    torch.cuda.synchronize()
    gtrace = [tuple(t) for t in g["trace"].tolist()]
    mism = term_iter_of(res["term_slot"].cpu().numpy(), gtrace) != g["term_iter"]
    # fp32: bit-exact termination indices; fp16 operands may move a ray sitting exactly on the T < 1e-4 threshold by one sample
    assert mism.mean() <= (0 if precision == "fp32" else 1e-3), f"{int(mism.sum())} rays differ in termination iteration"
    if not mism.any():
        assert replay_schedule(res["term_hist"].cpu().numpy(), N, int(g["max_steps"])) == gtrace
    good = ~mism
    worst = {k: assert_close(res[k2].reshape(-1, *v.shape[1:]).cpu().numpy()[good], v[good], what=f"{k} ({precision})")
             for k, k2, v in (("rgb_map", "rgb_map", g["rgb_map"]), ("depth_map", "depth_map", g["depth_map"]),
                              ("weights_sum", "weights_sum_eval", g["weights_sum"]))}
    if cfg["torso"]:
        assert_close(res["torso_alpha_map"][:, 0].cpu().numpy(), g["torso_alpha_map"], what="torso_alpha_map")
        assert_close(res["torso_rgb_map"].view(-1, 3).cpu().numpy(), g["torso_rgb_map"], what="torso_rgb_map")
    print(f"{name} {precision}: worst scaled err", {k: f"{v:.2e}" for k, v in worst.items()})
    # frame egress (base_nerf_infer.py:97-101: (rgb * 255).astype(uint8), truncation): the RGB8 frame packed by k_finish equals the
    # truncated reference image, except where the reference value lies within 1e-3 (relative, the float bar) of a code boundary
    with torch.no_grad():
        cf = model.cal_cond_feat(fi["cond"])
        out = model.render_fused(cf, 1, N, rays_o=ro, rays_d=rd, bg_color=fi["bg_color"], bg_coords=bgc, torso_pose=poses6,
                                 dt_gamma=float(g["dt_gamma"]), max_steps=int(g["max_steps"]), precision=precision, want=("rgb8",))
    rgb8 = out["rgb8"].cpu().numpy().astype(np.int32)
    ref255 = g["rgb_map"].astype(np.float64) * 255.0
    code = np.floor(ref255).astype(np.int32)
    near = np.abs(ref255 - np.round(ref255)) <= 1e-3 * ref255 + 255e-5
    okpix = (rgb8 == code) | (near & (np.abs(rgb8 - code) <= 1))
    assert okpix[good].all(), f"rgb8: {int((~okpix[good]).sum())} channels differ from trunc(reference * 255)"


def _frame_rays(fi, H, W):
    from geneface_b200 import utils
    rays = utils.get_rays(fi["pose"], fi["intrinsics"], H, W)
    return rays, utils.get_bg_coords(H, W, "cuda"), fi["poses6"]


def _reference_render(name, model, hp, torso, fi, rays, bgc, poses6, dt_gamma, max_steps):
    """The reference's own render() on our rays: live where oracle/_ref is built, else its recorded outputs."""
    from oracle import ref_model
    R = refgold.Reference(name, ref_model.available())
    if R.live:
        ref = ref_model.build(model.state_dict(), hp, torso=torso)
        res = ref_model.render(ref, rays["rays_o"], rays["rays_d"], fi["cond"], bgc, poses6, fi["bg_color"], dt_gamma, max_steps)
        N = rays["rays_d"].reshape(-1, 3).shape[0]
        R.put("trace", res["trace"])
        for k in ("n_marched", "term_iter"):
            R.put(k, res[k])
        for k in ("rgb_map", "depth_map", "weights_sum") + (("torso_alpha_map", "torso_rgb_map") if torso else ()):
            R.put(k, res[k].reshape(N, -1).float())
    return R


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp16", "fp32"])
@pytest.mark.parametrize("H,W", [(128, 128), (512, 64)])
def test_headline_configuration_vs_the_reference_render(H, W, precision):
    """The BENCHMARKED configuration (bench.py: head+torso, bound=4, 3 cascades, all-ones bitfield, sigma_scale 0.25, dt_gamma 0,
    max_steps 128) at 128x128 and 512 high x 64 wide (focal length of the 512-pixel image), fp16 tensor-core and fp32 precision, against the reference's own render()
    on identical rays: every ray composites exactly 128 samples, the loop trace is 128 x (N, 1), floats within 1e-3."""
    from geneface_b200 import synthetic
    model, hp = synthetic.build_model(torso=True, bitfield='F', seed=0, sigma_scale=0.25, bound=4)
    fi = synthetic.frame_inputs(H, W)
    N = H * W
    rays, bgc, poses6 = _frame_rays(fi, H, W)
    R = _reference_render(f"headline_{H}x{W}", model, hp, True, fi, rays, bgc, poses6, 0.0, 128)
    assert R["trace"] == [(N, 1)] * 128 and int(R["n_marched"].min()) == 128 == int(R["n_marched"].max())
    with torch.no_grad():
        res = model.render(rays["rays_o"], rays["rays_d"], fi["cond"], bgc, poses6, bg_color=fi["bg_color"], dt_gamma=0.0, max_steps=128,
                           precision=precision)
    torch.cuda.synchronize()
    assert np.array_equal(res["n_samples"].cpu().numpy(), R["n_marched"])
    assert replay_schedule(res["term_hist"].cpu().numpy(), N, 128) == R["trace"]
    assert np.array_equal(term_iter_of(res["term_slot"].cpu().numpy(), R["trace"]), R["term_iter"])
    for k, k2 in (("rgb_map", "rgb_map"), ("depth_map", "depth_map"), ("weights_sum_eval", "weights_sum"),
                  ("torso_alpha_map", "torso_alpha_map"), ("torso_rgb_map", "torso_rgb_map")):
        w = assert_close(res[k].reshape(N, -1).cpu().numpy()[R.rows(k2)], R[k2], what=f"{k} {precision} {H}x{W}")
        print(f"headline {H}x{W} {precision} {k}: worst scaled err {w:.2e}")


@pytest.mark.gpu
@pytest.mark.parametrize("bitfield", ["S", "R"])
def test_may_torso_fp16_vs_the_reference_render(bitfield):
    """The reference's deployment configuration (May head+torso: bound 1, max_steps 16, dt_gamma 1/256) with early termination, in the
    DEFAULT fp16 precision of the product path, against the reference's own render(): schedule exact, floats within 1e-3."""
    from geneface_b200 import synthetic
    H = W = 128
    model, hp = synthetic.build_model(torso=True, bitfield=bitfield, seed=4)
    fi = synthetic.frame_inputs(H, W)
    N = H * W
    rays, bgc, poses6 = _frame_rays(fi, H, W)
    R = _reference_render(f"may_torso_{bitfield}", model, hp, True, fi, rays, bgc, poses6, hp["dt_gamma"], hp["max_steps"])
    with torch.no_grad():
        res = model.render(rays["rays_o"], rays["rays_d"], fi["cond"], bgc, poses6, bg_color=fi["bg_color"], dt_gamma=hp["dt_gamma"],
                           max_steps=hp["max_steps"], precision="fp16")
    torch.cuda.synchronize()
    mism = term_iter_of(res["term_slot"].cpu().numpy(), R["trace"]) != R["term_iter"]
    assert mism.mean() <= 1e-3, f"{int(mism.sum())} rays differ in termination iteration"
    if not mism.any():
        assert replay_schedule(res["term_hist"].cpu().numpy(), N, hp["max_steps"]) == R["trace"]
    good = ~mism
    for k, k2 in (("rgb_map", "rgb_map"), ("depth_map", "depth_map"), ("weights_sum_eval", "weights_sum")):
        rows = R.rows(k2)
        assert_close(res[k].reshape(N, -1).cpu().numpy()[rows][good[rows]], R[k2][good[rows]], what=f"{k} fp16 May torso {bitfield}")


def _per_ray(v):
    return v.reshape(-1, 3) if v.ndim > 1 and v.shape[-1] == 3 else v.reshape(-1)


@pytest.mark.gpu
def test_train_step_gradients_vs_the_reference_train_step():
    """BASELINE.json configs[4] / SURVEY.md section 8d config 5: ONE training step (march_rays_train -> field -> composite_rays_train ->
    MSE -> backward) of the drop-in model against the reference's own RADNeRF.render() in train mode + autograd on its compiled
    extensions: same 4096 rays, perturb off, force_all_rays (no sample budget, so both sides see every sample).  The image and EVERY
    parameter gradient (hash-grid tables via the privatised backward, MLPs, condition nets, individual codes) must agree within 1e-3 of
    the gradient's scale.  The recorded golden keeps each gradient's largest entries and a seeded sample of the rest."""
    from geneface_b200 import synthetic
    from oracle import ref_model
    H = W = 512
    model, hp = synthetic.build_model(torso=False, bitfield='S', seed=0)
    fi = synthetic.frame_inputs(H, W)
    g = torch.Generator(device='cuda').manual_seed(3)
    inds = torch.randint(0, H * W, [4096], device='cuda', generator=g)
    rays, bgc, poses6 = _frame_rays(fi, H, W)
    rays_o, rays_d = rays['rays_o'][:, inds].contiguous(), rays['rays_d'][:, inds].contiguous()
    bgc = bgc[:, inds].contiguous()
    target = torch.rand(1, 4096, 3, device='cuda', generator=g)
    bg_color = fi['bg_color'][:, inds].contiguous()
    R = refgold.Reference("train_step", ref_model.available())
    models = (("ours", model),) + ((("ref", ref_model.build(model.state_dict(), hp, torso=False)),) if R.live else ())
    outs, grads = {}, {}
    for name, m in models:
        m.train()
        m.zero_grad(set_to_none=True)
        out = m.render(rays_o, rays_d, fi['cond'], bgc, poses6, index=0, dt_gamma=hp['dt_gamma'], bg_color=bg_color, perturb=False,
                       force_all_rays=True, max_steps=hp['max_steps'])
        loss = ((out['rgb_map'] - target) ** 2).mean() + 1e-3 * out['ambient'].mean() + 1e-3 * out['weights_sum'].mean()
        loss.backward()
        torch.cuda.synchronize()
        outs[name] = {k: out[k].detach().float().cpu().numpy() for k in ('rgb_map', 'weights_sum', 'ambient', 'depth_map')}
        grads[name] = {k: p.grad.detach().float().cpu().numpy().reshape(-1) for k, p in m.named_parameters() if p.grad is not None}
        m.eval()
    if R.live:
        for k, v in outs["ref"].items():
            R.put("out/" + k, _per_ray(v))
        R.put("grad_names", np.array(sorted(grads["ref"])))
        rs = np.random.RandomState(0)
        for k, gr in grads["ref"].items():
            R.put("max/" + k, np.float64(np.abs(gr).max()))
            top = np.argsort(-np.abs(gr), kind="stable")[:128]
            R.put("grad/" + k, gr, rows=np.concatenate([top, rs.choice(gr.size, min(gr.size, 128), replace=False)]))
    for k in ('rgb_map', 'weights_sum', 'ambient', 'depth_map'):
        assert_close(_per_ray(outs["ours"][k])[R.rows("out/" + k)], R["out/" + k], what=f"train-mode {k}")
    assert set(grads["ours"]) == set(R["grad_names"].tolist()), set(grads["ours"]) ^ set(R["grad_names"].tolist())
    worst = {}
    for k in R["grad_names"].tolist():
        scale = float(R["max/" + k])
        ours = grads["ours"][k][R.rows("grad/" + k)]
        if scale == 0:
            assert np.abs(grads["ours"][k]).max() == 0, k
            continue
        worst[k] = float(np.abs(ours - R["grad/" + k]).max() / scale)
        assert worst[k] <= 1e-3, f"grad of {k}: max |diff| / max |ref| = {worst[k]:.2e}"
    print("train-step gradient parity, worst per tensor:", {k: f"{v:.1e}" for k, v in sorted(worst.items(), key=lambda kv: -kv[1])[:6]})
    assert any('embeddings' in k for k in worst)
