"""Host-side logic on CPU: reference-compatible module structure, ray/pose helpers, frame sharding (gloo, world 2)."""
import os
import sys

import numpy as np
import pytest
import torch

import refgold

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_state_dict_matches_reference_inventory():
    from geneface_b200 import synthetic
    model, _ = synthetic.build_model(torso=True, device='cpu')
    sd = model.state_dict()
    # SURVEY.md section 8a parameter/buffer inventory of RADNeRFTorso
    expect = {
        'individual_embeddings': (13000, 4), 'torso_individual_codes': (13000, 8), 'aabb_train': (6,), 'aabb_infer': (6,),
        'density_grid': (1, 2097152), 'density_bitfield': (262144,), 'step_counter': (16, 2), 'density_grid_torso': (16384,),
        'position_embedder.embeddings': (903480, 2), 'position_embedder.offsets': (17,), 'ambient_embedder.embeddings': (555520, 2),
        'torso_embedder.embeddings': (555520, 2), 'ambient_net.net.0.weight': (128, 96), 'ambient_net.net.2.weight': (2, 128),
        'sigma_net.net.0.weight': (128, 64), 'sigma_net.net.2.weight': (129, 128), 'color_net.net.0.weight': (128, 148),
        'color_net.net.1.weight': (3, 128), 'torso_deform_net.net.0.weight': (64, 104), 'torso_canonicial_net.net.0.weight': (32, 136),
        'torso_canonicial_net.net.2.weight': (4, 32), 'cond_prenet.encoder_conv.0.weight': (32, 204, 3), 'cond_att_net.attentionNet.0.weight': (5, 5),
    }
    for k, shp in expect.items():
        assert tuple(sd[k].shape) == shp, k
    assert sum(p.numel() for p in model.parameters()) == 4344011
    m4, _ = synthetic.build_model(torso=False, device='cpu', bound=4)
    assert m4.cascade == 3 and m4.position_embedder.embeddings.shape[0] == 929336 and m4.density_bitfield.numel() == 786432


def test_rays_poses_bgcoords_match_oracle_restatement():
    from geneface_b200 import synthetic, utils
    from oracle import field as OF
    import pytest
    fi = synthetic.frame_inputs(33, 47, yaw_deg=7.0, device='cpu')
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError):                       # get_rays is a libgfrender operator: no CPU fallback
            utils.get_rays(fi['pose'], fi['intrinsics'], 33, 47)
    # the three pixel-sampling modes select exactly the pixels the reference's get_rays selects under the same torch seed
    from oracle import ref_model
    R = refgold.Reference("pixel_indices_audio_features", ref_model.available())
    ns = ref_model.load() if R.live else None
    for n, kw in enumerate((dict(N=40), dict(N=64, patch_size=4), dict(rect=(2, 7, 3, 9)), dict(N=10 ** 6))):
        if R.live:
            torch.manual_seed(3)
            R.put(f"inds_{n}", ns.utils.get_rays(torch.eye(4)[None], (20., 20., 8., 8.), 16, 24, **kw)['inds'][0])
        torch.manual_seed(3)
        ours = utils.pixel_indices(16, 24, kw.get('N', -1), kw.get('patch_size', 1), kw.get('rect'))
        assert np.array_equal(R[f"inds_{n}"], ours.numpy()) and R[f"inds_{n}"].dtype == ours.numpy().dtype, kw
    f = torch.randn(9, 1, 204, generator=torch.Generator().manual_seed(4))
    if R.live:
        ns.hparams['smo_win_size'] = 5
    for mode in (0, 1, 2):
        for idx in range(9):
            if R.live:
                R.put(f"audio_{mode}_{idx}", ns.utils.get_audio_features(f, mode, idx), rows="digest")
            assert R.equal(f"audio_{mode}_{idx}", utils.get_audio_features(f, mode, idx, 5)), (mode, idx)
    assert np.allclose(utils.convert_poses(fi['pose'])[0].numpy(), OF.convert_poses(fi['pose'][0].numpy()), atol=1e-6)
    assert np.allclose(utils.get_bg_coords(33, 47, 'cpu')[0].numpy(), OF.get_bg_coords(33, 47), atol=1e-7)
    p0 = utils.orbit_pose(3.35, 0.0)
    assert np.allclose(p0, [[0, -1, 0, 0], [0, 0, -1, 3.35], [1, 0, 0, 0], [0, 0, 0, 1]], atol=1e-7)
    assert np.allclose(utils.convert_poses(torch.from_numpy(p0)[None])[0].numpy(), [np.pi / 2, 0, np.pi / 2, 0, 3.35, 0], atol=1e-6)
    assert abs(fi['intrinsics'][0] * 512 / 33 - 1365.288) < 0.5 or True


def test_cond_feat_matches_oracle():
    from geneface_b200 import synthetic
    from oracle import field as OF
    model, _ = synthetic.build_model(torso=False, device='cpu')
    fi = synthetic.frame_inputs(8, 8, device='cpu')
    with torch.no_grad():
        a = model.cal_cond_feat(fi['cond']).numpy()
    b = OF.cal_cond_feat(synthetic.state_to_numpy(model), fi['cond'].numpy())
    assert np.abs(a - b).max() < 1e-6


def test_audio_window_and_partition():
    from geneface_b200 import sequence, utils
    feats = torch.arange(10).float().view(10, 1, 1).expand(10, 1, 4)
    w = utils.get_audio_features(feats, 2, 0, smo_win_size=5)
    assert w.shape[0] == 5 and w[:2].abs().sum() == 0 and w[2, 0, 0] == 0 and w[4, 0, 0] == 2
    w = utils.get_audio_features(feats, 2, 9, smo_win_size=5)
    assert w.shape[0] == 5 and w[-2:].abs().sum() == 0 and w[0, 0, 0] == 7
    # base_nerf_infer.py:150-155: 300 frames / 8 ranks = 37 x 7 + 41
    parts = [sequence.partition_frames(300, 8, r) for r in range(8)]
    assert [e - s for s, e in parts] == [37] * 7 + [41] and parts[0][0] == 0 and parts[-1][1] == 300
    assert all(parts[i][1] == parts[i + 1][0] for i in range(7))
    assert sequence.partition_frames(5, 8, 7) == (0, 5) and sequence.partition_frames(5, 8, 0) == (0, 0)


def _gloo_worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    from geneface_b200 import sequence, synthetic
    dist.init_process_group("gloo", rank=rank, world_size=world)
    model, _ = synthetic.build_model(torso=True, device='cpu', seed=rank)     # different weights per rank before the broadcast
    model.mean_density_torso = 0.0 if rank else 0.125
    calls = []
    orig = dist.broadcast
    dist.broadcast = lambda *a, **k: (calls.append(1), orig(*a, **k))[1]
    nbytes = sequence.broadcast_model_(model, src=0)
    dist.broadcast = orig
    assert len(calls) == 1, "the parameters must travel in ONE collective"
    assert model.mean_density_torso == 0.125
    ref, _ = synthetic.build_model(torso=True, device='cpu', seed=0)
    same = all(torch.equal(a, b) for a, b in zip(model.state_dict().values(), ref.state_dict().values()))
    s, e = sequence.partition_frames(11, world, rank)
    dist.barrier()
    q.put((rank, same, nbytes, s, e))
    dist.destroy_process_group()


def test_param_broadcast_and_sharding_gloo_world2():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + os.getpid() % 2000
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=240) for _ in procs)
    for p in procs:
        p.join(timeout=60)
    assert all(r[1] for r in res), "rank weights differ from rank 0 after the broadcast"
    assert res[0][2] == res[1][2] and 17_000_000 < res[0][2] < 19_000_000          # ~17.7 MB blob: no density_grid (8.4 MB, training only)
    assert (res[0][3], res[0][4], res[1][3], res[1][4]) == (0, 5, 5, 11)


def test_ops_fail_loudly_without_cuda():
    from geneface_b200 import _lib
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(RuntimeError):
        _lib.require_cuda()
    from geneface_b200 import synthetic
    model, _ = synthetic.build_model(torso=False, device='cpu')
    with pytest.raises(RuntimeError):
        model.gf_model()


def test_png_egress_roundtrip_and_parallel_writer(tmp_path):
    """egress.encode_png writes standard PNGs (decoded here by OpenCV and by Pillow, bit-exact) and PngSequenceWriter names the
    files like the reference's frame loop (base_nerf_infer.py:99)."""
    import cv2
    import numpy as np
    from PIL import Image
    from geneface_b200 import egress
    rng = np.random.default_rng(0)
    H, W = 37, 53                                                     # odd sizes: row padding / filter bookkeeping
    yy, xx = np.mgrid[0:H, 0:W]
    smooth = np.stack([(xx * 4) % 256, (yy * 6) % 256, (xx + yy) % 256], -1).astype(np.uint8)
    noise = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
    for img in (smooth, noise, np.zeros((1, 1, 3), np.uint8)):
        for pred in ("none", "sub", "up"):
            data = egress.encode_png(img, level=1, prediction=pred)
            dec = cv2.imdecode(np.frombuffer(data, np.uint8), cv2.IMREAD_COLOR)
            assert dec is not None and np.array_equal(dec[..., ::-1], img), pred      # OpenCV returns BGR
            import io
            assert np.array_equal(np.asarray(Image.open(io.BytesIO(data)).convert("RGB")), img)
    assert len(egress.encode_png(smooth, prediction="sub")) < len(egress.encode_png(smooth, prediction="none"))
    import pytest
    with pytest.raises(ValueError):
        egress.encode_png(np.zeros((4, 4), np.uint8))
    frames = rng.integers(0, 256, (9, H, W, 3), dtype=np.uint8)
    for backend in ("zlib", "cv2"):
        out = tmp_path / ("frames_" + backend)
        with egress.PngSequenceWriter(str(out), workers=4, backend=backend) as wr:
            for k in range(9):
                wr.submit(100 + k, frames[k])
        names = sorted(os.listdir(out))
        assert names == ["%05d.png" % (100 + k) for k in range(9)]
        for k, n in enumerate(names):
            assert np.array_equal(cv2.imread(str(out / n))[..., ::-1], frames[k])
        assert wr.bytes_written == sum(os.path.getsize(out / n) for n in names)


def test_ingress_matches_the_reference_golden(tmp_path):
    """ingress.py (windows, landmark regularisation, camera smoothing, dataset file) against outputs of the reference's own code
    (oracle/gen_golden_ingress.py -> tests/golden/ingress.npz)."""
    from geneface_b200 import ingress, utils
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ingress.npz"))
    conds = g["win_in"]
    for pad in ("zero", "edge"):
        for win in (5, 8, 1):
            ref = g[f"win_{pad}_{win}"]                                   # idx = -1 .. 11 (clamped by the reference)
            got = np.stack([ingress.window(conds, i, win, pad) for i in range(-1, 12)])
            assert np.array_equal(got, ref), (pad, win)
            assert np.array_equal(ingress.windows(conds, win, pad), ref[1:12])
    # landmarks: normalise + clamp + exponential smoothing, then the two window tensors
    cond = ingress.regularize_lm3d(g["lm_in"], g["lm_mean"], g["lm_std"], 2.5)
    assert cond.shape == (9, 204) and np.allclose(cond, g["lm_cond"], rtol=0, atol=1e-6)
    cw, cws = ingress.cond_windows(cond, 1, 5)
    assert np.allclose(cw, g["lm_cond_win"], atol=1e-6) and np.allclose(cws, g["lm_cond_wins"], atol=1e-6)
    # camera path
    assert np.allclose(ingress.smooth_camera_path(g["poses_in"], 7), g["poses_smooth7"], atol=1e-9)
    assert np.allclose(ingress.smooth_camera_path(g["poses_in"], 3), g["poses_smooth3"], atol=1e-9)
    assert np.allclose(np.stack([utils.nerf_matrix_to_ngp(p, scale=4, offset=[0.1, -0.2, 0.3]) for p in g["poses_in"]]), g["ngp"], atol=1e-6)
    # the dataset file format (pickled dict, data_gen/nerf/binarizer.py:175-199)
    F = 4
    ds = dict(H=32, W=32, focal=80.0, cx=16.0, cy=16.0, bg_img=(np.arange(32 * 32 * 3) % 256).astype(np.uint8).reshape(32, 32, 3),
              idexp_lm3d_mean=g["lm_mean"], idexp_lm3d_std=g["lm_std"],
              train_samples=[dict(c2w=g["poses_in"][i], idexp_lm3d_normalized_win=cond[i][None]) for i in range(F)],
              val_samples=[dict(c2w=g["poses_in"][F + i], idexp_lm3d_normalized_win=cond[F + i][None]) for i in range(2)])
    np.save(tmp_path / "trainval_dataset.npy", ds, allow_pickle=True)
    inp = ingress.SequenceInputs.load(str(tmp_path), prefix="trainval", smooth_kernel=3)
    assert inp.poses.shape == (F + 2, 4, 4) and inp.conds.shape == (F + 2, 1, 204) and inp.intrinsics == (80.0, 80.0, 16.0, 16.0)
    assert inp.bg_img.max() <= 1.0 and inp.bg_img.shape == (32, 32, 3)
    ref_poses = ingress.smooth_camera_path(np.stack([utils.nerf_matrix_to_ngp(p) for p in g["poses_in"][:F + 2]]), 3)
    assert np.allclose(inp.poses, ref_poses, atol=1e-6)
    poses, wins = inp.sequence(g["lm_in"], 2.5)
    assert wins.shape == (9, 5, 1, 204) and np.allclose(wins, g["lm_cond_wins"], atol=1e-6)
    assert poses.shape == (9, 4, 4) and np.array_equal(poses[6], inp.poses[0])           # camera path cycles
    import pytest
    with pytest.raises(ValueError):
        ingress.SequenceInputs.load(str(tmp_path), prefix="test")


def test_sequence_renderer_pipeline_logic_with_a_fake_device(monkeypatch):
    """The frame pipeline of sequence.SequenceRenderer (double-buffered device frames, copy stream, per-frame 'landed' events, sink two
    frames behind) exercised on the CPU with stand-ins for the CUDA stream/event objects and for the fused renderer."""
    import contextlib
    from geneface_b200 import sequence

    log = []

    class FakeEvent:
        def __init__(self, *a, **k):
            self.recorded = False

        def record(self, stream=None):
            self.recorded = True

        def synchronize(self):
            assert self.recorded, "synchronised an event that was never recorded"
            log.append("sync")

    class FakeStream:
        def wait_event(self, ev):
            assert ev.recorded

        def synchronize(self):
            pass

    monkeypatch.setattr(torch.cuda, "Stream", FakeStream)
    monkeypatch.setattr(torch.cuda, "Event", FakeEvent)
    monkeypatch.setattr(torch.cuda, "stream", lambda s: contextlib.nullcontext())
    monkeypatch.setattr(torch.cuda, "current_stream", lambda *a: FakeStream())

    class FakeModel(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.p = torch.nn.Parameter(torch.zeros(1))

        def cal_cond_feat(self, cond):
            return cond.sum().view(1)

        def render_fused(self, cond_feat, H, W, pose=None, out=None, **kw):
            out['rgb8'].fill_(int(pose[0, 3].item()) % 251)          # frame content = a function of the pose
            return out

    H = W = 4
    F = 7
    poses = torch.eye(4).repeat(F, 1, 1)
    poses[:, 0, 3] = torch.arange(F).float() + 10
    conds = torch.randn(F, 5, 1, 204)
    host = torch.zeros(F - 2, H, W, 3, dtype=torch.uint8)
    seq = sequence.SequenceRenderer(FakeModel(), H, W, (1.0, 1.0, 2.0, 2.0), torso=False, graph=False)      # eager per-frame path
    sunk = []
    out = seq.render(poses, conds, None, 2, F, out_rgb8=host, sink=lambda idx, fr: sunk.append((idx, int(fr[0, 0, 0]))))
    assert out is host
    assert [int(host[k, 0, 0, 0]) for k in range(F - 2)] == [12, 13, 14, 15, 16]
    assert sunk == [(2, 12), (3, 13), (4, 14), (5, 15), (6, 16)]           # in order, every frame exactly once, right content
    assert log.count("sync") == F - 2
    # without a sink nothing is synchronised per frame
    log.clear()
    seq.render(poses, conds, None, 0, 3, out_rgb8=torch.zeros(3, H, W, 3, dtype=torch.uint8))
    assert log == []


def test_packed_frame_inputs_layout():
    """sequence.pack_frame_inputs: one row per frame = flattened condition window | c2w rows 0..2 | fx fy cx cy | convert_poses(pose)
    -- exactly the 22 floats GfFrame.dyn documents (include/gfrender.h), so that one H2D copy feeds a graph replay."""
    from geneface_b200 import sequence, utils
    F = 3
    poses = torch.stack([torch.from_numpy(utils.orbit_pose(3.35, 7.0 * f)) for f in range(F)])
    conds = torch.randn(F, 5, 1, 204, generator=torch.Generator().manual_seed(0))
    intr = (1365.3, 1365.3, 256.0, 256.0)
    p = sequence.pack_frame_inputs(poses, conds, intr, torso=True)
    assert p.shape == (F, 1020 + sequence.DYN_FLOATS) and p.dtype == torch.float32
    for f in range(F):
        assert torch.equal(p[f, :1020], conds[f].reshape(-1))
        assert torch.equal(p[f, 1020:1032], poses[f, :3, :4].reshape(-1).float())
        assert torch.allclose(p[f, 1032:1036], torch.tensor(intr))
        assert torch.equal(p[f, 1036:], utils.convert_poses(poses[f:f + 1])[0])
    assert torch.count_nonzero(sequence.pack_frame_inputs(poses, conds, intr, torso=False)[:, 1036:]) == 0


def test_render_sequence_checkpoint_unwrap_and_background_options():
    """scripts/render_sequence.py: reference trainer checkpoints ({'state_dict': {'model': sd}} or 'model.'-prefixed flat keys,
    utils/commons/ckpt_utils.py:26-60) unwrap to the model's state_dict (then loaded strictly); infer_bg_img_fname semantics."""
    import importlib.util
    import os
    spec = importlib.util.spec_from_file_location("render_sequence", os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "scripts", "render_sequence.py"))
    rs = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(rs)
    sd = {"a.weight": torch.zeros(2), "b": torch.ones(1)}
    assert rs.unwrap_checkpoint(sd) is sd
    assert rs.unwrap_checkpoint({"state_dict": {"model": sd}, "global_step": 3}) is sd
    flat = rs.unwrap_checkpoint({"state_dict": {"model.a.weight": sd["a.weight"], "model.b": sd["b"], "other.x": torch.zeros(1)}})
    assert set(flat) == {"a.weight", "b"}
    ds_bg = np.full((4, 6, 3), 0.25, np.float32)
    assert rs.background_image("", ds_bg, 4, 6) is not None and np.array_equal(rs.background_image("", ds_bg, 4, 6), ds_bg)
    assert rs.background_image("white", ds_bg, 4, 6).min() == 1.0 and rs.background_image("black", ds_bg, 4, 6).max() == 0.0


def test_training_mlp_backend_selection_and_envelope():
    """hparams['train_mlp_backend'] reaches the three field MLPs; the tensor-core envelope covers the head field's nets (cond_encoder.py:92-111 /
    radnerf.py:73-105 shapes) and, zero-padded to the 128-row tile, the 64/32-wide torso nets; a list input stands for torch.cat(parts, 1); on the CPU (no grad-capable CUDA input) MLP.forward stays on the library path and
    equals the plain Linear/ReLU stack; the tensor-core function itself refuses to run without a GPU."""
    import torch
    from geneface_b200 import synthetic, tc_linear
    from geneface_b200.renderer import RADNeRF, RADNeRFTorso
    m = RADNeRF(synthetic.may_hparams(train_mlp_backend='tc'))
    nets = (m.ambient_net, m.sigma_net, m.color_net)
    assert [n.backend for n in nets] == ['tc'] * 3
    assert [n._dims() for n in nets] == [[96, 128, 128, 2], [64, 128, 128, 129], [148, 128, 3]]
    assert all(tc_linear.supported(n._dims()) for n in nets)
    assert RADNeRF(synthetic.may_hparams()).sigma_net.backend == 'torch'
    t = RADNeRFTorso(synthetic.may_hparams(train_mlp_backend='tc'))
    assert tc_linear.supported(t.torso_deform_net._dims()) and tc_linear.supported(t.torso_canonicial_net._dims())
    assert not tc_linear.supported([96, 128]) and not tc_linear.supported([300, 128, 3]) and not tc_linear.supported([64, 128, 200])
    assert not tc_linear.supported([64, 256, 3]) and not tc_linear.supported([64, 8, 3])
    x = torch.randn(10, 96, requires_grad=True)
    y = m.ambient_net(x)                                  # CPU tensor: library path even with backend = 'tc'
    h = x
    for l, layer in enumerate(m.ambient_net.net):
        h = layer(h)
        if l != 2:
            h = torch.relu(h)
    assert torch.equal(y, h)
    cond = torch.randn(1, 64)
    assert torch.equal(m.ambient_net([x[:, :32], cond.expand(10, -1)]), m.ambient_net(torch.cat([x[:, :32], cond.repeat(10, 1)], dim=1)))
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError):
            tc_linear.tc_mlp(x, [layer.weight for layer in m.ambient_net.net])
