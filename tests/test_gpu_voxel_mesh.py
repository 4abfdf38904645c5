"""Marching-cubes meshes on the GPU (s3d_voxel_mesh): bit-exact against the reference statement (tests/mesh_oracle.py), on
random, binary, non-finite, empty and full grids and on the very voxels the forward returns; every other output of the
forward is unchanged, and runner.py --test --save-meshes writes the same meshes as OBJ files."""
import ctypes
import json
import os
import sys

import numpy as np
import pytest
import torch

from stereo_3d_reconstruction_b200 import lib, models as M, ops
from stereo_3d_reconstruction_b200.utils import synthetic
from tests import mesh_oracle as O
from tests.common import small_cfg

pytestmark = pytest.mark.gpu


def _random(B, n, seed, special=True):
    rng = np.random.default_rng(seed)
    vol = rng.random((B, n, n, n)).astype(np.float32)
    if special:
        sel = rng.random((B, n, n, n))
        vol[sel < 0.03] = np.nan
        vol[(sel >= 0.03) & (sel < 0.05)] = np.inf
        vol[(sel >= 0.05) & (sel < 0.07)] = -np.inf
        vol[(sel >= 0.07) & (sel < 0.1)] = -0.5
        vol[(sel >= 0.1) & (sel < 0.13)] = 2.5
    return vol


def _binary(B, n, t, seed, p=0.3):
    rng = np.random.default_rng(seed)
    return np.where(rng.random((B, n, n, n)) < p, np.float32(t), np.float32(0)).astype(np.float32)


def _check_mesh(verts, faces, counts, want):
    """GPU outputs (CPU copies) of a batch against the oracle's per-sample meshes."""
    for b, (v, f) in enumerate(want):
        assert counts[b].tolist() == [len(v), len(f)], b
        assert np.array_equal(faces[b, :len(f)], f), b
        assert np.array_equal(verts[b, :len(v)].view(np.uint32), v.view(np.uint32)), b


def _run(vol, t, flat=False):
    B, n = vol.shape[0], vol.shape[1]
    x = torch.from_numpy(np.ascontiguousarray(vol)).cuda()
    if flat:
        x = x.reshape(B, -1)
    mv, mf = ops.voxel_mesh_bounds(n)
    out = (torch.full((B, mv, 3), -7.0, device='cuda'), torch.full((B, mf, 3), -7, dtype=torch.int32, device='cuda'),
           torch.full((B, 2), -7, dtype=torch.int32, device='cuda'))
    n0 = lib.launches()
    got = ops.voxel_mesh(x, t, out=out)
    assert lib.launches() - n0 == (1 if B else 0)
    assert all(a is b for a, b in zip(got, out))
    v, f, c = (o.cpu().numpy() for o in out)
    want = O.mesh(vol, t)
    _check_mesh(v, f, c, want)
    for b, (wv, wf) in enumerate(want):                             # rows past the counts are not written
        assert (v[b, len(wv):] == -7.0).all() and (f[b, len(wf):] == -7).all()
    return want


def test_bounds():
    assert ops.voxel_mesh_bounds(32) == (114444, 179685)
    for n in (1, 2, 5, 64):
        assert ops.voxel_mesh_bounds(n) == O.bounds(n)


@pytest.mark.parametrize('n,B', [(1, 3), (2, 8), (5, 64), (32, 4), (64, 2)])
@pytest.mark.parametrize('t', [0.2, 0.5, 1.0])
def test_random_fields_match_oracle(n, B, t):
    want = _run(_random(B, n, seed=n * 100 + B + int(t * 10)), t, flat=n == 5)
    if n >= 5:
        assert all(len(f) > 0 for _, f in want)


@pytest.mark.parametrize('n,B', [(2, 16), (5, 64), (32, 64), (64, 1)])
@pytest.mark.parametrize('t', [0.2, 0.5, 1.0])
def test_binary_fields_match_oracle(n, B, t):
    _run(_binary(B, n, t, seed=n + B), t)


def test_single_cell_configurations():
    vol = np.zeros((256, 2, 2, 2), np.float32)
    for case in range(256):
        for c in range(8):
            if (case >> c) & 1:
                vol[case, (c >> 2) & 1, (c >> 1) & 1, c & 1] = 0.9
    for t in (0.3, 0.9):
        want = _run(vol, t)
        for v, f in want[1:]:
            assert O.closed_manifold(v, f)


def test_empty_and_full():
    n = 8
    vol = np.stack([np.zeros((n,) * 3), np.ones((n,) * 3), np.full((n,) * 3, np.nan), np.full((n,) * 3, np.inf),
                    np.full((n,) * 3, 0.49)]).astype(np.float32)
    want = _run(vol, 0.5)
    assert [len(f) for _, f in want] == [0, 12 * n * n - 4, 0, 12 * n * n - 4, 0]       # a cube with its 8 corners cut
    assert all(O.closed_manifold(v, f) and O.signed_volume(v, f) > 0 for v, f in (want[1], want[3]))


def test_smooth_shapes():
    n = 32
    g = (np.arange(n) + 0.5) / n - 0.5
    z, y, x = np.meshgrid(g, g, g, indexing='ij')
    d = np.sqrt(x * x + y * y + z * z)
    torus = 0.12 - np.sqrt((np.sqrt(x * x + y * y) - 0.28) ** 2 + z * z)
    vol = np.clip(0.5 + np.stack([0.35 - d, torus, np.minimum(0.4 - d, d - 0.2)]) * n, 0, 1).astype(np.float32)
    want = _run(vol, 0.5)
    assert [O.euler(v, f) for v, f in want] == [2, 0, 4]


def test_bad_arguments_rejected_before_any_launch():
    L = lib.load()
    B, n = 2, 8
    mv, mf = ops.voxel_mesh_bounds(n)
    vol = torch.rand(B, n, n, n, device='cuda')
    v = torch.empty(B, mv, 3, device='cuda')
    f = torch.empty(B, mf, 3, dtype=torch.int32, device='cuda')
    c = torch.full((B, 2), -5, dtype=torch.int32, device='cuda')
    s = torch.cuda.current_stream().cuda_stream

    def call(vol_=vol.data_ptr(), B_=B, n_=n, t_=0.5, v_=v.data_ptr(), mv_=mv, f_=f.data_ptr(), mf_=mf, c_=c.data_ptr()):
        return L.s3d_voxel_mesh(vol_, B_, n_, t_, v_, mv_, f_, mf_, c_, s)
    assert call(B_=0) == 0 and call(t_=1.0) == 0
    torch.cuda.synchronize()
    c.fill_(-5)
    for bad in (dict(vol_=None), dict(v_=None), dict(f_=None), dict(c_=None), dict(n_=0), dict(n_=65), dict(B_=-1),
                dict(t_=0.0), dict(t_=-0.5), dict(t_=1.5), dict(t_=float('nan')), dict(t_=float('inf')),
                dict(mv_=mv - 1), dict(mf_=mf - 1)):
        rc = call(**bad)
        assert rc == -1, bad
        with pytest.raises(lib.S3dError):
            lib.check(rc, 's3d_voxel_mesh')
    torch.cuda.synchronize()
    assert (c == -5).all()                                           # nothing ran
    a, b = ctypes.c_int(), ctypes.c_int()
    assert L.s3d_voxel_mesh_bounds(0, ctypes.byref(a), ctypes.byref(b)) == -1
    assert L.s3d_voxel_mesh_bounds(65, ctypes.byref(a), ctypes.byref(b)) == -1
    assert L.s3d_voxel_mesh_bounds(4, None, ctypes.byref(b)) == -1
    n0 = lib.launches()
    for bad_vol, t in ((vol.double(), 0.5), (vol.half(), 0.5), (vol[:, :, :, :7].contiguous(), 0.5),
                       (vol.reshape(B, -1)[:, 1:].contiguous(), 0.5), (vol[0], 0.5), (torch.rand(1, 65, 65, 65, device='cuda'), 0.5),
                       (vol, 0.0), (vol, 1.5), (vol, float('nan')), (vol, float('-inf')), (vol, 'x'), (vol, 1e-46)):
        with pytest.raises(ValueError):
            ops.voxel_mesh(bad_vol, t)
    for bad_out in ((v, f), (v[:, :-1].contiguous(), f, c), (v, f.float(), c), (v, f, c[:1].contiguous()),
                    (v.cpu(), f, c)):
        with pytest.raises((ValueError, lib.S3dError)):
            ops.voxel_mesh(vol, 0.5, out=bad_out)
    with pytest.raises(lib.S3dError):
        ops.voxel_mesh(vol.cpu(), 0.5)
    assert lib.launches() == n0


# ---- the model ------------------------------------------------------------------------------------------------------------
def _model(prec='bf16', default=False, **kw):
    if default:
        from config import cfg as dcfg
        cfg = dcfg.clone()
        cfg.NETWORK.PRECISION = prec
        for k, v in kw.items():
            sec, key = k.split('__')
            cfg[sec][key] = v
    else:
        cfg = small_cfg(NETWORK__PRECISION=prec, **kw)
    return cfg, M.build_model('Stereo2Voxel', cfg, seed=3).cuda().pack()


def _inputs(cfg, B, seed):
    H, W = cfg.CONST.IMG_H, cfg.CONST.IMG_W
    left, right, d = synthetic.stereo_pair(B, H, W, 2 * cfg.NETWORK.MAX_DISP, seed=seed)
    gt = synthetic.gt_volume(B, cfg.CONST.N_VOX, seed=seed + 50)
    return (left.cuda(), right.cuda()), gt.cuda(), synthetic.disparity_gt(d, H, W).cuda()


def _check_model_mesh(cfg, vox, mesh):
    v, f, c = (t.cpu().numpy() for t in mesh)
    want = O.mesh(vox.cpu().numpy(), float(cfg.TEST.MESH_THRESH))
    _check_mesh(v, f, c, want)
    ref = ops.voxel_mesh(vox.contiguous(), cfg.TEST.MESH_THRESH)
    for b in range(vox.shape[0]):
        nv, nf = int(c[b, 0]), int(c[b, 1])
        assert torch.equal(ref[2][b].cpu(), mesh[2][b].cpu())
        assert torch.equal(ref[0][b, :nv], mesh[0][b, :nv]) and torch.equal(ref[1][b, :nf], mesh[1][b, :nf])
    return want


@pytest.mark.parametrize('default', [False, True])
def test_model_mesh_exact_and_outputs_unchanged(default):
    cfg, model = _model('bf16', default)
    args, gt, _ = _inputs(cfg, 2, seed=1)
    with torch.no_grad():
        for g in (None, gt):
            ga = () if g is None else (g,)
            n0 = lib.launches()
            plain = [t.clone() for t in model(*args, *ga)]
            n1 = lib.launches()
            full = [t.clone() for t in model(*args, *ga, mesh=True)]
            n2 = lib.launches()
            assert (n2 - n1) - (n1 - n0) == 1                       # voxel_mesh_kernel
            assert len(full) == len(plain) + 3
            for a, b in zip(plain, full):
                assert torch.equal(a, b)
            want = _check_model_mesh(cfg, full[2], full[-3:])
            assert all(len(f) > 0 for _, f in want)


def test_model_launches_unchanged_without_flag():
    cfg, model = _model()
    args, gt, dgt = _inputs(cfg, 2, seed=0)
    with torch.no_grad():
        counts = []
        for kw in (dict(), dict(mesh=False), dict(mesh=True)):
            n0 = lib.launches()
            model(*args, gt, disp_gt=dgt, **kw)
            counts.append(lib.launches() - n0)
    assert counts[0] == counts[1] and counts[2] == counts[0] + 1


def test_model_tuple_positions_with_every_option():
    cfg, model = _model()
    args, gt, dgt = _inputs(cfg, 2, seed=4)
    kw = dict(disp_gt=dgt, lr_check=True, uncertainty=True, surface=True)
    with torch.no_grad():
        base = [t.clone() for t in model(*args, gt, **kw)]
        full = [t.clone() for t in model(*args, gt, mesh=True, **kw)]
        part = [t.clone() for t in model(*args, gt, disp_gt=dgt, uncertainty=True, mesh=True)]
    assert len(base) == 10 and len(full) == 13 and len(part) == 10
    for a, b in zip(base, full):
        assert torch.equal(a, b)
    for a, b in zip(full[-3:], part[-3:]):
        assert torch.equal(a, b)
    _check_model_mesh(cfg, full[2], full[-3:])


def test_graphed_matches_eager():
    cfg, model = _model()
    seen = []
    for seed in (0, 1):
        args, gt, dgt = _inputs(cfg, 2, seed=seed)
        with torch.no_grad():
            for ga, kw in (((gt,), dict(disp_gt=dgt, surface=True)), ((), {})):
                eager = [t.clone() for t in model(*args, *ga, mesh=True, **kw)]
                graphed = [t.clone() for t in model.graphed(*args, *ga, mesh=True, **kw)]
                assert len(graphed) == len(eager)
                for a, b in zip(eager, graphed):
                    assert torch.equal(a, b)
        seen.append(eager[-3])
    assert not torch.equal(seen[0], seen[1])
    with torch.no_grad():
        assert len(model.graphed(*args)) == 3
    assert len(model._graphs) == 3                                  # mesh is part of the graph key


def test_micro_batch_concatenates_chunks():
    cfg, model = _model(CONST__MICRO_BATCH=2)
    args, gt, dgt = _inputs(cfg, 5, seed=6)
    with torch.no_grad():
        full = [t.clone() for t in model(*args, gt, disp_gt=dgt, mesh=True)]
        parts = [[t.clone() for t in model(args[0][s:s + 2], args[1][s:s + 2], gt[s:s + 2], disp_gt=dgt[s:s + 2], mesh=True)]
                 for s in range(0, 5, 2)]
    for i, t in enumerate(full[:-3]):
        assert torch.equal(t, torch.cat([p[i] for p in parts]))
    c = torch.cat([p[-1] for p in parts])                           # rows past the counts are not written: compare up to them
    assert torch.equal(full[-1], c)
    for b, (nv, nf) in enumerate(c.tolist()):
        p = parts[b // 2]
        assert torch.equal(full[-3][b, :nv], p[-3][b % 2, :nv]) and torch.equal(full[-2][b, :nf], p[-2][b % 2, :nf])
    _check_model_mesh(cfg, full[2], full[-3:])


def test_value_errors_before_any_launch():
    cfg, model = _model()
    args, gt, _ = _inputs(cfg, 2, seed=0)
    model(*args)                                                    # packed, workspace built
    n0 = lib.launches()
    for bad in (0.0, -0.5, 1.5, float('nan'), float('inf'), None, 'x'):
        cfg.TEST.MESH_THRESH = bad
        with pytest.raises(ValueError):
            model(*args, gt, mesh=True)
        with pytest.raises(ValueError):
            model.graphed(*args, mesh=True)
    assert lib.launches() == n0
    pcfg = small_cfg(NETWORK__PRECISION='bf16')
    pm = M.build_model('Stereo2Point', pcfg, seed=0).cuda().pack()
    with pytest.raises(ValueError):
        pm(*args, mesh=True)
    with pytest.raises(ValueError):
        pm.graphed(*args, mesh=True)
    assert lib.launches() == n0


def test_runner_save_meshes(monkeypatch, capsys, tmp_path):
    import runner
    from config import cfg as dcfg
    from stereo_3d_reconstruction_b200.core import test as T
    n, bs = 3, 2
    out_dir = str(tmp_path / 'meshes')
    monkeypatch.setattr(sys, 'argv', ['runner.py', '--test', '--batch-size', str(bs), '--n-samples', str(n),
                                      '--save-meshes', out_dir])
    runner.main()
    res = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    assert sorted(os.listdir(out_dir)) == sorted(['%06d.obj' % i for i in range(n)] + ['%06d_gt.obj' % i for i in range(n)])
    cfg = dcfg.clone()
    model = M.build_model('Stereo2Voxel', cfg, seed=cfg.CONST.SEED).cuda().pack()
    old = T.test_voxel(cfg, model, n, bs, eval_disp=True).cpu()
    nh = 2 * len(cfg.TEST.VOXEL_THRESH) + 1
    assert res['iou'] == json.loads(json.dumps(T.iou_summary(old[:nh], cfg.TEST.VOXEL_THRESH)))['iou']
    H, W, nv = cfg.CONST.IMG_H, cfg.CONST.IMG_W, cfg.CONST.N_VOX
    for s in range(0, n, bs):
        ids = list(range(s, min(s + bs, n)))
        pairs = [synthetic.stereo_pair(1, H, W, 2 * cfg.NETWORK.MAX_DISP, seed=i) for i in ids]
        gt = torch.cat([synthetic.gt_volume(1, nv, seed=100000 + i) for i in ids])
        with torch.no_grad():
            out = model(torch.cat([p[0] for p in pairs]).cuda(), torch.cat([p[1] for p in pairs]).cuda(), mesh=True)
        v, f, c = (t.cpu().numpy() for t in out[-3:])
        gwant = O.mesh((gt != 0).float().numpy(), 0.5)
        for b, i in enumerate(ids):
            rv, rf = O.read_obj(os.path.join(out_dir, '%06d.obj' % i))
            assert c[b].tolist() == [len(rv), len(rf)]
            assert np.array_equal(rv.view(np.uint32), v[b, :len(rv)].view(np.uint32)) and np.array_equal(rf, f[b, :len(rf)])
            gv, gf = O.read_obj(os.path.join(out_dir, '%06d_gt.obj' % i))
            assert np.array_equal(gv.view(np.uint32), gwant[b][0].view(np.uint32)) and np.array_equal(gf, gwant[b][1])
    monkeypatch.setattr(sys, 'argv', ['runner.py', '--test', '--model', 'Stereo2Point', '--save-meshes', out_dir])
    with pytest.raises(SystemExit) as e:
        runner.main()
    assert 'Stereo2Voxel only' in str(e.value)
