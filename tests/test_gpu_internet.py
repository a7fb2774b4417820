"""Second client of the hot path (N3): the UNCHANGED reference `dynaboa_internet.py` (compiled by build() into the git-ignored
oracle/_ref/ -- oracle/build_ref.py -- or taken from the checkout named by DBOA_REFERENCE_ROOT) on the drop-in tree, fed by
a small synthetic "Internet video" on disk (PNG frames + the reference's npz annotation layout) whose crops and keypoints go
through the GPU input side (N2), against the CPU oracle run on the oracle-processed frames.  Also the library's own
``InternetAdaptor`` (autograd and fused paths)."""
import os
import runpy
import sys
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from conftest import rel_err
from oracle import ref_harness

pytestmark = pytest.mark.gpu
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DRIVER = ref_harness.driver('dynaboa_internet')
SHADOWED = ('constants', 'config', 'model', 'utils', 'base_adaptor', 'boa_dataset', 'learn2learn')
FLAGS = dict(inner_step=1, retrieval=0, lower_level_mixtrain=0, upper_level_mixtrain=0, dynamic_boa=0)
N = 3


def make_video(root):
    """N frames 240 x 320 (smooth content, moving box), 49 keypoints projected inside the box, reference npz layout."""
    import cv2
    os.makedirs(os.path.join(root, 'images'), exist_ok=True)
    rng = np.random.default_rng(11)
    base = cv2.GaussianBlur(rng.uniform(0, 255, size=(240, 320, 3)).astype(np.float32), (0, 0), 3)
    names, centers, scales, parts, frames = [], [], [], [], []
    for t in range(N):
        frame = np.clip(np.roll(base, 3 * t, axis=1) + rng.normal(0, 2, base.shape), 0, 255).astype(np.uint8)
        name = f'f{t:03d}.png'
        cv2.imwrite(os.path.join(root, 'images', name), frame[:, :, ::-1])
        center, scale = np.array([150.0 + 4 * t, 118.0 + t]), 0.9 + 0.01 * t
        kp = np.concatenate([center + rng.uniform(-70, 70, size=(49, 2)), np.ones((49, 1))], 1)
        names.append(name); centers.append(center); scales.append(scale); parts.append(kp); frames.append(frame)
    np.savez(os.path.join(root, 'video.npz'), imgname=np.array(names), center=np.stack(centers), scale=np.array(scales), part=np.stack(parts))
    return frames, centers, scales, parts


def oracle_trajectory(frames, centers, scales, parts, masks):
    from dynaboa_b200 import constants as C, synthetic
    from oracle import adaptor_ref, dataprocess_ref as R
    opts = adaptor_ref.default_options(**FLAGS)
    ora = adaptor_ref.OracleAdaptor(opts, synthetic.make_basemodel(), {g: synthetic.make_smpl_model(g) for g in ('neutral', 'male', 'female')},
                                    synthetic.make_extra_regressors(), dict(np.load(os.path.join(REPO, 'dynaboa_b200/assets/gmm_08.npz'))),
                                    joint_map=C.JOINT_MAP_49, vertex_ids=C.SMPL_EXTRA_VERTEX_IDS, h36m_to_j14=C.H36M_TO_J14)
    calls = {'i': 0}

    def mask_fn(B):
        m = masks[calls['i']]
        calls['i'] += 1
        return [(m[it, 0], m[it, 1]) for it in range(3)]
    ora.mask_fn = mask_fn
    preds = []
    for t in range(N):
        img = torch.from_numpy(R.rgb_processing(frames[t].astype(np.float32), list(centers[t]), float(scales[t])))[None]
        kp = torch.from_numpy(R.j2d_processing(parts[t].astype(np.float32).astype(np.float64), list(centers[t]), float(scales[t])))[None]
        ora.global_step, ora.fit_losses = t, {}
        ora.adaptation({'image': img, 'smpl_j2d': kp}, with_inference=False)
        preds.append(ora.predict(img))
    return preds


@pytest.mark.skipif(DRIVER is None, reason='no reference driver: build() makes oracle/_ref/ where a reference checkout is readable')
def test_unchanged_internet_driver_on_gpu_input_side(asset_dir, tmp_path, monkeypatch):
    import joblib
    from dynaboa_b200 import config, hmr as hmr_mod
    root = tmp_path / 'video'
    frames, centers, scales, parts = make_video(str(root))
    g = torch.Generator().manual_seed(5)
    masks = [(torch.rand(3, 2, 1, 1024, generator=g) >= 0.5).float() * 2.0 for _ in range(N)]
    calls = {'i': 0}

    def provider(B, dev):
        m = masks[min(calls['i'], N - 1)]
        calls['i'] += 1
        return m.to(dev)
    monkeypatch.setattr(hmr_mod, 'DEFAULT_MASK_PROVIDER', provider)
    monkeypatch.setenv('DYNABOA_INTERNET_ROOT', str(root))
    monkeypatch.chdir(tmp_path)
    dropin = os.path.join(REPO, 'dynaboa_b200', 'dropin')
    saved = {m: sys.modules.pop(m) for m in list(sys.modules) if m.split('.')[0] in SHADOWED}
    monkeypatch.setattr(sys, 'path', [dropin, REPO] + sys.path)
    argv = [DRIVER, '--expdir', str(tmp_path / 'exps'), '--expname', 'net', '--dataset', 'internet', '--model_file', config.BASE_MODEL]
    for k, v in FLAGS.items():
        argv += [f'--{k}', str(v)]
    monkeypatch.setattr(sys, 'argv', argv)
    try:
        runpy.run_path(DRIVER, run_name='__main__')
    finally:
        for m in list(sys.modules):
            if m.split('.')[0] in SHADOWED:
                del sys.modules[m]
        sys.modules.update(saved)
    ref = oracle_trajectory(frames, centers, scales, parts, masks)
    for t in range(N):
        pred = joblib.load(tmp_path / 'exps' / 'net' / 'result' / f'Pred_{t}.pt')
        assert rel_err(pred['rotmat'], ref[t]['rotmat']) < 1e-3 and rel_err(pred['beta'], ref[t]['betas']) < 1e-3, t
        assert rel_err(pred['verts'], ref[t]['vertices']) < 1e-3, t


@pytest.mark.parametrize('fused', [False, True])
def test_internet_adaptor_paths(asset_dir, tmp_path, monkeypatch, fused):
    from dynaboa_b200 import config
    from dynaboa_b200.adaptor import InternetAdaptor
    root = tmp_path / 'video'
    frames, centers, scales, parts = make_video(str(root))
    monkeypatch.setenv('DYNABOA_INTERNET_ROOT', str(root))
    from oracle import adaptor_ref
    o = vars(adaptor_ref.default_options(**FLAGS))
    o.update(expdir=str(tmp_path), expname='net', tensorboard=0, cache_results=0, model_file=config.BASE_MODEL, dataset='internet',
             save_res=0, seq_seed=22, teacher_dropout=0)
    ad = InternetAdaptor(SimpleNamespace(**o))
    ad.excute(fused=fused)
    masks = [torch.ones(3, 2, 1, 1024) for _ in range(N)]           # deterministic teacher (eval mode = identity masks)
    ref = oracle_trajectory(frames, centers, scales, parts, masks)
    batch = ad.dataloader.dataset[N - 1]
    pred = ad.predict(batch['image'][None])
    assert rel_err(pred['rotmat'], ref[-1]['rotmat']) < 1e-3 and rel_err(pred['vertices'], ref[-1]['vertices']) < 1e-3
