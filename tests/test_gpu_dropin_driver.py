"""The UNCHANGED reference driver (`dynaboa_benchmark.py`, compiled by build() into the git-ignored oracle/_ref/ --
oracle/build_ref.py -- or taken from the checkout named by DBOA_REFERENCE_ROOT) executed on the GPU on top of the drop-in module
tree, against the trajectory the reference itself produced on CPU (tests/golden/adapt_c2.npz, recorded by
oracle/make_golden.py from the same file).  This is the north-star claim "dynaboa_benchmark.py drops in unchanged", run
rather than AST-checked (tests/test_dropin_surface.py checks the interface without the reference)."""
import os
import runpy
import sys

import numpy as np
import pytest
import torch

from conftest import rel_err
from oracle import ref_harness

pytestmark = pytest.mark.gpu
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DRIVER = ref_harness.driver('dynaboa_benchmark')
SHADOWED = ('constants', 'config', 'model', 'utils', 'base_adaptor', 'boa_dataset', 'learn2learn')


@pytest.mark.skipif(DRIVER is None, reason='no reference driver: build() makes oracle/_ref/ where a reference checkout is readable')
def test_unchanged_reference_driver_follows_reference_trajectory(asset_dir, tmp_path, golden, monkeypatch):
    import joblib
    from dynaboa_b200 import hmr as hmr_mod
    gd = golden('adapt_c2')
    n_frames = 3
    masks_all = torch.from_numpy(gd['teacher_masks']).float()
    calls = {'i': 0}

    def provider(B, dev):                       # c2: one teacher forward per frame -> call index = frame index
        m = masks_all[min(calls['i'], masks_all.shape[0] - 1), 0]
        calls['i'] += 1
        return m.to(dev)
    monkeypatch.setattr(hmr_mod, 'DEFAULT_MASK_PROVIDER', provider)
    monkeypatch.setenv('DBOA_SYNTHETIC_FRAMES', str(n_frames))
    monkeypatch.chdir(tmp_path)
    dropin = os.path.join(REPO, 'dynaboa_b200', 'dropin')
    saved = {m: sys.modules.pop(m) for m in list(sys.modules) if m.split('.')[0] in SHADOWED}
    monkeypatch.setattr(sys, 'path', [dropin, REPO] + sys.path)
    from dynaboa_b200 import config
    monkeypatch.setattr(sys, 'argv', [DRIVER, '--expdir', str(tmp_path / 'exps'), '--expname', 'c2', '--model_file', config.BASE_MODEL,
                                      '--inner_step', '1', '--retrieval', '0', '--lower_level_mixtrain', '0', '--upper_level_mixtrain', '0',
                                      '--dynamic_boa', '0'])
    try:
        with pytest.warns(UserWarning, match='SYNTHETIC'):
            runpy.run_path(DRIVER, run_name='__main__')
    finally:
        for m in list(sys.modules):
            if m.split('.')[0] in SHADOWED:
                del sys.modules[m]
        sys.modules.update(saved)
    out = tmp_path / 'exps' / 'c2'
    res = joblib.load(out / 'res.pt')
    assert len(res['mpjpe']) == n_frames and calls['i'] == n_frames
    for t in range(n_frames):
        assert abs(np.mean(res['mpjpe'][t]) - gd['metrics'][t][0].mean()) <= 1e-3 * gd['metrics'][t][0].mean(), t
        assert abs(np.mean(res['pampjpe'][t]) - gd['metrics'][t][1].mean()) <= 2e-3 * gd['metrics'][t][1].mean(), t
        assert abs(float(res['pve'][t]) - gd['metrics'][t][2].mean()) <= 1e-3 * gd['metrics'][t][2].mean(), t
        pred = joblib.load(out / 'result' / f'Pred_{t}.pt')
        assert rel_err(pred['rotmat'], gd['rotmat'][t]) < 1e-3 and rel_err(pred['beta'], gd['betas'][t]) < 1e-3, t
        assert rel_err(pred['verts'][:, ::10], gd['verts_sub'][t]) < 1e-3, t
    for name in ('res.txt', 'lower_res.pt', 'steps_statistic_res.pt', 'feat_sims.pt', 'optim_step_record.pt', 'lowerlevel_kp2dloss.pt',
                 'upperlevel_kp2dloss.pt', 'setting.txt'):
        assert (out / name).exists(), name          # the reference's result files
