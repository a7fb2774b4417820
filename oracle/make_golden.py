"""Golden-vector generator (run where a checkout of the reference is at hand).

    DBOA_REFERENCE_ROOT=/path/to/DynaBOA python -m oracle.make_golden [name ...]      # writes tests/golden/*.npz

What it does (test infrastructure only; nothing here ships or runs on the GPU box):

1. imports the reference's own modules that are importable offline -- model/hmr.py,
   utils/geometry.py, utils/smplify/prior.py, utils/pose_utils.py -- runs them on seeded
   inputs, asserts the restatements in ``oracle/`` reproduce them, and stores the reference
   outputs as fixtures;
2. executes the reference's own ``base_adaptor.BaseAdaptor`` methods and
   ``dynaboa_benchmark.Adaptor.adaptation`` / ``inference`` UNMODIFIED on CPU -- the two missing
   third-party packages (smplx, learn2learn) and the viz-only imports are replaced by the
   restatements/stubs below, ``__init__``'s file loading is replaced by the synthetic assets --
   asserts ``oracle/adaptor_ref.py`` reproduces the trajectory, and stores it as fixtures;
3. records which names the reference driver ``dynaboa_benchmark.py`` takes from ``self`` and which modules it imports
   (``driver_surface.npz``), the interface the drop-in tree has to provide.

The reference is read from DBOA_REFERENCE_ROOT at run time and never copied.
"""
import importlib
import importlib.util
import os
import random
import shutil
import sys
import tempfile
import types

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get('DBOA_REFERENCE_ROOT')
OUT = os.path.join(REPO, 'tests', 'golden')
sys.path.insert(0, REPO)

from dynaboa_b200 import constants as C, synthetic  # noqa: E402
from oracle import adaptor_ref, eval_ref, geometry_ref, hmr_ref, l2l_ref, prior_ref, smplx_ref  # noqa: E402


def _load_by_path(name, path):
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _same(a, b, what, tol=0.0):
    a, b = torch.as_tensor(a), torch.as_tensor(b)
    err = (a.double() - b.double()).abs().max().item() if a.numel() else 0.0
    scale = max(b.double().abs().max().item(), 1e-30) if b.numel() else 1.0
    assert err <= tol * scale, f'{what}: restatement differs from reference, err={err:.3e} (scale {scale:.3e})'
    return err


# ---------------------------------------------------------------------------------------
# part 1: leaf modules
# ---------------------------------------------------------------------------------------
def golden_geometry():
    sys.path.insert(0, REF)
    ref = importlib.import_module('utils.geometry')
    g = torch.Generator().manual_seed(22)
    out = {}
    x6 = torch.randn(64, 6, generator=g)
    x6[0] = torch.tensor([1., 0, 0, 1, 0, 0])
    out['rot6d_in'], out['rot6d_out'] = x6, ref.rot6d_to_rotmat(x6)
    _same(geometry_ref.rot6d_to_rotmat(x6), out['rot6d_out'], 'rot6d')
    aa = torch.randn(96, 3, generator=g) * torch.tensor([0.05, 0.5, 1.5, 3.0]).repeat_interleave(24).unsqueeze(1)
    aa[0] = 0.0
    out['rodrigues_in'], out['rodrigues_out'] = aa, ref.batch_rodrigues(aa)
    _same(geometry_ref.batch_rodrigues(aa), out['rodrigues_out'], 'batch_rodrigues')
    # rotation matrices covering all four quaternion branches (large angles flip the masks)
    big = torch.randn(160, 3, generator=g)
    big = big / big.norm(dim=1, keepdim=True) * torch.linspace(0.01, 3.13, 160).unsqueeze(1)
    R = ref.batch_rodrigues(big)
    out['r2aa_in'], out['r2aa_out'] = R, ref.rotation_matrix_to_angle_axis(R.clone())
    _same(geometry_ref.rotation_matrix_to_angle_axis(R), out['r2aa_out'], 'rotmat->aa')
    # gradient of sum(w * aa) wrt R through the reference
    w = torch.randn(160, 3, generator=g)
    Rg = R.clone().requires_grad_(True)
    (ref.rotation_matrix_to_angle_axis(Rg) * w).sum().backward()
    Rg2 = R.clone().requires_grad_(True)
    (geometry_ref.rotation_matrix_to_angle_axis(Rg2) * w).sum().backward()
    _same(Rg2.grad, Rg.grad, 'rotmat->aa grad', tol=1e-6)
    out['r2aa_w'], out['r2aa_grad'] = w, Rg.grad
    pts = torch.randn(4, 49, 3, generator=g) * 0.4
    cam = torch.tensor([[0.9, 0.01, -0.02], [1.1, 0.1, 0.05], [0.7, -0.08, 0.0], [0.95, 0.0, 0.0]])
    t = torch.stack([cam[:, 1], cam[:, 2], 2 * C.FOCAL_LENGTH / (C.IMG_RES * cam[:, 0] + 1e-9)], -1)
    ref_p = ref.perspective_projection(pts, torch.eye(3).unsqueeze(0).expand(4, -1, -1), t, C.FOCAL_LENGTH,
                                       torch.zeros(4, 2))
    _same(geometry_ref.weak_perspective_project(cam, pts)[0], ref_p, 'projection')
    out['proj_pts'], out['proj_cam'], out['proj_out'] = pts, cam, ref_p / (C.IMG_RES / 2.0)
    np.savez_compressed(os.path.join(OUT, 'geometry.npz'), **{k: v.detach().numpy() for k, v in out.items()})
    print('geometry ok')


def golden_prior(workdir):
    ref = _load_by_path('ref_prior', os.path.join(REF, 'utils/smplify/prior.py'))
    prior = ref.MaxMixturePrior(prior_folder=os.path.join(workdir, 'data/spin_data'), num_gaussians=8,
                                dtype=torch.float32)
    gmm = dict(np.load(os.path.join(REPO, 'dynaboa_b200/assets/gmm_08.npz')))
    consts = prior_ref.gmm_constants(gmm)
    _same(consts['precisions'], prior.precisions, 'gmm precisions')
    _same(consts['nll_weights'], prior.nll_weights, 'gmm nll_weights')
    g = torch.Generator().manual_seed(23)
    pose = torch.randn(32, 69, generator=g) * 0.3
    pose[:8] = prior.means + 0.05 * torch.randn(8, 69, generator=g)
    p1 = pose.clone().requires_grad_(True)
    ref_out = prior(p1, None)
    ref_out.sum().backward()
    p2 = pose.clone().requires_grad_(True)
    mine = prior_ref.merged_nll(p2, consts)
    mine.sum().backward()
    _same(mine, ref_out, 'merged nll')
    _same(p2.grad, p1.grad, 'merged nll grad', tol=1e-6)
    np.savez_compressed(os.path.join(OUT, 'prior.npz'), pose=pose.numpy(), nll=ref_out.detach().numpy(),
                        grad=p1.grad.numpy(), neg_log_w=(-torch.log(prior.nll_weights)).numpy())
    print('prior ok')


def _feature_digest(feats):
    """Small per-feature digest: (sum, abs-sum, first 32 values in NCHW flatten order)."""
    dig = np.zeros((len(feats), 2), np.float64)
    head = np.zeros((len(feats), 32), np.float32)
    for i, f in enumerate(feats):
        f = f.detach().double()
        dig[i] = [f.sum().item(), f.abs().sum().item()]
        head[i] = f.flatten()[:32].float().numpy()
    return dig, head


def golden_hmr(workdir):
    sys.path.insert(0, REF)
    ref = _load_by_path('ref_hmr', os.path.join(REF, 'model/hmr.py'))
    model = ref.hmr(os.path.join(workdir, 'data/smpl_mean_params.npz'))
    ck = synthetic.make_basemodel()
    sd = hmr_ref.strip_prefix(ck['model'])
    model.load_state_dict(sd, strict=True)
    model.eval()
    g = torch.Generator().manual_seed(24)
    x = torch.randn(2, 3, 224, 224, generator=g)
    with torch.no_grad():
        rot, shape, cam, feats = model(x, need_feature=True)
        mine = hmr_ref.forward(x, sd, need_feature=True)
    _same(mine[0], rot, 'hmr rotmat')
    _same(mine[1], shape, 'hmr shape')
    _same(mine[2], cam, 'hmr cam')
    for i, (a, b) in enumerate(zip(mine[3], feats)):
        _same(a, b, f'hmr feature {i}')
    dig, head = _feature_digest(feats)
    # gradient digest: d(sum of outputs weighted) / d params through the reference
    xg = x[:1]
    w_r, w_s, w_c = torch.randn(1, 24, 3, 3, generator=g), torch.randn(1, 10, generator=g), torch.randn(1, 3, generator=g)
    model.zero_grad()
    r, s, c = model(xg)
    ((r * w_r).sum() + (s * w_s).sum() + (c * w_c).sum()).backward()
    names = ['conv1.weight', 'bn1.weight', 'layer1.0.conv2.weight', 'layer2.0.downsample.0.weight',
             'layer3.5.bn3.bias', 'layer4.2.conv3.weight', 'fc1.weight', 'fc2.bias', 'decpose.weight', 'deccam.bias']
    pg = dict(model.named_parameters())
    p2 = {k: v.clone().requires_grad_(True) for k, v in sd.items() if k not in ('init_pose', 'init_shape', 'init_cam')}
    full = dict(p2); full.update({k: sd[k] for k in ('init_pose', 'init_shape', 'init_cam')})
    r2, s2, c2 = hmr_ref.forward(xg, full)
    ((r2 * w_r).sum() + (s2 * w_s).sum() + (c2 * w_c).sum()).backward()
    grads = {}
    for n in names:
        _same(p2[n].grad, pg[n].grad, f'hmr grad {n}', tol=1e-6)
        gflat = pg[n].grad.flatten()
        grads['grad_' + n] = np.concatenate([[gflat.double().norm().item()], gflat[:64].double().numpy()])
    np.savez_compressed(os.path.join(OUT, 'hmr_forward.npz'), seed_x=24, rotmat=rot.numpy(), shape=shape.numpy(),
                        cam=cam.numpy(), feat_digest=dig, feat_head=head,
                        **{f'feat{i}': feats[i].numpy() for i in range(5, 15)},
                        w_r=w_r.numpy(), w_s=w_s.numpy(), w_c=w_c.numpy(), **grads)
    print('hmr ok')


def golden_smpl():
    """smplx restatement outputs (PARITY UNPINNED upstream; pins the oracle against drift and
    gives the CUDA tests a committed fixture) + analytic checks."""
    body = synthetic.make_smpl_model('neutral')
    ex = synthetic.make_extra_regressors()
    m = {k: (torch.as_tensor(v, dtype=torch.long) if k == 'parents' else torch.as_tensor(v)) for k, v in body.items()
         if k != 'faces'}
    g = torch.Generator().manual_seed(25)
    betas = torch.randn(3, 10, generator=g)
    aa = torch.randn(3, 72, generator=g) * 0.3
    R = geometry_ref.batch_rodrigues(aa.view(-1, 3)).view(3, 24, 3, 3)
    jm, vid = torch.tensor(C.JOINT_MAP_49), torch.tensor(C.SMPL_EXTRA_VERTEX_IDS)
    Jx = torch.as_tensor(ex['J_regressor_extra'])
    out = smplx_ref.smpl_forward(m, Jx, jm, vid, betas, R[:, 1:], R[:, :1], pose2rot=False)
    out_aa = smplx_ref.smpl_forward(m, Jx, jm, vid, betas, aa[:, 3:], aa[:, :3], pose2rot=True)
    # rest pose: vertices = template + shape blend
    eye = torch.eye(3).expand(3, 24, 3, 3)
    rest = smplx_ref.smpl_forward(m, Jx, jm, vid, betas, eye[:, 1:], eye[:, :1], pose2rot=False)
    v_shaped = m['v_template'] + torch.einsum('bl,mkl->bmk', betas, m['shapedirs'])
    _same(rest.vertices, v_shaped, 'rest pose', tol=1e-5)
    # global rotation only: vertices rotate rigidly about the root joint
    Rg = eye.clone(); Rg[:, 0] = R[:, 0]
    rot = smplx_ref.smpl_forward(m, Jx, jm, vid, betas, Rg[:, 1:], Rg[:, :1], pose2rot=False)
    J0 = torch.einsum('bik,ji->bjk', v_shaped, m['J_regressor'])[:, :1]
    _same(rot.vertices, torch.einsum('bij,bvj->bvi', R[:, 0], v_shaped - J0) + J0, 'rigid root rotation', tol=1e-5)
    np.savez_compressed(os.path.join(OUT, 'smpl.npz'), betas=betas.numpy(), aa=aa.numpy(), rotmat=R.numpy(),
                        vertices=out.vertices.numpy(), joints=out.joints.numpy(),
                        vertices_aa=out_aa.vertices.numpy(), joints_aa=out_aa.joints.numpy())
    print('smpl ok')


# ---------------------------------------------------------------------------------------
# part 2: the reference's own adaptor code on CPU
# ---------------------------------------------------------------------------------------
from .ref_harness import _StubSMPLX, _FakeH36M, install_stubs as _install_stubs, make_reference_adaptor as _make_reference_adaptor  # noqa: E402,F401
from .ref_harness import ref_options as _ref_options  # noqa: E402


SAMPLE_PER_TENSOR = 16


def sample_indices(name, numel):
    """Deterministic sample positions used by golden files and by the GPU parity tests."""
    import zlib
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    return rng.integers(0, numel, size=SAMPLE_PER_TENSOR)


def _theta_samples(named):
    return np.stack([v.detach().flatten()[sample_indices(k, v.numel())].double().numpy() for k, v in named])


def _seeded_masks(B):
    """Same draws nn.Dropout makes inside the reference teacher (global CPU generator)."""
    out = []
    for _ in range(3):
        m1 = torch.nn.functional.dropout(torch.ones(B, 1024), 0.5, True)
        m2 = torch.nn.functional.dropout(torch.ones(B, 1024), 0.5, True)
        out.append((m1, m2))
    return out


def golden_adapt(workdir, tag, n_frames, **over):
    opts = _ref_options(**over)
    cwd = os.getcwd()
    os.chdir(workdir)
    try:
        ad = _make_reference_adaptor(workdir, opts)
    finally:
        os.chdir(cwd)
    stream = synthetic.SyntheticStream(length=n_frames, batch_size=opts.batch_size)
    oracle = adaptor_ref.OracleAdaptor(
        opts, synthetic.make_basemodel(), {g: synthetic.make_smpl_model(g) for g in ('neutral', 'male', 'female')},
        synthetic.make_extra_regressors(), dict(np.load(os.path.join(REPO, 'dynaboa_b200/assets/gmm_08.npz'))),
        bank=synthetic.make_exemplar_bank(), clusters=synthetic.make_clusters(), joint_map=C.JOINT_MAP_49,
        vertex_ids=C.SMPL_EXTRA_VERTEX_IDS, h36m_to_j14=C.H36M_TO_J14)
    oracle.mask_fn = _seeded_masks
    names = [k for k, _ in ad.model.module.named_parameters()]
    rec = {k: [] for k in ('metrics', 'upper_loss', 'lower_loss0', 'rotmat', 'betas', 'cam', 'joints', 'verts_sub',
                           'theta_samples', 'grad_samples', 'grad_norms', 'dyn_steps', 'cos12')}
    masks_all = []
    for t in range(n_frames):
        batch = stream[t]
        # --- reference
        random.seed(1000 + t); torch.manual_seed(1000 + t)
        ad.global_step, ad.fit_losses = t, {}
        ad.model.eval()
        os.chdir(workdir)
        try:
            mpjpe, pampjpe, pve = ad.adaptation(batch)
        finally:
            os.chdir(cwd)
        ref_upper = ad.fit_losses.get('ul/unlabelloss')
        # --- oracle restatement on the same RNG streams
        random.seed(1000 + t); torch.manual_seed(1000 + t)
        oracle.global_step, oracle.fit_losses = t, {}
        orec = oracle.adaptation(batch, with_inference=True)
        # record the teacher masks this frame consumed (replayed by the GPU parity test)
        torch.manual_seed(1000 + t)
        n_teacher = 1 + orec['dynamic_steps'] if (opts.use_meanteacher and opts.use_temporal_losses_upper) else 0
        masks_all.append(np.stack([np.stack([np.stack([m.numpy() for m in pair]) for pair in _seeded_masks(opts.batch_size)])
                                   for _ in range(max(n_teacher, 1))]))
        # --- compare trajectories
        # Adam moves every weight by ~lr per outer step in the direction of sign(g), so fp32 rounding
        # noise in near-zero gradients can flip individual entries: bound |diff| by the steps taken.
        n_outer = sum(1 + d for d in rec['dyn_steps']) + 1 + orec['dynamic_steps']
        bound = 4 * opts.lr * n_outer
        for k, p in ad.model.module.named_parameters():
            err = (oracle.theta[k].detach() - p.detach()).abs().max().item()
            assert err <= bound, f'{tag} frame {t} theta[{k}] err {err:.3e} > {bound:.3e}'
        for k, p in ad.teacher.named_parameters():
            err = (oracle.teacher[k] - p.detach()).abs().max().item()
            assert err <= bound, f'{tag} frame {t} teacher[{k}] err {err:.3e} > {bound:.3e}'
        _same(orec['metrics'][-1][0], mpjpe, f'{tag} mpjpe', tol=1e-3)
        _same(orec['metrics'][-1][1], pampjpe, f'{tag} pampjpe', tol=1e-3)
        if ref_upper is not None:
            # the reference accumulates the later terms IN PLACE into this logged tensor
            # (base_adaptor.py:303,308,315 ``loss +=``), so it holds the total upper-level loss
            if orec['dynamic_steps'] == 0:
                _same(orec['upper_loss'], ref_upper, f'{tag} upper loss', tol=1e-3)
        pred = oracle.predict(batch['image'])
        with torch.no_grad():
            r_rot, r_shape, r_cam = ad.model(batch['image'])
            r_out = ad.decode_smpl_params(r_rot, r_shape)
        _same(pred['rotmat'], r_rot, f'{tag} pred rotmat', tol=1e-3)
        _same(pred['joints'], r_out['s3d'], f'{tag} pred joints', tol=1e-3)
        _same(pred['vertices'], r_out['vts'], f'{tag} pred verts', tol=1e-3)
        rec['metrics'].append(np.stack([np.asarray(m[0]).reshape(-1) for m in [(mpjpe,), (pampjpe,), (np.asarray(pve),)]]))
        rec['upper_loss'].append(orec['upper_loss'])
        rec['lower_loss0'].append(orec['lower_losses'][0] if orec['lower_losses'] else 0.0)
        rec['rotmat'].append(r_rot.numpy()); rec['betas'].append(r_shape.numpy()); rec['cam'].append(r_cam.numpy())
        rec['joints'].append(r_out['s3d'].numpy()); rec['verts_sub'].append(r_out['vts'][:, ::10].numpy())
        params = list(ad.model.module.named_parameters())
        rec['theta_samples'].append(_theta_samples(params))
        rec['grad_samples'].append(_theta_samples([(k, p.grad) for k, p in params]))
        rec['grad_norms'].append(np.array([p.grad.double().norm().item() for _, p in params]))
        rec['dyn_steps'].append(orec['dynamic_steps'])
        rec['cos12'].append(orec['cos'][0][12] if orec['cos'] else 1.0)
        print(f'  {tag} frame {t}: upper={orec["upper_loss"]:.6f} mpjpe={float(np.mean(mpjpe)):.3f} '
              f'pampjpe={float(np.mean(pampjpe)):.3f} dyn={orec["dynamic_steps"]}')
    maxm = max(m.shape[0] for m in masks_all)
    masks = np.zeros((n_frames, maxm) + masks_all[0].shape[1:], np.float32)
    for t, m in enumerate(masks_all):
        masks[t, :m.shape[0]] = m
    np.savez_compressed(os.path.join(OUT, f'adapt_{tag}.npz'), param_names=np.array(names),
                        options=np.array(repr(sorted(vars(opts).items()))),
                        teacher_masks=masks.astype(np.uint8),
                        **{k: np.stack([np.asarray(x) for x in v]) for k, v in rec.items()})
    print(f'adapt {tag} ok')


def golden_dp(R=2, n_frames=3):
    """Data-parallel trajectory (oracle/dp_ref.py: R replicas in lock step, rank-mean outer gradient, rank-summed cosine
    terms): 1 inner step, deterministic teacher, dynamic loop armed with a low threshold so that it fires.  The reference has no
    distributed mode; this fixture pins the B200 implementation's NCCL path to the CPU emulation of SURVEY.md section 8e."""
    from oracle import dp_ref
    opts = adaptor_ref.default_options(inner_step=1, retrieval=0, lower_level_mixtrain=0, upper_level_mixtrain=0, dynamic_boa=1,
                                       cos_sim_threshold=1e-7, optim_steps=2, teacher_dropout=0)
    streams = [synthetic.SyntheticStream(length=n_frames, batch_size=1, rank=r) for r in range(R)]

    def make(rank):
        return adaptor_ref.OracleAdaptor(
            opts, synthetic.make_basemodel(), {g: synthetic.make_smpl_model(g) for g in ('neutral', 'male', 'female')},
            synthetic.make_extra_regressors(), dict(np.load(os.path.join(REPO, 'dynaboa_b200/assets/gmm_08.npz'))),
            joint_map=C.JOINT_MAP_49, vertex_ids=C.SMPL_EXTRA_VERTEX_IDS, h36m_to_j14=C.H36M_TO_J14)
    records, oracles = dp_ref.run(make, streams, n_frames)
    names = list(oracles[0].theta.keys())
    for k in names:                                        # replicas must stay identical
        assert torch.equal(oracles[0].theta[k], oracles[1].theta[k]), k
    out = dict(options=np.array(repr(sorted(vars(opts).items()))), param_names=np.array(names),
               dyn_steps=np.array([[rec['dynamic_steps'] for rec in records[r]] for r in range(R)]),
               upper_loss=np.array([[rec['upper_loss'] for rec in records[r]] for r in range(R)]),
               theta_samples=_theta_samples([(k, oracles[0].theta[k]) for k in names]))
    for r in range(R):
        pred = oracles[r].predict(streams[r][n_frames - 1]['image'])
        for key in ('rotmat', 'betas', 'cam', 'joints'):
            out[f'{key}_r{r}'] = pred[key].numpy()
    assert (out['dyn_steps'][0] == out['dyn_steps'][1]).all()
    np.savez_compressed(os.path.join(OUT, 'adapt_dp2.npz'), **out)
    print('adapt dp2 ok: dynamic steps', out['dyn_steps'].tolist(), 'upper', out['upper_loss'].tolist())


def golden_dataprocess():
    """Input side: the reference's OWN crop / transform code (utils/dataprocess.py, imported unmodified with
    skimage.transform.resize -- not installed here -- stubbed by its scipy restatement) on a seeded image; asserts the oracle
    restatement reproduces it and stores inputs + outputs."""
    import types
    from oracle import dataprocess_ref as R
    sk, skt = types.ModuleType('skimage'), types.ModuleType('skimage.transform')
    skt.resize = lambda img, res: R.resize(img, res)
    sk.transform = skt
    sys.modules.setdefault('skimage', sk); sys.modules.setdefault('skimage.transform', skt)
    if 'constants' not in sys.modules:            # the reference module does `import constants` (its own constants.py)
        sys.modules['constants'] = _load_by_path('constants', os.path.join(REF, 'constants.py'))
    ref = _load_by_path('ref_dataprocess', os.path.join(REF, 'utils', 'dataprocess.py'))
    rng = np.random.default_rng(7)
    img = rng.uniform(0, 255, size=(120, 160, 3)).astype(np.float32)
    boxes = [([80.0, 60.0], 0.5), ([20.0, 100.0], 0.8), ([150.5, 10.25], 0.35), ([81.0, 59.0], 1.3), ([60.0, 60.0], 0.2)]
    kp = np.concatenate([rng.uniform(-10, 170, size=(49, 2)), (rng.random((49, 1)) > 0.3).astype(np.float64)], 1)
    crops, kps = [], []
    for center, scale in boxes:
        a = ref.crop(img.copy(), center, scale, [224, 224])
        b = R.crop(img.copy(), center, scale, [224, 224])
        assert np.array_equal(a, b), (center, scale)
        rgb = np.transpose(a.astype('float32'), (2, 0, 1)) / 255.0
        rgb = (rgb - R.IMG_NORM_MEAN[:, None, None].astype('float32')) / R.IMG_NORM_STD[:, None, None].astype('float32')
        assert np.array_equal(rgb.astype('float32'), R.rgb_processing(img, center, scale))
        ka = kp.copy()
        for i in range(ka.shape[0]):
            ka[i, 0:2] = ref.transform(ka[i, 0:2] + 1, center, scale, [224, 224])
        ka[:, :-1] = 2. * ka[:, :-1] / 224 - 1.
        assert np.array_equal(ka.astype('float32'), R.j2d_processing(kp, center, scale))
        crops.append(R.rgb_processing(img, center, scale)[:, ::4, ::4])
        kps.append(ka.astype('float32'))
    np.savez_compressed(os.path.join(OUT, 'dataprocess.npz'), img=img, kp=kp, centers=np.array([b[0] for b in boxes]),
                        scales=np.array([b[1] for b in boxes]), crops_sub=np.stack(crops), kps=np.stack(kps))
    print('dataprocess.npz ok')


def golden_eval():
    """Evaluation metrics: the reference's own Procrustes (utils/pose_utils.py) inside the arithmetic of
    dynaboa_benchmark.py:217-240, on seeded meshes (small vertex count keeps the fixture small).  Sample 2 is a mirrored
    copy of its ground truth (det(U V^T) < 0: the orientation fix is exercised), sample 3 a similarity transform of it."""
    ref = _load_by_path('ref_pose_utils', os.path.join(REF, 'utils', 'pose_utils.py'))
    rng = np.random.RandomState(5)
    B, NV, NJ = 5, 640, 17
    jmap = np.asarray(C.H36M_TO_J14, dtype=np.int64)
    J = rng.rand(NJ, NV).astype(np.float32) ** 8
    J /= J.sum(1, keepdims=True)
    gt = (rng.randn(B, NV, 3) * 0.4).astype(np.float32)
    pred = (gt + rng.randn(B, NV, 3) * 0.05).astype(np.float32)
    pred[2] = gt[2] * np.array([-1.0, 1.0, 1.0], dtype=np.float32)
    q, _ = np.linalg.qr(rng.randn(3, 3))
    q *= np.sign(np.linalg.det(q))
    pred[3] = (1.7 * gt[3].dot(q.T) + np.array([0.3, -0.2, 0.1])).astype(np.float32)
    gt_neutral = (gt + rng.randn(B, NV, 3) * 0.01).astype(np.float32)
    # reference arithmetic with the reference's own Procrustes
    gt_k = np.matmul(J[None], gt)
    gt_k = gt_k[:, jmap] - gt_k[:, [0]]
    pr_k = np.matmul(J[None], pred)
    pr_k = pr_k[:, jmap] - pr_k[:, [0]]
    mpjpe = np.sqrt(((pr_k - gt_k) ** 2).sum(-1)).mean(-1)
    hat = ref.compute_similarity_transform_batch(pr_k, gt_k)
    pampjpe = np.sqrt(((hat - gt_k) ** 2).sum(-1)).mean(-1)
    pve = np.sqrt(np.sum((gt_neutral - pred) ** 2, axis=2)).mean()
    m2, p2, v2 = eval_ref.eval_metrics(pred, gt, gt_neutral, J, jmap)
    _same(m2, mpjpe, 'eval mpjpe', 1e-6)
    _same(p2, pampjpe, 'eval pampjpe', 1e-5)
    _same(v2, pve, 'eval pve', 1e-6)
    assert pampjpe[3] < 1e-5 * np.abs(gt_k[3]).max() * 50, 'a similarity transform must align exactly'
    np.savez_compressed(os.path.join(OUT, 'eval_metrics.npz'), pred=pred, gt=gt, gt_neutral=gt_neutral, J=J, joint_map=jmap,
                        mpjpe=mpjpe, pampjpe=pampjpe, pve=np.float64(pve))
    print('eval_metrics.npz', mpjpe, pampjpe, pve)


# ---------------------------------------------------------------------------------------
# part 3: the webcam client -- the reference ``Adaptor`` CLASS of dynaboa_webcam.py executed unmodified on CPU
# ---------------------------------------------------------------------------------------
def _load_webcam_class():
    """dynaboa_webcam.py cannot be imported (cv2, OpenPose bindings, an ffmpeg loop at import): take its ``Adaptor`` class
    definition out of the syntax tree and execute exactly that, in a namespace holding the names its methods use."""
    import ast
    from torchvision.transforms import Normalize
    sys.path.insert(0, REF)
    geometry = importlib.import_module('utils.geometry')
    model = importlib.import_module('model')
    prior = importlib.import_module('utils.smplify.prior')
    path = os.path.join(REF, 'dynaboa_webcam.py')
    tree = ast.parse(open(path).read())
    cls = next(n for n in tree.body if isinstance(n, ast.ClassDef) and n.name == 'Adaptor')
    ns = dict(torch=torch, nn=torch.nn, F=torch.nn.functional, np=np, random=random, os=os, l2l=sys.modules['learn2learn'],
              Normalize=Normalize, constants=importlib.import_module('constants'), config=importlib.import_module('config'),
              hmr=model.hmr, SMPL=model.SMPL, MaxMixturePrior=prior.MaxMixturePrior,
              perspective_projection=geometry.perspective_projection,
              rotation_matrix_to_angle_axis=geometry.rotation_matrix_to_angle_axis, crop=None, transform=None)
    exec(compile(ast.Module(body=[cls], type_ignores=[]), path, 'exec'), ns)
    return ns['Adaptor'], ns


def webcam_detections(batch, t):
    """(B, 25, 3) OpenPose-style detections of a synthetic frame: the projected OpenPose joints with noise, some of them
    undetected (confidence 0) in a pattern that changes from frame to frame."""
    kp = batch['op_j2d'][:, :25].clone()
    kp[:, (3 * t) % 25, 2] = 0.0
    kp[:, (7 * t + 11) % 25, 2] = 0.0
    return kp


def golden_webcam(workdir, n_frames=6):
    from . import webcam_ref
    opts = webcam_ref.webcam_options(interval=2, dynamic_boa=1, cos_sim_threshold=1e-7, optim_steps=2)
    opts.model_file, opts.test_basemodel = 'data/basemodel.pt', 0
    cwd = os.getcwd()
    os.chdir(workdir)
    try:
        if not os.path.exists('data/gmm_08.pkl'):
            os.symlink(os.path.join(REF, 'data/gmm_08.pkl'), 'data/gmm_08.pkl')
        RefAdaptor, ns = _load_webcam_class()
        ad = RefAdaptor.__new__(RefAdaptor)
        ad.options, ad.device = opts, torch.device('cpu')
        ad.seed_everything(opts.seed)
        ad.history, ad.global_step = {}, 0
        # _initialize_training (:45-83) with the device fixed to the CPU instead of 'cuda'
        ck = torch.load(opts.model_file, weights_only=False)
        ad.model = ns['l2l'].algorithms.MAML(ns['hmr'](ns['config'].SMPL_MEAN_PARAMS), lr=opts.fastlr, first_order=True)
        ad.model.load_state_dict(ck['model'], strict=True)
        ad.model.eval()
        ad.teacher = ns['hmr'](ns['config'].SMPL_MEAN_PARAMS)
        for p in ad.teacher.parameters():
            p.detach_()
        ad.teacher.load_state_dict({k.replace('module.', ''): v for k, v in ck['model'].items()}, strict=True)
        ad.teacher.eval()
        ad.optimizer = torch.optim.Adam(ad.model.parameters(), lr=opts.lr, betas=(opts.beta1, opts.beta2))
        ad.gmm_f = ns['MaxMixturePrior'](prior_folder='data/', num_gaussians=8, dtype=torch.float32)
        ad.smpl_neutral = ns['SMPL'](ns['config'].SMPL_MODEL_DIR, create_transl=False)
    finally:
        os.chdir(cwd)
    oracle = webcam_ref.OracleWebcam(
        opts, synthetic.make_basemodel(), {g: synthetic.make_smpl_model(g) for g in ('neutral', 'male', 'female')},
        synthetic.make_extra_regressors(), dict(np.load(os.path.join(REPO, 'dynaboa_b200/assets/gmm_08.npz'))),
        joint_map=C.JOINT_MAP_49, vertex_ids=C.SMPL_EXTRA_VERTEX_IDS, h36m_to_j14=C.H36M_TO_J14)
    stream = synthetic.SyntheticStream(length=n_frames, batch_size=1)
    names = [k for k, _ in ad.model.module.named_parameters()]
    rec = {k: [] for k in ('kp25', 'verts_sub', 'cam', 'theta_samples', 'dyn_steps')}
    n_outer = 0
    for t in range(n_frames):
        batch = stream[t]
        kp = webcam_detections(batch, t)
        # the input processing (:197-218) is replaced by already processed tensors: skimage is not in this image, the crop is
        # pinned separately (golden_dataprocess); everything from save_hist on is the reference's code
        ad.dataprocess = lambda img, k, scaleFactor=1.0, _b=batch, _k=kp: (_b['image'].clone(), _k.clone(), np.array([[112., 112., 200.]]))
        ad.optimized_step = 0
        res = ad.online_adaptation(None, np.zeros((1, 25, 3)))
        steps = oracle.online_adaptation(batch['image'], kp)
        dyn = min(int(ad.optimized_step), opts.optim_steps)
        assert dyn == min(steps, opts.optim_steps), (t, ad.optimized_step, steps)
        n_outer += 1 + dyn
        bound = 4 * opts.lr * n_outer
        for k, p in ad.model.module.named_parameters():
            err = (oracle.theta[k].detach() - p.detach()).abs().max().item()
            assert err <= bound, f'webcam frame {t} theta[{k}] err {err:.3e} > {bound:.3e}'
        for k, p in ad.teacher.named_parameters():
            assert (oracle.teacher[k] - p.detach()).abs().max().item() <= bound, (t, k)
        pred = oracle.predict(batch['image'])
        _same(pred['vertices'], res['vts'].detach(), 'webcam verts', tol=1e-3)
        rec['kp25'].append(kp.numpy()); rec['verts_sub'].append(res['vts'].detach()[:, ::10].numpy()); rec['cam'].append(res['cam'].detach().numpy())
        rec['theta_samples'].append(_theta_samples(list(ad.model.module.named_parameters())))
        rec['dyn_steps'].append(dyn)
        print(f'  webcam frame {t}: dyn={dyn} |cam|={float(res["cam"].abs().sum()):.5f}')
    np.savez_compressed(os.path.join(OUT, 'adapt_webcam.npz'), param_names=np.array(names),
                        options=np.array(repr(sorted(vars(opts).items()))), **{k: np.stack([np.asarray(x) for x in v]) for k, v in rec.items()})
    print('adapt webcam ok')


# ---------------------------------------------------------------------------------------
# part 4: the interface of the unchanged driver (read from its syntax tree, never executed)
# ---------------------------------------------------------------------------------------
def golden_driver_surface():
    import ast
    tree = ast.parse(open(os.path.join(REF, 'dynaboa_benchmark.py')).read())
    used, assigned = set(), set()
    for node in ast.walk(tree):
        if isinstance(node, ast.Attribute) and isinstance(node.value, ast.Name) and node.value.id == 'self':
            (assigned if isinstance(node.ctx, ast.Store) else used).add(node.attr)
    methods = {n.name for c in tree.body if isinstance(c, ast.ClassDef) for n in c.body if isinstance(n, ast.FunctionDef)}
    imports = set()
    for node in tree.body:
        if isinstance(node, ast.ImportFrom):
            imports.add(node.module)
        elif isinstance(node, ast.Import):
            imports.update(a.name for a in node.names)
    names = dict(self_used=used, self_assigned=assigned, driver_methods=methods, imports=imports)
    np.savez_compressed(os.path.join(OUT, 'driver_surface.npz'), **{k: np.array(sorted(v), dtype=str) for k, v in names.items()})
    print('driver_surface.npz', {k: len(v) for k, v in names.items()})


def main():
    assert REF and os.path.isdir(REF), 'set DBOA_REFERENCE_ROOT to a checkout of the reference'
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(os.cpu_count())
    workdir = tempfile.mkdtemp(prefix='dboa_golden_')
    try:
        synthetic.write_asset_dir(os.path.join(workdir, 'data'))
        os.makedirs(os.path.join(workdir, 'data/spin_data'), exist_ok=True)
        os.symlink(os.path.join(REF, 'data/gmm_08.pkl'), os.path.join(workdir, 'data/spin_data/gmm_08.pkl'))
        which = sys.argv[1:] or ['geometry', 'prior', 'hmr', 'smpl', 'eval', 'c2', 'c3', 'c5', 'dp2', 'dataprocess', 'webcam', 'surface']
        if 'surface' in which:
            golden_driver_surface()
        if 'dp2' in which:
            golden_dp()
        if 'dataprocess' in which:
            golden_dataprocess()
        if 'geometry' in which:
            golden_geometry()
        if 'prior' in which:
            golden_prior(workdir)
        if 'hmr' in which:
            golden_hmr(workdir)
        if 'smpl' in which:
            golden_smpl()
        if 'eval' in which:
            golden_eval()
        _install_stubs()
        if 'c2' in which:   # BASELINE.json configs[1]
            golden_adapt(workdir, 'c2', 8, inner_step=1, retrieval=0, lower_level_mixtrain=0,
                         upper_level_mixtrain=0, dynamic_boa=0)
        if 'c3' in which:   # BASELINE.json configs[2]: 3 inner steps, retrieval minibatch of 8 exemplars
            golden_adapt(workdir, 'c3', 2, inner_step=3, retrieval=1, sample_num=8, lower_level_mixtrain=1,
                         upper_level_mixtrain=1, dynamic_boa=0)
        if 'c5' in which:   # dynamic loop exercised (threshold lowered so it fires on random weights)
            golden_adapt(workdir, 'c5', 2, inner_step=1, retrieval=1, sample_num=1, lower_level_mixtrain=1,
                         upper_level_mixtrain=1, dynamic_boa=1, cos_sim_threshold=1e-7, optim_steps=2)
        if 'webcam' in which:   # third client (dynaboa_webcam.py): OpenPose joints, motion + teacher in the upper level, dynamic loop
            golden_webcam(workdir)
    finally:
        shutil.rmtree(workdir, ignore_errors=True)


if __name__ == '__main__':
    main()
