"""The reference's OWN adaptor code on CPU (test / benchmark infrastructure only; never imported by the product).

``make_reference_adaptor`` builds ``dynaboa_benchmark.Adaptor`` from the reference tree -- a checkout named by
``DBOA_REFERENCE_ROOT``, else the bytecode build() made under the git-ignored ``oracle/_ref/`` (oracle/build_ref.py) -- with the
constructor's I/O replaced: the two third-party packages that are not in this image (``smplx``,
``learn2learn``) are the restatements of this package, the datasets are the synthetic stream / exemplar bank, the device is the
CPU.  Everything that runs per frame -- ``model/hmr.py``, ``base_adaptor.BaseAdaptor``'s losses and levels,
``dynaboa_benchmark.Adaptor.adaptation`` / ``inference``, ``utils/geometry.py``, ``utils/smplify/prior.py``,
``utils/pose_utils.py`` -- is the reference's unmodified code.  Used by oracle/make_golden.py (golden trajectories) and by
``bench.py`` (``cpu_baseline.kind = "reference"``, ``--impl reference``).
"""
import importlib
import os
import sys
import types

import numpy as np
import torch

from dynaboa_b200 import constants as C
from dynaboa_b200 import synthetic
from . import adaptor_ref, l2l_ref, smplx_ref


BUILT = os.path.join(os.path.dirname(os.path.abspath(__file__)), '_ref')      # made by build() (oracle/build_ref.py)


def _module_file(root, name):
    """``<root>/<name>.py``, or its bytecode ``<root>/<name>.pyc`` (the form under oracle/_ref); None when neither exists."""
    for ext in ('.py', '.pyc'):
        path = os.path.join(root, name + ext)
        if os.path.exists(path):
            return path
    return None


def reference_root():
    """The reference checkout named by DBOA_REFERENCE_ROOT, else the reference files build() compiled into oracle/_ref/, else
    None (``DBOA_REFERENCE_ROOT=none`` disables both): the callers then fall back to the oracle port or skip."""
    env = os.environ.get('DBOA_REFERENCE_ROOT')
    if env == 'none':
        return None
    for root in (env, BUILT):
        if root and _module_file(root, 'dynaboa_benchmark') and _module_file(root, os.path.join('model', 'hmr')):
            return root
    return None


REF = reference_root()


def available():
    return REF is not None


def driver(name):
    """Path of the reference's driver script ``name`` (``dynaboa_benchmark``, ``dynaboa_internet``), or None."""
    return _module_file(REF, name) if REF else None


class _StubSMPLX(torch.nn.Module):
    """Stand-in for ``smplx.SMPL`` (45-joint output) built on the restatement."""

    def __init__(self, model_path, gender='neutral', create_transl=False, batch_size=1, **kw):
        super().__init__()
        data = dict(np.load(os.path.join(model_path, f'SMPL_{gender.upper()}.npz')))
        for k in ('v_template', 'shapedirs', 'posedirs', 'J_regressor', 'lbs_weights'):
            self.register_buffer(k, torch.as_tensor(data[k]))
        self.register_buffer('parents', torch.as_tensor(data['parents'], dtype=torch.long))
        self.faces = data['faces']
        self._vid = torch.as_tensor(C.SMPL_EXTRA_VERTEX_IDS, dtype=torch.long)

    def forward(self, betas=None, body_pose=None, global_orient=None, pose2rot=True, **kw):
        m = {k: getattr(self, k) for k in ('v_template', 'shapedirs', 'posedirs', 'J_regressor', 'parents',
                                           'lbs_weights')}
        full_pose = torch.cat([global_orient, body_pose], dim=1)
        verts, J_tr = smplx_ref.lbs(betas, full_pose, m, pose2rot)
        joints = torch.cat([J_tr, verts[:, self._vid]], dim=1)
        return types.SimpleNamespace(vertices=verts, joints=joints, betas=betas, global_orient=global_orient,
                                     body_pose=body_pose, full_pose=full_pose)


def install_stubs():
    def mod(name, **attrs):
        m = types.ModuleType(name)
        m.__dict__.update(attrs)
        sys.modules[name] = m
        return m
    alg = mod('learn2learn.algorithms', MAML=l2l_ref.MAML)
    mod('learn2learn', algorithms=alg)

    def SMPLOutput(**kw):
        return types.SimpleNamespace(**kw)
    mod('smplx.utils', SMPLOutput=SMPLOutput)
    mod('smplx.lbs', vertices2joints=lambda Jr, v: torch.einsum('bik,ji->bjk', v, Jr))
    mod('smplx', SMPL=_StubSMPLX)
    mod('skimage.transform', resize=None)
    mod('skimage')
    mod('trimesh')
    mod('pyrender.constants', RenderFlags=None)
    mod('pyrender')
    mod('render_demo', Renderer=None, convert_crop_cam_to_orig_img=None)   # viz only (save_res=0)
    mod('human_body_prior.tools.model_loader', load_vposer=None)
    mod('human_body_prior.tools')
    mod('human_body_prior')


class _FakeH36M:
    """Stands in for ``SourceDataset`` (JPEG decoding is out of scope): tensor-only items with the
    leading axis of 1 the reference's ``__getitem__`` produces (base_adaptor.py:492-504)."""

    def __init__(self, bank):
        self.bank = bank

    def __getitem__(self, i):
        return {k: v[i:i + 1].clone() for k, v in self.bank.items()}


def make_reference_adaptor(workdir, opts, n_exemplars=64):
    """``dynaboa_benchmark.Adaptor`` of the reference on the CPU.  ``workdir`` holds ``data/`` (synthetic.write_asset_dir) and
    ``data/spin_data/gmm_08.pkl``; the reference resolves its assets relative to the working directory, so callers run the
    adaptor's methods with ``workdir`` as the current directory (``in_dir`` below)."""
    if REF not in sys.path:
        sys.path.insert(0, REF)
    install_stubs()
    with in_dir(workdir):
        gmm = os.path.join('data', 'spin_data', 'gmm_08.pkl')
        if not os.path.exists(gmm):
            os.makedirs(os.path.dirname(gmm), exist_ok=True)
            os.symlink(os.path.join(REF, 'data', 'gmm_08.pkl'), gmm)
        bench = importlib.import_module('dynaboa_benchmark')
        ad = bench.Adaptor.__new__(bench.Adaptor)
        ad.options = opts
        ad.exppath = os.path.join(workdir, 'exp')
        os.makedirs(os.path.join(ad.exppath, 'result'), exist_ok=True)
        ad.device = torch.device('cpu')
        ad.seed_everything(opts.seed)
        ad.options.mixtrain = opts.lower_level_mixtrain or opts.upper_level_mixtrain
        cl = synthetic.make_clusters(n_exemplars)
        ad.centers = torch.from_numpy(cl['centers']).float()
        ad.index = cl['index']
        ad.h36m_dataset = _FakeH36M(synthetic.make_exemplar_bank(n_exemplars))
        ad.set_model_optim()
        ad.set_teacher()
        ad.set_criterion()
        ad.setup_smpl()
    ad.history, ad.kp2dlosses_lower, ad.kp2dlosses_upper = {}, [], {}
    ad.feat_sims, ad.optim_step_record = {}, []
    ad.mpjpe_all_lower = [[] for _ in range(opts.inner_step)]
    ad.pampjpe_all_lower = [[] for _ in range(opts.inner_step)]
    ad.mpjpe_statistics, ad.pampjpe_statistics = {}, {}
    return ad


class in_dir:
    def __init__(self, path):
        self.path = path

    def __enter__(self):
        self.prev = os.getcwd()
        os.chdir(self.path)

    def __exit__(self, *exc):
        os.chdir(self.prev)


def ref_options(**over):
    o = adaptor_ref.default_options(**over)
    o.expdir, o.expname, o.dataset, o.model_file, o.save_res = 'exps', 'x', '3dpw', 'data/basemodel.pt', 0
    o.record_lowerlevel, o.seq_seed = 1, 22
    return o
