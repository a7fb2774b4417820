"""Static check of the drop-in boundary (SURVEY.md §8b): every attribute / method the UNCHANGED reference
driver touches on ``self`` exists on our BaseAdaptor (or is created by the driver itself), and every module it
imports resolves inside dynaboa_b200/dropin.  The driver's side of the boundary is the fixture
tests/golden/driver_surface.npz, read from its syntax tree by oracle/make_golden.py; the reference is never executed."""
import ast
import os
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_driver_surface_is_provided(golden):
    ref = golden('driver_surface')
    used, assigned, driver_methods = ({str(s) for s in ref[k]} for k in ('self_used', 'self_assigned', 'driver_methods'))
    src = open(os.path.join(REPO, 'dynaboa_b200', 'base_adaptor.py')).read()
    base = ast.parse(src)
    provided = {n.name for c in base.body if isinstance(c, ast.ClassDef) and c.name == 'BaseAdaptor' for n in c.body
                if isinstance(n, ast.FunctionDef)}
    for node in ast.walk(base):
        if isinstance(node, ast.Attribute) and isinstance(node.value, ast.Name) and node.value.id == 'self' and isinstance(node.ctx, ast.Store):
            provided.add(node.attr)
    dead = {'load_ckpt'}     # reference dead code (dynaboa_benchmark.py:102-103, never reached: self.load is False)
    missing = used - assigned - driver_methods - provided - dead
    assert not missing, f'reference driver uses self.{sorted(missing)} which BaseAdaptor does not provide'
    dropin = os.path.join(REPO, 'dynaboa_b200', 'dropin')
    for m in (str(s) for s in ref['imports']):
        top = m.split('.')[0]
        if top in ('constants', 'utils', 'base_adaptor', 'model', 'config', 'boa_dataset'):
            path = os.path.join(dropin, *m.split('.'))
            assert os.path.exists(path + '.py') or os.path.isdir(path), f'drop-in tree lacks module {m}'


def test_dropin_modules_import_without_gpu():
    names = ('constants', 'config', 'model', 'model.hmr', 'model.smpl', 'utils', 'utils.geometry', 'utils.pose_utils', 'utils.smplify',
             'utils.smplify.prior', 'base_adaptor', 'boa_dataset', 'boa_dataset.pw3d', 'learn2learn', 'learn2learn.algorithms')
    saved = {m: sys.modules.pop(m) for m in names if m in sys.modules}
    sys.path.insert(0, os.path.join(REPO, 'dynaboa_b200', 'dropin'))
    try:
        import importlib
        for m in names:
            importlib.import_module(m)
        import base_adaptor
        import learn2learn as l2l
        assert hasattr(base_adaptor, 'BaseAdaptor') and hasattr(l2l.algorithms, 'MAML')
    finally:
        sys.path.pop(0)
        for m in names:
            sys.modules.pop(m, None)
        sys.modules.update(saved)


def test_maml_learner_exposes_fast_weights():
    """learn2learn's cloned module yields its fast (non-leaf) weights from parameters() / named_parameters(); the wrapper
    does the same for a learner and keeps nn.Module's leaf traversal for the meta-model (reference: l2l 0.1.5 BaseLearner /
    clone_module as used at base_adaptor.py:119, dynaboa_benchmark.py:136).  CPU only: the learner state is emulated with a
    flat arena, the clone itself is a CUDA call."""
    from dynaboa_b200 import hmr as hmr_mod, maml, synthetic
    m = hmr_mod.hmr(synthetic.make_mean_params())
    mm = maml.MAML(m, lr=1e-3, first_order=True)
    leaf = list(mm.named_parameters())
    assert len(leaf) == 169 and leaf[0][0] == 'module.conv1.weight' and all(p.is_leaf for _, p in leaf)
    object.__setattr__(m, '_fast', m.arena.detach().clone().requires_grad_() * 1.0)
    try:
        fast = list(mm.named_parameters())
        assert [n for n, _ in fast] == [n for n, _ in leaf]
        assert all(not p.is_leaf for _, p in fast) and [tuple(p.shape) for _, p in fast] == [tuple(p.shape) for _, p in leaf]
        assert len(list(mm.parameters())) == 169
    finally:
        object.__setattr__(m, '_fast', None)
