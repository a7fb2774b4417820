"""Split-K plans of the tcgen05 kernels: the fused forward convolution (csrc/conv_wide.cu), the fused data gradient
(csrc/dgrad_wide.cu) and the weight gradient (csrc/conv_wgrad_wide.cu).

A launch splits the reduction of every output tile into nz K-slices (one thread-block cluster, reduced through distributed
shared memory) of `per` k-blocks each; the last slice may be shorter.  The plan follows from the shape, the batch, the SM count
and the CTA budgets, so at the default budgets each shape exercises one plan.  Here dboa_set_split_limits forces nz = 1 .. 16 on
ResNet-50 layer geometries, dboa_last_wide_plan confirms that the intended plan ran, and every output is checked against an fp64
restatement (the references and tolerances of tests/test_gpu_fused.py), inside guard bands that must stay bit-for-bit intact,
and for run-to-run determinism.  The whole network then runs under the widest and the narrowest plans against the CPU oracle."""
import ctypes as C
import math

import pytest
import torch
import torch.nn.functional as F

from conftest import rel_err

pytestmark = pytest.mark.gpu

DMAX = {0: 4, 1: 3, 2: 2}                 # operand ring depth of each kernel (wz::DMAX, dz::DMAX, the two wgrad stages)
NAMES = {0: 'forward', 1: 'dgrad', 2: 'wgrad'}
GUARD = 4096                              # sentinel elements before and after every output
FIX_FWD, FIX_BWD = 2.0 ** 24, 2.0 ** 28   # fixed-point scales of the forward statistics / backward sums
PLANS = []                                # (kernel, case id, plan) of every checked launch, for the coverage table


@pytest.fixture(scope='module')
def L():
    from dynaboa_b200 import _lib
    lib = _lib.load()
    assert lib.dboa_get_chain_flags() == 0
    try:
        yield _lib
    finally:
        for k in range(3):                # later modules run at the default plans
            lib.dboa_set_split_limits(k, -1, -1, -1)


def n_sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def force(L, kernel, nz):
    """limits under which the planner reaches `nz` where the shape allows it: a budget of every SM, at most nz slices, slices of
    one k-block and up"""
    L.call('dboa_set_split_limits', kernel, 0 if kernel == 0 else n_sms(), nz, 1)


def last_plan(L, kernel):
    out = (C.c_longlong * 5)()
    L.call('dboa_last_wide_plan', kernel, out)
    return dict(zip(('nz', 'per', 'D', 'grid', 'last'), (int(v) for v in out)))


def check_plan(L, kernel, case, nz, nkb, tiles):
    """the launch that just ran used nz slices of ceil(nkb / nz) k-blocks over `tiles` tiles"""
    p = last_plan(L, kernel)
    per = -(-nkb // nz)
    assert p['nz'] == nz, (NAMES[kernel], case, p)
    assert p['per'] == per and p['last'] == nkb - (nz - 1) * per and p['last'] >= 1, (NAMES[kernel], case, p)
    ring = p['D'] == DMAX[kernel] if kernel == 2 else 1 <= p['D'] <= min(per, DMAX[kernel])      # the weight gradient always has two stages
    assert p['grid'] == tiles * nz and ring, (NAMES[kernel], case, p)
    PLANS.append((kernel, case, p))


class Guarded:
    """an output tensor inside one larger buffer whose GUARD elements on either side hold random bits"""

    def __init__(self, shape, dtype=torch.float32, fill=float('nan'), init=None):
        n = math.prod(shape)
        ibits = torch.int32 if dtype == torch.float32 else torch.int64
        g = torch.Generator(device='cuda').manual_seed(n)
        bits = torch.randint(-2 ** 31, 2 ** 31 - 1, (n + 2 * GUARD,), generator=g, device='cuda', dtype=torch.int64)
        self.buf = bits.to(ibits).view(dtype)
        self.t = self.buf[GUARD:GUARD + n].view(shape)
        if init is not None:
            self.t.copy_(init)
        else:
            self.t.fill_(fill)
        self.sentinel = self.buf.view(ibits).clone()
        self.ibits = ibits

    def ptr(self):
        return self.t.data_ptr()

    def intact(self):
        b, s = self.buf.view(self.ibits), self.sentinel
        return torch.equal(b[:GUARD], s[:GUARD]) and torch.equal(b[-GUARD:], s[-GUARD:])


def check_guards(outs, tag):
    for name, g in outs.items():
        if g is not None:
            assert g.intact(), (tag, name, 'store outside the tensor')


def check_same(a, b, tag):
    """two runs of one launch on fresh buffers: bit-identical outputs (fixed-order DSMEM reduction, integer atomics)"""
    for name in a:
        if a[name] is not None:
            assert torch.equal(a[name].t.view(a[name].ibits), b[name].t.view(b[name].ibits)), (tag, name, 'not deterministic')


def nhwc(t):
    return t.permute(0, 3, 1, 2)


def wmat(w):
    return w.permute(0, 2, 3, 1).reshape(w.shape[0], -1).contiguous()


def group_view(t, B):
    """NHWC (B, H, W, C) -> (B, 4, H * W * C / 4) by GroupNorm group"""
    Cc = t.shape[-1]
    return t.double().reshape(B, -1, 4, Cc // 4).permute(0, 2, 1, 3).reshape(B, 4, -1)


def fixed_sums(x, B):
    """the accumulators a producing launch leaves for x: (sum, sum of squares) per (sample, group), 64-bit fixed point"""
    g = group_view(x, B)
    return (torch.stack([g.sum(-1), (g * g).sum(-1)], -1) * FIX_FWD).round().long().contiguous()


def gn(x, B, gamma, beta):
    """GroupNorm(4) of an NHWC tensor in fp64, and its (mean, rstd)"""
    g = group_view(x, B)
    mean, var = g.mean(-1), g.var(-1, unbiased=False)
    Cc = x.shape[-1]
    ex = lambda v: v.repeat_interleave(Cc // 4, dim=1)[:, None, None, :]
    rstd = 1.0 / (var + 1e-5).sqrt()
    return (x.double() - ex(mean)) * ex(rstd) * gamma.double() + beta.double(), torch.stack([mean, rstd], -1)


def check_conv(y, part_out, a_nhwc, w, stride, pad, B, tag):
    """y = conv(a, w) and the fixed-point statistics of y, as tests/test_gpu_fused.py checks them"""
    ref = F.conv2d(nhwc(a_nhwc).double(), w.double(), stride=stride, padding=pad)
    assert torch.isfinite(y).all(), tag
    assert rel_err(nhwc(y), ref) < 3e-5, tag
    acc = part_out.double().cpu() / FIX_FWD
    n = ref[0].numel() / 4
    mean, var = acc[..., 0] / n, acc[..., 1] / n - (acc[..., 0] / n) ** 2
    g = ref.reshape(B, 4, -1)
    rm, rv = g.mean(-1).cpu(), g.var(-1, unbiased=False).cpu()
    assert (mean - rm).abs().max() <= 1e-5 * rv.sqrt().max() + 1e-6, tag
    assert ((var - rv).abs() / rv).max() < 3e-5, tag


# ---------------------------------------------------------------------------------------------------------------------------
# forward: one problem in mode 1 (GroupNorm + ReLU of the operand on load, operand and statistics written to the tape)
# ---------------------------------------------------------------------------------------------------------------------------
def rows_of(Ho):
    return Ho if Ho * Ho <= 128 else 128 // Ho


def fwd_tiles(B, Ho, Cout):
    return B * -(-Ho // rows_of(Ho)) * (Cout // 64)


class FwdProb:
    def __init__(self, L, B, Hi, Cin, Cout, k, stride, mode, x, w, part_in, gamma, beta, res=None, part2_in=None, gamma2=None, beta2=None,
                 want_a=True):
        self.B, self.Ho, self.Cout = B, Hi // stride, Cout
        Ho = self.Ho
        self.out = {'y': Guarded((B, Ho, Ho, Cout)),
                    'part_out': Guarded((B, 4, 2), torch.int64, 0),
                    'a_out': Guarded((B, Hi, Hi, Cin)) if want_a else None,
                    'stats_out': Guarded((B, 4, 2)) if want_a else None,
                    'stats2_out': Guarded((B, 4, 2)) if want_a and mode == 3 else None}
        s = L.FusedConvStruct()
        for name, t in (('x', x), ('res', res), ('w', w), ('part_in', part_in), ('part2_in', part2_in), ('gamma', gamma), ('beta', beta),
                        ('gamma2', gamma2), ('beta2', beta2)):
            setattr(s, name, None if t is None else t.data_ptr())
        for name, g in self.out.items():
            setattr(s, name, None if g is None else g.ptr())
        s.mode, s.Hi, s.Cin, s.Cout, s.k, s.stride, s.pad = mode, Hi, Cin, Cout, k, stride, k // 2
        self.struct = s
        self.keep = (x, w, part_in, gamma, beta, res, part2_in, gamma2, beta2)


def fwd_launch(L, probs):
    arr = (L.FusedConvStruct * len(probs))(*[p.struct for p in probs])
    L.call('dboa_conv_fused_fwd', arr, len(probs), probs[0].B, L.stream())
    torch.cuda.synchronize()


FWD = [  # B, Hi, Cin, Cout, k, stride, nz           plan (per, last slice) at that nz
    (1, 7, 512, 512, 3, 1, 1), (1, 7, 512, 512, 3, 1, 2), (1, 7, 512, 512, 3, 1, 4), (1, 7, 512, 512, 3, 1, 8),
    (1, 7, 512, 512, 3, 1, 16),                      # 9, 9: 16-CTA cluster, slices longer than the ring
    (1, 14, 512, 512, 3, 2, 16),                     # stride 2 (layer4.0 conv2)
    (1, 14, 1024, 256, 1, 1, 16),                    # 2, 2: slices shorter than the ring
    (1, 7, 2048, 512, 1, 1, 16),                     # 4, 4: slices exactly the ring
    (1, 28, 128, 128, 3, 1, 8),                      # 5, 1: ragged, last slice of ONE k-block
    (1, 56, 64, 64, 3, 1, 4),                        # 5, 3: ragged, partial 128-row tiles (2 rows of 56)
    (1, 56, 64, 64, 1, 1, 2),                        # 1, 1: one k-block per slice, ring depth 1
    (2, 7, 512, 512, 3, 1, 8), (2, 28, 256, 256, 3, 2, 8), (2, 14, 1024, 256, 1, 1, 4), (1, 56, 256, 512, 1, 2, 2),
    (9, 7, 512, 512, 3, 1, 1), (9, 7, 512, 512, 3, 1, 2)]


def _fwd_once(L, case, x, w, part_in, gamma, beta):
    B, Hi, Cin, Cout, k, s, nz = case
    force(L, 0, nz)
    # a strided 1x1 convolution does not visit every operand pixel: it cannot materialise the operand
    p = FwdProb(L, B, Hi, Cin, Cout, k, s, 1, x, wmat(w), part_in, gamma, beta, want_a=not (k == 1 and s == 2))
    fwd_launch(L, [p])
    check_plan(L, 0, case, nz, k * k * Cin // 32, fwd_tiles(B, Hi // s, Cout))
    check_guards(p.out, case)
    return p


@pytest.mark.parametrize('case', FWD, ids=lambda c: 'B{}_H{}_{}x{}_k{}s{}_nz{}'.format(*c))
def test_forward_plan(L, case):
    B, Hi, Cin, Cout, k, s, nz = case
    g = torch.Generator().manual_seed(sum(case) + 5)
    x = (torch.randn(B, Hi, Hi, Cin, generator=g) * 1.5 + 0.4).cuda()
    w = (torch.randn(Cout, Cin, k, k, generator=g) / (k * k * Cin) ** 0.5).cuda()
    gamma, beta = (1 + 0.3 * torch.randn(Cin, generator=g)).cuda(), (0.2 * torch.randn(Cin, generator=g)).cuda()
    part_in = fixed_sums(x, B)
    p = _fwd_once(L, case, x, w, part_in, gamma, beta)
    a_ref, st = gn(x, B, gamma, beta)
    a_ref = a_ref.clamp_min(0)
    a = a_ref
    if p.out['a_out'] is not None:
        a = p.out['a_out'].t
        assert torch.isfinite(a).all() and rel_err(a, a_ref) < 1e-5, case
        so = p.out['stats_out'].t
        assert (so[..., 0].double().cpu() - st[..., 0].cpu()).abs().max() < 1e-5 * st[..., 1].cpu().reciprocal().max() + 1e-6, case
        assert rel_err(so[..., 1], st[..., 1]) < 2e-5, case
    check_conv(p.out['y'].t, p.out['part_out'].t, a, w, s, k // 2, B, case)
    check_same(p.out, _fwd_once(L, case, x, w, part_in, gamma, beta).out, case)


FWD2 = [  # B, H, C, planes, stride of the shortcut convolution, mode, nz: conv1 + shortcut convolution of a bottleneck in one launch
    (1, 28, 512, 128, 1, 2, 1), (1, 28, 512, 128, 1, 2, 2), (1, 14, 1024, 256, 2, 2, 4), (1, 14, 1024, 256, 2, 3, 4),
    (2, 14, 1024, 256, 2, 3, 2), (9, 7, 2048, 512, 1, 3, 1)]


@pytest.mark.parametrize('case', FWD2, ids=lambda c: 'B{}_H{}_C{}_p{}_s{}_mode{}_nz{}'.format(*c))
def test_forward_two_problem_plan(L, case):
    """conv1 and the shortcut convolution share one launch and one operand, formed on load from the previous block's raw output
    and either a materialised shortcut (mode 2) or the raw shortcut convolution output and its GroupNorm (mode 3)"""
    B, H, Cc, planes, s, mode, nz = case
    g = torch.Generator().manual_seed(sum(case) + 9)
    rn = lambda *sh: torch.randn(*sh, generator=g).cuda()
    x = rn(B, H, H, Cc) + 0.3
    ga, be, ga2, be2 = 1 + 0.3 * rn(Cc), 0.2 * rn(Cc), 1 + 0.3 * rn(Cc), 0.2 * rn(Cc)
    part_in = fixed_sums(x, B)
    if mode == 2:
        res = rn(B, H, H, Cc).abs()
        extra = dict(res=res)
        block_out = (gn(x, B, ga, be)[0] + res.double()).clamp_min(0)
    else:
        res = rn(B, H, H, Cc) * 2 - 0.5
        extra = dict(res=res, part2_in=fixed_sums(res, B), gamma2=ga2, beta2=be2)
        block_out = (gn(x, B, ga, be)[0] + gn(res, B, ga2, be2)[0]).clamp_min(0)
    w1 = rn(planes, Cc, 1, 1) / Cc ** 0.5
    wd = rn(4 * planes, Cc, 1, 1) / Cc ** 0.5

    def once():
        force(L, 0, nz)
        c1 = FwdProb(L, B, H, Cc, planes, 1, 1, mode, x, wmat(w1), part_in, ga, be, **extra)
        ds = FwdProb(L, B, H, Cc, 4 * planes, 1, s, mode, x, wmat(wd), part_in, ga, be, want_a=False, **extra)
        fwd_launch(L, [c1, ds])
        check_plan(L, 0, case, nz, Cc // 32, fwd_tiles(B, H, planes) + fwd_tiles(B, H // s, 4 * planes))
        check_guards(c1.out, (case, 'conv1'))
        check_guards(ds.out, (case, 'shortcut'))
        return c1, ds

    c1, ds = once()
    a = c1.out['a_out'].t
    assert torch.isfinite(a).all() and rel_err(a, block_out) < 1e-5, case
    check_conv(c1.out['y'].t, c1.out['part_out'].t, a, w1, 1, 0, B, (case, 'conv1'))
    check_conv(ds.out['y'].t, ds.out['part_out'].t, a, wd, s, 0, B, (case, 'shortcut'))
    if mode == 3:
        assert rel_err(c1.out['stats2_out'].t[..., 1], gn(res, B, ga2, be2)[1][..., 1]) < 2e-5, case
    c1b, dsb = once()
    check_same(c1.out, c1b.out, (case, 'conv1'))
    check_same(ds.out, dsb.out, (case, 'shortcut'))


# ---------------------------------------------------------------------------------------------------------------------------
# data gradient
# ---------------------------------------------------------------------------------------------------------------------------
DGRAD = [  # B, H, Cin, Cout, k, nprep, addend, nz
    (1, 7, 512, 512, 3, 1, False, 1), (1, 7, 512, 512, 3, 1, False, 2), (1, 7, 512, 512, 3, 1, True, 4), (1, 7, 512, 512, 3, 0, False, 8),
    (1, 7, 512, 512, 3, 1, False, 16),                # 9, 9: 16-CTA cluster
    (1, 14, 256, 1024, 1, 0, True, 16),               # 2, 2: slices shorter than the ring
    (1, 28, 128, 128, 3, 1, False, 8),                # 5, 1: ragged, last slice of ONE k-block, partial tiles
    (1, 56, 64, 64, 3, 2, True, 4),                   # 5, 3: ragged
    (1, 56, 64, 64, 1, 1, False, 2),                  # 1, 1: one k-block per slice
    (1, 14, 1024, 256, 1, 2, True, 4), (2, 7, 2048, 512, 1, 1, True, 2), (2, 28, 128, 128, 3, 2, False, 4),
    (2, 14, 256, 1024, 1, 1, False, 8), (9, 7, 512, 512, 3, 1, False, 1), (9, 7, 512, 512, 3, 2, True, 2)]


def dgrad_reference(B, H, Cin, Cout, k, g, with_add, nprep):
    rn = lambda *s: torch.randn(*s, generator=g).cuda()
    dz, y_c = rn(B, H, H, Cout) * 0.1, rn(B, H, H, Cout) + 0.2
    gamma_c = 1 + 0.3 * rn(Cout)
    w = rn(Cout, Cin, k, k) / (k * k * Cin) ** 0.5
    _, st_c = gn(y_c, B, torch.ones(Cout, device='cuda'), torch.zeros(Cout, device='cuda'))
    ex = lambda v, Cc: v.repeat_interleave(Cc // 4, dim=1)[:, None, None, :]
    xh_c = (y_c.double() - ex(st_c[..., 0], Cout)) * ex(st_c[..., 1], Cout)
    q_c = dz.double() * gamma_c.double()
    sums_c = torch.stack([group_view(q_c, B).sum(-1), (group_view(q_c, B) * group_view(xh_c, B)).sum(-1)], -1)
    N = H * H * Cout // 4
    dy = ex(st_c[..., 1], Cout) * (q_c - ex(sums_c[..., 0] / N, Cout) - xh_c * ex(sums_c[..., 1] / N, Cout))
    dX = torch.nn.grad.conv2d_input((B, Cin, H, H), w.double(), dy.permute(0, 3, 1, 2), padding=k // 2).permute(0, 2, 3, 1)
    addend = rn(B, H, H, Cin) * 0.05 if with_add else None
    if addend is not None:
        dX = dX + addend.double()
    ins = dict(dz=dz, y_c=y_c, w=wmat(w), stats_c=st_c.float().contiguous(), sums_c=(sums_c * FIX_BWD).round().long().contiguous(),
               gamma_c=gamma_c, addend=addend)
    preps = []
    if nprep > 0:
        ins['mask'] = rn(B, H, H, Cin)
        for _ in range(nprep):
            y_p, gamma_p = rn(B, H, H, Cin) - 0.1, 1 + 0.3 * rn(Cin)
            preps.append((y_p, gamma_p, gn(y_p, B, torch.ones(Cin, device='cuda'), torch.zeros(Cin, device='cuda'))[1].float().contiguous()))
    return ins, preps, dy, dX, ex


def dgrad_launch(L, case, ins, preps, accumulate=0, base=None):
    B, H, Cin, Cout, k = case[:5]
    nz = case[-1]
    force(L, 1, nz)
    f = L.DgradFusedStruct()
    outs = {'dy_out': Guarded((B, H, H, Cout)), 'out': Guarded((B, H, H, Cin), init=base)}
    for name, t in ins.items():
        setattr(f, name, None if t is None else t.data_ptr())
    for name in ('dy_out', 'out'):
        setattr(f, name, outs[name].ptr())
    for j, (y_p, gamma_p, st_p) in enumerate(preps):
        outs[f'prep_sums{j}'] = Guarded((B, 4, 2), torch.int64, 0)
        outs[f'prep_dgb{j}'] = Guarded((Cin, 2), torch.int64, 0)
        f.prep_y[j], f.prep_stats[j], f.prep_gamma[j] = y_p.data_ptr(), st_p.data_ptr(), gamma_p.data_ptr()
        f.prep_sums[j], f.prep_dgb[j] = outs[f'prep_sums{j}'].ptr(), outs[f'prep_dgb{j}'].ptr()
    f.nprep, f.accumulate = len(preps), accumulate
    L.call('dboa_dgrad_fused', C.byref(f), B, H, Cin, Cout, k, L.stream())
    torch.cuda.synchronize()
    bh = rows_of(H)
    check_plan(L, 1, case, nz, k * k * Cout // 32, B * -(-H // bh) * (Cin // 64))
    check_guards(outs, case)
    return outs


@pytest.mark.parametrize('case', DGRAD, ids=lambda c: 'B{}_H{}_{}x{}_k{}_prep{}_add{}_nz{}'.format(*c[:5], c[5], int(c[6]), c[7]))
def test_dgrad_plan(L, case):
    B, H, Cin, Cout, k, nprep, with_add, nz = case
    g = torch.Generator().manual_seed(sum(case[:5]) + 23)
    ins, preps, dy, dX, ex = dgrad_reference(B, H, Cin, Cout, k, g, with_add, nprep)
    outs = dgrad_launch(L, case, ins, preps)
    assert rel_err(outs['dy_out'].t, dy) < 2e-5, case
    if nprep == 0:
        assert rel_err(outs['out'].t, dX) < 3e-5, case
    else:
        dz_p = dX * (ins['mask'] > 0)
        assert rel_err(outs['out'].t, dz_p) < 3e-5, case
        for j, (y_p, gamma_p, st_p) in enumerate(preps):
            xh = (y_p.double() - ex(st_p[..., 0].double(), Cin)) * ex(st_p[..., 1].double(), Cin)
            q = dz_p * gamma_p.double()
            ref_sums = torch.stack([group_view(q, B).sum(-1), (group_view(q, B) * group_view(xh, B)).sum(-1)], -1)
            got = outs[f'prep_sums{j}'].t.double() / FIX_BWD
            assert (got - ref_sums).abs().max() <= 3e-5 * ref_sums.abs().max() + 1e-6, (case, j)
            ref_dg, ref_db = (dz_p * xh).sum((0, 1, 2)), dz_p.sum((0, 1, 2))
            got_g = outs[f'prep_dgb{j}'].t.double() / FIX_BWD
            assert (got_g[:, 0] - ref_dg).abs().max() <= 3e-5 * ref_dg.abs().max() + 1e-6, (case, j)
            assert (got_g[:, 1] - ref_db).abs().max() <= 3e-5 * ref_db.abs().max() + 1e-6, (case, j)
    check_same(outs, dgrad_launch(L, case, ins, preps), case)


@pytest.mark.parametrize('case', [(1, 7, 512, 512, 3, 0, True, 8), (1, 28, 128, 128, 3, 0, False, 8), (2, 14, 256, 1024, 1, 0, True, 2)],
                         ids=lambda c: 'B{}_H{}_{}x{}_k{}_add{}_nz{}'.format(*c[:5], int(c[6]), c[7]))
def test_dgrad_accumulate_plan(L, case):
    """accumulate = 1 without a mask: out += dX (+ addend) over a random base"""
    B, H, Cin, Cout, k, nprep, with_add, nz = case
    g = torch.Generator().manual_seed(sum(case[:5]) + 29)
    ins, preps, dy, dX, _ = dgrad_reference(B, H, Cin, Cout, k, g, with_add, 0)
    base = torch.randn(B, H, H, Cin, generator=g).cuda() * dX.abs().max().float()
    outs = dgrad_launch(L, case, ins, preps, accumulate=1, base=base)
    assert rel_err(outs['dy_out'].t, dy) < 2e-5, case
    assert rel_err(outs['out'].t - base, dX) < 3e-5, case
    check_same(outs, dgrad_launch(L, case, ins, preps, accumulate=1, base=base), case)


# ---------------------------------------------------------------------------------------------------------------------------
# weight gradient
# ---------------------------------------------------------------------------------------------------------------------------
WGRAD = [  # B, H (input), Cin, Cout, k, stride, nz
    (2, 56, 64, 256, 1, 1, 1), (2, 56, 64, 256, 1, 1, 4), (2, 56, 64, 256, 1, 1, 16),     # width 56; 7, 7 at nz = 16
    (1, 56, 64, 256, 1, 1, 8),                                                              # 7, 7
    (1, 28, 512, 128, 1, 1, 4),                                                             # width 28, ragged 4, 2
    (1, 56, 256, 512, 1, 2, 4), (1, 56, 128, 128, 3, 2, 4),                                 # stride 2 into width 28, ragged
    (2, 28, 512, 128, 1, 1, 2),
    (1, 14, 1024, 256, 1, 1, 4),                                                            # width 14: 1, 1 (one box per slice)
    (9, 14, 256, 256, 1, 1, 8),                                                             # 5, 1: ragged
    (9, 7, 512, 128, 1, 1, 2),                                                              # width 7, 8-row padded box, ragged 5, 4
    (9, 7, 2048, 512, 1, 1, 1), (1, 14, 512, 512, 3, 2, 1)]


@pytest.mark.parametrize('case', WGRAD, ids=lambda c: 'B{}_H{}_{}x{}_k{}s{}_nz{}'.format(*c))
def test_wgrad_plan(L, case):
    B, H, Cin, Cout, k, s, nz = case
    g = torch.Generator().manual_seed(sum(case) + 3)
    Ho = H // s
    x = torch.randn(B, H, H, Cin, generator=g).cuda()
    dy = torch.randn(B, Ho, Ho, Cout, generator=g).cuda()
    K = k * k * Cin
    base = (torch.randn(Cout, K, generator=g) * 0.1).cuda()

    def once():
        force(L, 2, nz)
        dw = Guarded((Cout, K), init=base)
        L.call('dboa_conv2d_wgrad_tma', L.ptr(dy), L.ptr(x), dw.ptr(), B, H, H, Cin, Cout, k, s, k // 2, K, L.stream())
        torch.cuda.synchronize()
        bh = 8 if Ho == 7 else 56 // Ho
        check_plan(L, 2, case, nz, B * -(-Ho // bh), Cout // 128 * Cin // 64 * k * k)
        check_guards({'dw': dw}, case)
        return {'dw': dw}

    out = once()
    ref = torch.nn.grad.conv2d_weight(nhwc(x).double(), (Cout, Cin, k, k), nhwc(dy).double(), stride=s, padding=k // 2)
    ref = ref.permute(0, 2, 3, 1).reshape(Cout, K)
    assert rel_err(out['dw'].t - base, ref) < 2e-5, case
    check_same(out, once(), case)


def test_plan_coverage():
    """the plan matrix above reached every cluster size it aims at, ragged last slices, slices shorter than the operand ring and
    slices of one k-block, for each kernel"""
    want = {0: {nz for *_, nz in FWD} | {nz for *_, nz in FWD2}, 1: {c[-1] for c in DGRAD}, 2: {nz for *_, nz in WGRAD}}
    ran = {k: {p['nz'] for kk, _, p in PLANS if kk == k} for k in range(3)}
    if any(not want[k] <= ran[k] for k in range(3)):
        pytest.skip('the plan matrix did not run in full')
    lines = ['kernel   nz reached              ragged (per, last)        per < ring   per = 1']
    for k in range(3):
        ps = [p for kk, _, p in PLANS if kk == k]
        ragged = sorted({(p['nz'], p['per'], p['last']) for p in ps if p['last'] != p['per']})
        short = sorted({p['nz'] for p in ps if p['per'] < DMAX[k]})
        one = sorted({p['nz'] for p in ps if p['per'] == 1})
        lines.append(f'{NAMES[k]:8} {str(sorted(ran[k])):23} {str(ragged):25} {str(short):12} {one}')
        assert ragged and short and one, NAMES[k]
        assert any(p['last'] < DMAX[k] for p in ps if p['last'] != p['per']), NAMES[k]        # a ragged slice shorter than the ring
    print('\n' + '\n'.join(lines))
    assert {1, 2, 4, 8, 16} <= ran[0] and {1, 2, 4, 8, 16} <= ran[1] and {1, 2, 4, 8, 16} <= ran[2]


# ---------------------------------------------------------------------------------------------------------------------------
# whole network under the extreme plans
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope='module')
def model():
    from dynaboa_b200 import synthetic
    from dynaboa_b200.hmr import hmr
    from oracle import hmr_ref
    m = hmr(synthetic.make_mean_params()).cuda()
    sd = hmr_ref.strip_prefix(synthetic.make_basemodel()['model'])
    m.load_state_dict(sd, strict=True)
    m.eval()
    return m, sd


def set_extreme(L, which):
    for k in range(3):
        if which == 'widest':
            L.call('dboa_set_split_limits', k, 0 if k == 0 else n_sms(), 16, 1)
        else:
            L.call('dboa_set_split_limits', k, -1, 1, -1)


@pytest.mark.parametrize('which', ['widest', 'narrowest'])
def test_network_forward_under_extreme_plans(L, model, which):
    from oracle import hmr_ref
    m, sd = model
    for B in (1, 9):
        x = torch.randn(B, 3, 224, 224, generator=torch.Generator().manual_seed(60 + B))
        with torch.no_grad():
            ref = hmr_ref.forward(x, sd)
        set_extreme(L, which)
        try:
            with torch.no_grad():
                got = m(x.cuda())
            torch.cuda.synchronize()
            if which == 'narrowest':
                assert last_plan(L, 0)['nz'] == 1
        finally:
            for k in range(3):
                L.call('dboa_set_split_limits', k, -1, -1, -1)
        for a, b, name in zip(got, ref, ('rotmat', 'shape', 'cam')):
            assert rel_err(a, b) < 1e-4, (which, B, name)


_ORACLE = {}


def oracle_gradient(sd, B):
    """input, loss weights, outputs and parameter gradients of the CPU oracle (torch autograd), once per batch size"""
    if B not in _ORACLE:
        from oracle import hmr_ref
        g = torch.Generator().manual_seed(90 + B)
        x = torch.randn(B, 3, 224, 224, generator=g)
        ws = torch.randn(B, 24, 3, 3, generator=g), torch.randn(B, 10, generator=g), torch.randn(B, 3, generator=g)
        pc = {k: v.clone().requires_grad_(True) for k, v in sd.items() if not k.startswith('init_')}
        full = dict(pc)
        full.update({k: sd[k] for k in ('init_pose', 'init_shape', 'init_cam')})
        outs = hmr_ref.forward(x, full)
        sum((o * w).sum() for o, w in zip(outs, ws)).backward()
        _ORACLE[B] = (x, ws, [o.detach() for o in outs], {k: v.grad for k, v in pc.items()})
    return _ORACLE[B]


@pytest.mark.parametrize('B', [1, 2])
@pytest.mark.parametrize('which', ['widest', 'narrowest'])
def test_network_gradient_under_extreme_plans(L, model, which, B):
    """all 169 gradient tensors against CPU autograd of the oracle, with the bounds of
    test_gpu_hmr.py::test_full_gradient_matches_oracle_autograd (the gradient is piecewise constant in places: L2 bounds)"""
    m, sd = model
    x, (w_r, w_s, w_c), (r, s_, c), grads = oracle_gradient(sd, B)
    set_extreme(L, which)
    try:
        for p in m.parameters():
            p.grad = None
        object.__setattr__(m, '_grad_arena', None)
        rot, shape, cam = m(x.cuda())
        ((rot * w_r.cuda()).sum() + (shape * w_s.cuda()).sum() + (cam * w_c.cuda()).sum()).backward()
        torch.cuda.synchronize()
        if which == 'narrowest':
            assert all(last_plan(L, k)['nz'] == 1 for k in range(3))
    finally:
        for k in range(3):
            L.call('dboa_set_split_limits', k, -1, -1, -1)
    for a, b, name in zip((rot, shape, cam), (r, s_, c), ('rotmat', 'shape', 'cam')):
        assert rel_err(a.detach(), b) < 1e-4, (which, B, name)
    worst, num, den = [], 0.0, 0.0
    for name, p in m.named_parameters():
        ref = grads[name].double()
        d = p.grad.contiguous().double().cpu() - ref
        worst.append(((d.norm() / ref.norm()).item(), name))
        num, den = num + float(d.pow(2).sum()), den + float(ref.pow(2).sum())
    worst.sort(reverse=True)
    total = (num / den) ** 0.5
    print(f'{which} B={B}: whole-gradient rel L2 {total:.2e}; worst tensors', worst[:3])
    assert total < 2e-3, (which, B, total)
    assert worst[0][0] < 1e-2, (which, B, worst[:4])
