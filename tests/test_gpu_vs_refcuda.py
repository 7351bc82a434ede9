"""Oracle #2: this repository's CUDA ops against the REFERENCE'S OWN CUDA ops (its three plugins built unmodified for
sm_100a, driven by its own Python wrappers bias_act.py:126-207, upfirdn2d.py:217-273, filtered_lrelu.py:159-272) on
identical seeded inputs, on the call signatures the networks make (SURVEY Appendix A; real spatial sizes, batch
reduced). This is the comparison the north_star states its tolerances for: 1e-3 relative fp32 activations, 1e-2
gradients -- checked ELEMENT-WISE (|a-b| <= rtol*|b| + rtol*FLOOR*max|b|), forward, dx and db, fp32 and fp16.

The reference side is stored in tests/golden/refcuda_*.npz (made on a B200 by oracle/pin_refcuda.py from the reference's
plugins): for every output tensor its shape, max|ref|, L2 norm and the values at NSAMP fixed positions spread over the
whole tensor. The element-wise bound is checked at those positions, against the full tensor's max|ref|; the max and the
norm of the whole tensor are checked against the bounds the element-wise rule implies."""
import math
import types

import numpy as np
import pytest
import scipy.signal
import torch

from _common import golden
from torch_utils.ops import bias_act, upfirdn2d, filtered_lrelu, conv2d_resample, conv2d_gradfix

pytestmark = pytest.mark.gpu
DEV = 'cuda'
FLOOR = 1e-2      # elements below 1 % of max|ref| are held to an absolute bound of rtol * 1 % * max|ref|
NSAMP = 256       # stored reference values per tensor


def sample_index(numel):
    """NSAMP distinct flat indices spread over [0, numel) (a Weyl sequence; 2654435761 is prime and larger than numel)."""
    if numel <= NSAMP:
        return torch.arange(numel)
    return (torch.arange(NSAMP, dtype=torch.int64) * 2654435761) % numel


def summarize(t):
    """-> {'v': sampled values (in t's dtype), 'shape', 'stats': [max|t|, ||t||]}: what the golden file keeps of a tensor."""
    t = t.detach()
    flat = t.reshape(-1)
    d = flat.double()
    return {'v': flat[sample_index(flat.numel()).to(flat.device)].cpu().numpy(), 'shape': np.array(t.shape, np.int64),
            'stats': np.array([float(d.abs().max()), float(d.norm())], np.float64)}


class Ref:
    """One stored reference tensor: golden key prefix `key` of file `op`."""

    def __init__(self, op, key):
        g = golden('refcuda_' + op)
        self.key = key
        self.v = torch.from_numpy(g[key + '/v'])
        self.shape = tuple(int(s) for s in g[key + '/shape'])
        self.scale, self.norm = (float(s) for s in g[key + '/stats'])

    def got(self, t, what):
        """Our tensor's values at the stored positions (float64), after the shape / dtype / finiteness checks."""
        assert tuple(t.shape) == self.shape and str(t.dtype).endswith(str(self.v.dtype)), (what, t.shape, self.shape, t.dtype, self.v.dtype)
        assert torch.isfinite(t).all(), what
        flat = t.detach().reshape(-1)
        return flat[sample_index(flat.numel()).to(flat.device)].double().cpu()


def elementwise(got, ref, rtol, what):
    g, w = ref.got(got, what), ref.v.double()
    # fp16 storage: intermediates are rounded at different points on the two sides (e.g. the reference rounds between its two
    # separable passes, upfirdn2d.py:244-245), an absolute error of a few 1e-4 of the tensor's scale that does not shrink
    # with the element -> a 10 % floor there
    floor = FLOOR if got.dtype != torch.float16 else 10 * FLOOR
    scale = ref.scale
    bound = rtol * w.abs() + rtol * floor * scale
    bad = (g - w).abs() > bound
    if bad.any():
        i = int(((g - w).abs() / bound).argmax())
        raise AssertionError(f'{what}: {int(bad.sum())} of {g.numel()} sampled elements outside rtol {rtol:g}; worst got {g[i]:.7g} '
                             f'want {w[i]:.7g} (max|ref| {scale:.4g})')
    # the whole tensor: the element-wise rule bounds the difference of the maxima and of the norms
    full = got.detach().double()
    gmax, gnorm = float(full.abs().max()), float(full.norm())
    assert abs(gmax - scale) <= rtol * (1 + floor) * scale, f'{what}: max|got| {gmax:.7g}, max|ref| {scale:.7g}'
    assert abs(gnorm - ref.norm) <= rtol * ref.norm + rtol * floor * scale * math.sqrt(full.numel()), \
        f'{what}: ||got|| {gnorm:.7g}, ||ref|| {ref.norm:.7g}'


def tols(dtype):
    # fp16 storage: both sides round their result to fp16 once -> up to 1 fp16 ulp (9.8e-4) apart element-wise
    return (1e-3, 1e-2) if dtype == torch.float32 else (4e-3, 1e-2)


def rnd(shape, seed, dtype=torch.float32, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(*shape, generator=g) * scale).to(dtype).to(DEV)


OURS = types.SimpleNamespace(bias_act=bias_act, upfirdn2d=upfirdn2d, filtered_lrelu=filtered_lrelu, conv2d_resample=conv2d_resample,
                             conv2d_gradfix=conv2d_gradfix)


# ------------------------------------------------------------------ bias_act (a1)

BIAS_ACT = [
    # lres G (N,C,T,H,W) lrelu clamp 256 (generator_lres.py:581-589)
    ((2, 512, 20, 3, 4), 1, 'lrelu', None, 256, torch.float32),
    ((2, 512, 32, 5, 8), 1, 'lrelu', None, 256, torch.float32),
    ((1, 256, 144, 9, 16), 1, 'lrelu', None, 256, torch.float32),
    ((1, 64, 160, 36, 64), 1, 'lrelu', None, 256, torch.float32),
    ((1, 3, 128, 36, 64), 1, 'linear', None, 256, torch.float32),           # ToRGB
    # lres D
    ((1, 32, 128, 64, 64), 1, 'lrelu', None, 256, torch.float32),
    ((2, 512, 16, 4, 4), 1, 'lrelu', None, 256, torch.float32),
    ((2, 64, 128, 32, 32), 1, 'linear', None, 256, torch.float32),          # skip branch
    # sres D (N,C,H,W) fp16 / fp32, gain sqrt2 (discriminator_sres.py:192-204)
    ((2, 64, 256, 256), 1, 'lrelu', math.sqrt(2), 256, torch.float16),
    ((2, 512, 32, 32), 1, 'lrelu', math.sqrt(2), 256, torch.float16),
    ((2, 512, 4, 4), 1, 'lrelu', math.sqrt(2), 256, torch.float32),
    # FC layers
    ((640, 1024), 1, 'lrelu', None, None, torch.float32),
    ((16, 512), 1, 'lrelu', None, None, torch.float32),
    # clamp-active and second-order activations
    ((2, 16, 8, 9, 16), 1, 'lrelu', None, 0.5, torch.float32),
    ((2, 16, 33, 17), 1, 'swish', None, 1.0, torch.float32),
    ((2, 16, 33, 17), 1, 'tanh', 2.0, None, torch.float16),
]


def run_bias_act(ops, shape, dim, act, gain, clamp, dtype):
    x, b, dy = rnd(shape, 1, dtype), rnd((shape[dim],), 2, dtype), rnd(shape, 3, dtype)
    xg, bg = x.clone().requires_grad_(True), b.clone().requires_grad_(True)
    y = ops.bias_act.bias_act(xg, bg, dim=dim, act=act, gain=gain, clamp=clamp)
    dx, db = torch.autograd.grad(y, [xg, bg], dy)
    return {'y': y.detach(), 'dx': dx, 'db': db}


@pytest.mark.parametrize('shape,dim,act,gain,clamp,dtype', BIAS_ACT)
def test_bias_act_vs_reference_cuda(shape, dim, act, gain, clamp, dtype):
    ra, rg = tols(dtype)
    case = BIAS_ACT.index((shape, dim, act, gain, clamp, dtype))
    got = run_bias_act(OURS, shape, dim, act, gain, clamp, dtype)
    elementwise(got['y'], Ref('bias_act', f'{case}/y'), ra, 'y')
    elementwise(got['dx'], Ref('bias_act', f'{case}/dx'), rg, 'dx')
    # db: the reference reduces dx with torch.sum (bias_act.py:186), ours inside the kernel; same dx => compare to fp32 sum accuracy
    elementwise(got['db'], Ref('bias_act', f'{case}/db'), rg, 'db')


def run_bias_act_r1(ops):
    # R1 penalty: grad of |dL/dx|^2 through bias_act (video_gan_lres.py:178-199)
    shape = (2, 32, 16, 16, 16)
    x, b, v = rnd(shape, 4), rnd((32,), 5), rnd(shape, 6)
    xg, bg = x.clone().requires_grad_(True), b.clone().requires_grad_(True)
    w1 = torch.full((1, 32, 1, 1, 1), 0.7, device=DEV).requires_grad_(True)      # stand-ins for the conv weights between
    w2 = torch.full((1, 32, 1, 1, 1), 1.3, device=DEV).requires_grad_(True)      # two activation layers
    h = ops.bias_act.bias_act(xg * w1, bg, act='lrelu', clamp=256)
    y = ops.bias_act.bias_act(h * w2, bg, act='lrelu', clamp=256)
    gx, = torch.autograd.grad((y * v).sum(), [xg], create_graph=True)            # d logits / d input, kept in the graph
    pen = gx.square().sum()
    g1, g2 = torch.autograd.grad(pen, [w1, w2])                                  # second order: through both backward ops
    return {'gx': gx.detach(), 'g1': g1, 'g2': g2}


def test_bias_act_r1_double_backward_vs_reference_cuda():
    got = run_bias_act_r1(OURS)
    elementwise(got['gx'], Ref('bias_act', 'r1/gx'), 1e-2, 'first-order grad')
    elementwise(got['g1'], Ref('bias_act', 'r1/g1'), 1e-2, 'd penalty / d w1')
    elementwise(got['g2'], Ref('bias_act', 'r1/g2'), 1e-2, 'd penalty / d w2')


# ------------------------------------------------------------------ upfirdn2d (a2, a7)

def kaiser(taps, scale):
    return torch.tensor(scipy.signal.firwin(numtaps=taps, cutoff=0.5, width=0.6, fs=2.0 * scale), dtype=torch.float32)


F4 = [1., 3., 3., 1.]
UPFIRDN = [
    # name, x shape, filter, kwargs, dtype
    ('U1 temporal kaiser down', (2, 1024, 640, 1), lambda: kaiser(12, 2)[:, None], dict(down=[1, 2], padding=[0, 0, 5, 5]), torch.float32),
    ('U1 small', (2, 1024, 40, 1), lambda: kaiser(12, 2)[:, None], dict(down=[1, 2], padding=[0, 0, 5, 5]), torch.float32),
    ('U2 temporal linear up', (1, 256, 80, 144), lambda: (torch.tensor(F4) / 8)[:, None], dict(up=[1, 2], padding=[0, 0, 2, 1], gain=2), torch.float32),
    ('U2 small', (2, 512, 20, 12), lambda: (torch.tensor(F4) / 8)[:, None], dict(up=[1, 2], padding=[0, 0, 2, 1], gain=2), torch.float32),
    ('U3 bilinear up', (1, 8192, 18, 32), lambda: upfirdn2d.setup_filter(F4, separable=True), dict(up=2, padding=[2, 1, 2, 1], gain=4), torch.float32),
    ('U3 tiny', (2, 16384, 3, 4), lambda: upfirdn2d.setup_filter(F4, separable=True), dict(up=2, padding=[2, 1, 2, 1], gain=4), torch.float32),
    ('U4 D spatial down', (1, 8192, 64, 64), lambda: upfirdn2d.setup_filter(F4, separable=True), dict(down=2, padding=[1, 1, 1, 1]), torch.float32),
    ('U4 small', (2, 16384, 8, 8), lambda: upfirdn2d.setup_filter(F4, separable=True), dict(down=2, padding=[1, 1, 1, 1]), torch.float32),
    ('U5 D temporal down', (1, 128, 128, 256), lambda: (torch.tensor(F4) / 8)[:, None], dict(down=[1, 2], padding=[0, 0, 1, 1]), torch.float32),
    ('U6 cond kaiser down4', (8, 27, 92, 92), lambda: kaiser(24, 4), dict(down=4, padding=6), torch.float32),
    ('U6 cond kaiser down2', (8, 27, 88, 88), lambda: kaiser(12, 2), dict(down=2, padding=3), torch.float32),
    ('U6 cond kaiser up2', (8, 27, 86, 86), lambda: kaiser(12, 2), dict(up=2, padding=[4, 3, 4, 3], gain=4), torch.float32),
    ('U6 cond kaiser up4', (8, 27, 86, 86), lambda: kaiser(24, 4), dict(up=4, padding=[9, 6, 9, 6], gain=16), torch.float32),
    ('U7 D lr upsample', (2, 12, 36, 64), lambda: kaiser(8, 2), dict(up=4, padding=[5, 2, 5, 2], gain=16), torch.float32),
    ('U8 2-D filter pad', (2, 64, 128, 128), lambda: upfirdn2d.setup_filter(F4, separable=False), dict(padding=2), torch.float16),
    ('U8 2-D filter down2', (2, 64, 128, 128), lambda: upfirdn2d.setup_filter(F4, separable=False), dict(down=2, padding=1), torch.float16),
    ('U8 2-D filter down2 fp32', (2, 512, 16, 16), lambda: upfirdn2d.setup_filter(F4, separable=False), dict(down=2, padding=1), torch.float32),
    ('U9 ADA sym6 up', (4, 3, 144, 256), lambda: kaiser(12, 2), dict(up=2, padding=-6, flip_filter=True, gain=4), torch.float32),
    ('U9 ADA sym6 down', (4, 3, 300, 500), lambda: kaiser(12, 2), dict(down=2, padding=-6, flip_filter=True), torch.float32),
    ('U3 fp16', (2, 512, 18, 32), lambda: upfirdn2d.setup_filter(F4, separable=True), dict(up=2, padding=[2, 1, 2, 1], gain=4), torch.float16),
]


def run_upfirdn2d(ops, shape, mkf, kw, dtype):
    f = mkf().to(DEV)
    x = rnd(shape, 7, dtype)
    xg = x.clone().requires_grad_(True)
    y = ops.upfirdn2d.upfirdn2d(xg, f, **kw)
    dy = rnd(tuple(y.shape), 8, dtype)
    dx, = torch.autograd.grad(y, [xg], dy)
    return {'y': y.detach(), 'dx': dx}


@pytest.mark.parametrize('name,shape,mkf,kw,dtype', UPFIRDN, ids=[u[0] for u in UPFIRDN])
def test_upfirdn2d_vs_reference_cuda(name, shape, mkf, kw, dtype):
    ra, rg = tols(dtype)
    got = run_upfirdn2d(OURS, shape, mkf, kw, dtype)
    elementwise(got['y'], Ref('upfirdn2d', f'{name}/y'), ra, f'{name} y')
    elementwise(got['dx'], Ref('upfirdn2d', f'{name}/dx'), rg, f'{name} dx')


# ------------------------------------------------------------------ filtered_lrelu (a3)

FL = [
    # (C, H, W), up, down, padding, dtype -- sres G layer table (SURVEY Appendix A); taps = 6*factor
    ('L0-2 29x36 up2 down2 fp32', (512, 31, 38), 2, 2, [9, 8, 9, 8], torch.float32),
    ('L3 up4 down2', (512, 31, 38), 4, 2, [-6, -9, -6, -9], torch.float16),
    ('L4 up2 down2', (512, 40, 54), 2, 2, [9, 8, 9, 8], torch.float16),
    ('L5 up4 down2', (512, 40, 54), 4, 2, [-6, -9, -6, -9], torch.float16),
    ('L6', (512, 58, 86), 2, 2, [9, 8, 9, 8], torch.float16),
    ('L7', (256, 58, 86), 4, 2, [-6, -9, -6, -9], torch.float16),
    ('L8', (256, 94, 150), 2, 2, [9, 8, 9, 8], torch.float16),
    ('L9', (181, 94, 150), 2, 2, [9, 8, 9, 8], torch.float16),
    ('L10 up4', (64, 94, 150), 4, 2, [-6, -9, -6, -9], torch.float16),
    ('L11', (45, 166, 278), 2, 2, [9, 8, 9, 8], torch.float16),
    ('L13 crop', (32, 166, 278), 2, 2, [-11, -12, -11, -12], torch.float16),
    ('L4 fp32', (64, 40, 54), 2, 2, [9, 8, 9, 8], torch.float32),
    ('L5 fp32', (64, 40, 54), 4, 2, [-6, -9, -6, -9], torch.float32),
    ('ToRGB', (3, 144, 256), 1, 1, [0, 0, 0, 0], torch.float16),
]
FL_SCALES = {1.0: 'unit', 300.0: 'clamping'}


def run_filtered_lrelu(ops, chw, up, down, pad, dtype, scale):
    nt = 2
    fu = kaiser(6 * up, up).to(DEV) if up > 1 else None
    fd = kaiser(6 * down, down).to(DEV) if down > 1 else None
    x = rnd((nt,) + chw, 9, dtype, scale)
    b = rnd((chw[0],), 10, dtype)
    gain, slope = (1.0, 1.0) if up == 1 else (math.sqrt(2), 0.2)
    xg, bg = x.clone().requires_grad_(True), b.clone().requires_grad_(True)
    y = ops.filtered_lrelu.filtered_lrelu(xg, fu=fu, fd=fd, b=bg, up=up, down=down, padding=pad, gain=gain, slope=slope, clamp=256)
    dy = rnd(tuple(y.shape), 11, dtype)
    dx, db = torch.autograd.grad(y, [xg, bg], dy)
    return {'y': y.detach(), 'dx': dx, 'db': db}


@pytest.mark.parametrize('scale', [1.0, 300.0], ids=['unit', 'clamping'])
@pytest.mark.parametrize('name,chw,up,down,pad,dtype', FL, ids=[f[0] for f in FL])
def test_filtered_lrelu_vs_reference_cuda(name, chw, up, down, pad, dtype, scale):
    ra, rg = tols(dtype)
    if dtype == torch.float16:
        ra = 6e-3         # two-stage fp32 pipeline rounded to fp16 once on each side; signs of tiny values may differ
    got = run_filtered_lrelu(OURS, chw, up, down, pad, dtype, scale)
    key = f'{name}/{FL_SCALES[scale]}'
    elementwise(got['y'], Ref('filtered_lrelu', f'{key}/y'), ra, f'{name} y')
    # gradients: an element whose pre-activation sits within rounding of 0 or of the clamp may take the other branch on
    # either side (both are "right"); such flips are rare and bounded -- allow 1e-4 of the elements beyond 1e-2
    ref = Ref('filtered_lrelu', f'{key}/dx')
    g, w = ref.got(got['dx'], f'{name} dx'), ref.v.double()
    bound = rg * w.abs() + rg * FLOOR * ref.scale
    frac = float(((g - w).abs() > bound).double().mean())
    assert frac <= 1e-4, f'{name} dx: {frac:.2e} of sampled elements outside {rg:g}'
    assert float((g - w).norm() / w.norm()) <= rg * 0.1, f'{name} dx L2 (sampled elements)'
    full = got['dx'].double()
    assert abs(float(full.norm()) - ref.norm) <= rg * 0.1 * ref.norm, f'{name} dx: ||got|| {float(full.norm()):.7g}, ||ref|| {ref.norm:.7g}'
    elementwise(got['db'], Ref('filtered_lrelu', f'{key}/db'), 2e-2 if dtype == torch.float16 else rg, f'{name} db')


# ------------------------------------------------------------------ conv2d_resample (a4) on the sres D shapes

CR = [
    # name, x shape, w shape, kwargs, dtype  (discriminator_sres.py:192-204: f = [1,3,3,1] 2-D, flip_weight = (up == 1))
    ('fromrgb 1x1', (2, 24, 256, 256), (64, 24, 1, 1), dict(), torch.float16),
    ('b256 conv0 3x3', (2, 64, 128, 128), (64, 64, 3, 3), dict(padding=1), torch.float16),
    ('b256 conv1 3x3 down2', (2, 64, 128, 128), (128, 64, 3, 3), dict(down=2, padding=1, f=True), torch.float16),
    ('b256 skip 1x1 down2', (2, 64, 128, 128), (128, 64, 1, 1), dict(down=2, f=True), torch.float16),
    ('b32 conv1 down2', (2, 512, 32, 32), (512, 512, 3, 3), dict(down=2, padding=1, f=True), torch.float16),
    ('b16 conv0 fp32', (2, 512, 16, 16), (512, 512, 3, 3), dict(padding=1), torch.float32),
    ('b16 conv1 down2 fp32', (2, 512, 16, 16), (512, 512, 3, 3), dict(down=2, padding=1, f=True), torch.float32),
    ('b16 skip fp32', (2, 512, 16, 16), (512, 512, 1, 1), dict(down=2, f=True), torch.float32),
    ('epilogue 4x4 fp32', (2, 512, 4, 4), (512, 512, 3, 3), dict(padding=1), torch.float32),
]


def run_conv2d_resample(ops, xs, ws, kw, dtype):
    # The reference's conv is cuDNN (conv2d_gradfix.py:37-45 -> F.conv2d; fp32 with TF32 off as train_sres.py sets it);
    # ours is the tcgen05 kernel where native. Tolerance: fp16 operands, fp32 accumulation on both sides.
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    kw = dict(kw)
    f = upfirdn2d.setup_filter(F4, separable=False).to(DEV) if kw.pop('f', False) else None
    fan = ws[1] * ws[2] * ws[3]
    x = rnd(xs, 12, dtype)
    w = rnd(ws, 13, dtype, 1.0 / math.sqrt(fan))
    xg, wg = x.clone().requires_grad_(True), w.clone().requires_grad_(True)
    y = ops.conv2d_resample.conv2d_resample(xg, wg, f=f, **kw)
    dy = rnd(tuple(y.shape), 14, dtype)
    dx, dw = torch.autograd.grad(y, [xg, wg], dy)
    return {'y': y.detach(), 'dx': dx, 'dw': dw}


@pytest.mark.parametrize('name,xs,ws,kw,dtype', CR, ids=[c[0] for c in CR])
def test_conv2d_resample_vs_reference_cuda(name, xs, ws, kw, dtype):
    got = run_conv2d_resample(OURS, xs, ws, kw, dtype)
    ra, rg = (1e-3, 1e-2) if dtype == torch.float32 else (6e-3, 1.5e-2)
    elementwise(got['y'], Ref('conv2d_resample', f'{name}/y'), ra, f'{name} y')
    elementwise(got['dx'], Ref('conv2d_resample', f'{name}/dx'), rg, f'{name} dx')
    elementwise(got['dw'], Ref('conv2d_resample', f'{name}/dw'), rg, f'{name} dw')


def run_modulated_conv(ops):
    # generator_sres.py:44-67: grouped conv with per-sample weights, padding k-1, followed by filtered_lrelu
    nt, cin, cout, h, w_ = 4, 155, 128, 40, 54
    x = rnd((1, nt * cin, h, w_), 15, torch.float16)
    wt = rnd((nt * cout, cin, 3, 3), 16, torch.float16, 1.0 / math.sqrt(cin * 9))
    b = rnd((cout,), 17, torch.float16)
    fu, fd = kaiser(12, 2).to(DEV), kaiser(12, 2).to(DEV)
    xg, wg = x.clone().requires_grad_(True), wt.clone().requires_grad_(True)
    y = ops.conv2d_gradfix.conv2d(xg, wg, padding=2, groups=nt).reshape(nt, cout, h + 2, w_ + 2)
    y = ops.filtered_lrelu.filtered_lrelu(y, fu=fu, fd=fd, b=b, up=2, down=2, padding=[9, 8, 9, 8], clamp=256)
    dy = rnd(tuple(y.shape), 18, torch.float16)
    dx, dw = torch.autograd.grad(y, [xg, wg], dy)
    return {'y': y.detach(), 'dx': dx, 'dw': dw}


def test_modulated_conv_path_vs_reference_cuda():
    got = run_modulated_conv(OURS)
    elementwise(got['y'], Ref('conv2d_resample', 'modulated/y'), 6e-3, 'y')
    for n in ('dx', 'dw'):
        ref = Ref('conv2d_resample', f'modulated/{n}')
        a, r = ref.got(got[n], n), ref.v.double()
        assert float((a - r).norm() / r.norm()) <= 1e-2, f'{n} (sampled elements)'
        full = got[n].double()
        assert abs(float(full.norm()) - ref.norm) <= 1e-2 * ref.norm, f'{n}: ||got|| {float(full.norm()):.7g}, ||ref|| {ref.norm:.7g}'


# every stored case: golden file -> [(key prefix, function of the ops namespace -> {tensor name: tensor})]
def golden_cases():
    out = {'bias_act': [(str(i), lambda ops, c=c: run_bias_act(ops, *c)) for i, c in enumerate(BIAS_ACT)]
           + [('r1', run_bias_act_r1)],
           'upfirdn2d': [(u[0], lambda ops, u=u: run_upfirdn2d(ops, *u[1:])) for u in UPFIRDN],
           'filtered_lrelu': [(f'{f[0]}/{tag}', lambda ops, f=f, v=v: run_filtered_lrelu(ops, *f[1:], v))
                              for f in FL for v, tag in FL_SCALES.items()],
           'conv2d_resample': [(c[0], lambda ops, c=c: run_conv2d_resample(ops, *c[1:])) for c in CR]
           + [('modulated', run_modulated_conv)]}
    return out
