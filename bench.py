"""Benchmark of the hot path: one G+D training step's worth of torch_utils.ops calls.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload lres|sres] [--impl ours|reference] [--dump-outputs DIR]

A "step" replays, through this repository's public ops (torch_utils.ops.* -> C ABI -> sm_100a
kernels), every hot-path operator call that one LongVideoGAN training step issues, at the real
shapes: the call trace was recorded from the unmodified reference networks
(tools/trace_reference_workload.py -> workloads/*.json) and is replayed as
    update_G : G forward+backward, D forward+backward          (video_gan_lres.py:100-131)
    update_D : G forward (no grad), D forward+backward on fake and on real   (:133-176)
i.e. G ops 2x forward + 1x backward, D ops 3x (forward + backward), on synthetic tensors
(N(0,1) activations, Kaiser/binomial-shaped filters). Convolutions outside the torch_utils.ops
API (F.conv3d / F.conv1d, SURVEY.md row N1) are not part of this path and are not replayed.

Default workload = BASELINE.json configs[1]: train_lres, 128-frame 64x36 video, per-GPU batch 8.
With --gpus N (torchrun, one rank per GPU) each rank runs the same per-GPU batch (weak scaling)
and the step ends with the flat-buffer NCCL gradient all-reduce of G and D
(long-video-gan_b200/lvg_dist/grad_sync.py, replacing utils.sync_grads).

Output: ONE JSON line on rank 0 (see the keys below). `value` = frames/s with inputs resident
in HBM; `e2e` = the same with the step's real-video batch copied from pinned host memory and
the result read back inside the timed region; `roofline` = achieved algorithmic HBM GB/s of the
dominant kernel (bias_act), timed with CUDA events inside the timed steps; `cpu_baseline` = the
CPU oracle (oracle/, a port of the reference's _ref path) on a bounded sample, reported only.

Inputs are seeded: with the same arguments every run replays the same tensors. --dump-outputs DIR writes, after the
timed steps, what the last timed step of each measured run computed -- a fixed, seeded sample (OutputSampler.N elements)
of every output and gradient the replayed calls hand back, and of the optimiser's parameters -- as float32
DIR/<run>.<net>.<call>_<op>.<what>.npy, so that two builds can be compared output for output. The sample is gathered on
the device inside the step (CUDA graphs included), which adds small gather launches to every step timed in that mode
-- the e2e and eager figures of a dump run as well as `value`; runs without --dump-outputs have none.
"""
import argparse
import json
import os
import subprocess
import sys
import time
import zlib

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, 'long-video-gan_b200'))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

WORKLOADS = {
    # name: (trace file, G pass, D pass, per-GPU batch, frames per sample)
    'lres': ('lres_step.json', 'lres_G', 'lres_D', 8, 128),
    'sres': ('sres_step.json', 'sres_G', 'sres_D', 16, 8),
}
GRAD_ELEMS = {'lres': (83_200_000, 46_400_000), 'sres': (27_200_000, 24_000_000)}   # G, D parameter counts (SURVEY.md 2b)
HOT_OPS = ('bias_act', 'upfirdn2d', 'filtered_lrelu', 'conv2d_resample', 'conv2d')
CONV_OPS = ('conv3d', 'conv1d')      # F.conv3d / F.conv1d of the low-res networks (SURVEY row N1): replayed with --scope full


SCOPE = {'ops': HOT_OPS, 'full': HOT_OPS + CONV_OPS}
_scope = 'full'


def load_trace(name, scope=None):
    fname, gkey, dkey, batch, frames = WORKLOADS[name]
    keep = SCOPE[scope or _scope]
    tr = json.load(open(os.path.join(ROOT, 'workloads', fname)))
    return [c for c in tr[gkey] if c['op'] in keep], [c for c in tr[dkey] if c['op'] in keep], batch, frames


def make_filter(shape, gen):
    """Low-pass-like synthetic taps of the recorded shape (values do not affect timing)."""
    if shape is None:
        return None
    if len(shape) == 2 and min(shape) > 1:
        # the networks' 2-D filters are outer products of 1-D taps (setup_filter([1, 3, 3, 1]), upfirdn2d.py:103-108)
        fy, fx = torch.rand(shape[0], generator=gen) + 0.1, torch.rand(shape[1], generator=gen) + 0.1
        f = torch.outer(fy, fx)
        return (f / f.sum()).float()
    f = torch.rand(*shape, generator=gen) + 0.1
    return (f / f.sum()).float()


def scaled(shape, batch):
    return [shape[0] * batch] + list(shape[1:])


# ---------------------------------------------------------------------------------------------
# our arm: replay through torch_utils.ops on the GPU

def run_backward(y, leaves, dy):
    """Backward of ONE replayed call -> the gradients of `leaves`. A training step calls loss.backward() once; replaying
    the calls one by one would pay torch.autograd.grad's Python-side argument validation (~50 us) per call, which is
    harness overhead, not operator cost -- so the autograd engine is entered directly (what torch.autograd.grad does
    after validating)."""
    try:
        return torch.autograd.variable.Variable._execution_engine.run_backward(
            (y,), (dy,), False, False, tuple(leaves), allow_unreachable=True, accumulate_grad=False)
    except (AttributeError, TypeError):
        return torch.autograd.grad(y, leaves, dy, allow_unused=True)


class OutputSampler:
    """Gathers a fixed sample of every tensor handed to `keep` into a float32 device buffer per key (one take + one copy
    launch, so it can sit inside a captured graph). The sample positions of a key are drawn, seeded by the key, when the
    key is first seen -- in an eager warm-up step, before any capture."""
    N = 4096

    def __init__(self, prefix):
        self.prefix = prefix
        self.idx, self.buf = {}, {}

    def keep(self, key, t):
        if t is None:
            return
        key = self.prefix + key
        if key not in self.idx:
            n = t.numel()
            sel = np.sort(np.random.default_rng(zlib.crc32(key.encode())).choice(n, min(n, self.N), replace=False))
            self.idx[key] = torch.from_numpy(sel).to(t.device)
            self.buf[key] = torch.empty(len(sel), dtype=torch.float32, device=t.device)
        self.buf[key].copy_(torch.take(t.detach(), self.idx[key]))

    def snapshot(self):
        return {k: v.cpu().numpy() for k, v in self.buf.items()}


class Replay:
    def __init__(self, calls, batch, device, dtype_policy, ops=None, tag=''):
        if ops is None:
            from torch_utils.ops import bias_act, upfirdn2d, filtered_lrelu, conv2d_resample, conv2d_gradfix, conv_nd
            ops = dict(bias_act=bias_act, upfirdn2d=upfirdn2d, filtered_lrelu=filtered_lrelu, conv2d_resample=conv2d_resample,
                       conv2d=conv2d_gradfix, conv3d=conv_nd.conv3d, conv1d=conv_nd.conv1d)
        self.ops = ops
        self.last_y = None
        self.sampler = None          # an OutputSampler when the outputs are dumped
        self.device = device
        self.pool = {}
        self.items = []
        gen = torch.Generator().manual_seed(0)
        for c in calls:
            dt = torch.float16 if (c.get('fp16') and dtype_policy == 'mixed') else torch.float32
            if c['op'] == 'conv2d':
                # modulated convolution: the batch lives in the groups (x [1, G*Cin, H, W], w [G*Cout, Cin, k, k])
                xs = [1, c['x'][1] * batch] + list(c['x'][2:])
                x = self._buf('x', xs, dt)
                item = dict(c=c, x=x, dtype=dt, groups=c['groups'] * batch, key=f"{tag}{len(self.items):03d}_{c['op']}")
                ws = [c['w'][0] * batch] + list(c['w'][1:])
                item['w'] = (torch.randn(*ws, device=device) / np.sqrt(np.prod(c['w'][1:]))).to(dt)
                self.items.append(item)
                continue
            x = self._buf('x', scaled(c['x'], batch), dt)
            item = dict(c=c, x=x, dtype=dt, key=f"{tag}{len(self.items):03d}_{c['op']}")
            if c['op'] in CONV_OPS:
                item['w'] = (torch.randn(*c['w'], device=device) / np.sqrt(np.prod(c['w'][1:]))).to(dt)
                item['nograd'] = c['groups'] > 1          # BlurredNoise.blur: fixed filters on a noise input (generator_lres.py:378-387)
            elif c['op'] == 'bias_act':
                item['b'] = torch.randn(c['x'][c['dim']], device=device, dtype=dt) if c['b'] else None
            elif c['op'] == 'upfirdn2d':
                item['f'] = None if c['f'] is None else make_filter(c['f'], gen).to(device)
            elif c['op'] == 'filtered_lrelu':
                item['fu'] = None if c['fu'] is None else make_filter(c['fu'], gen).to(device)
                item['fd'] = None if c['fd'] is None else make_filter(c['fd'], gen).to(device)
                item['b'] = torch.randn(c['x'][1], device=device, dtype=dt) if c['b'] else None
            elif c['op'] == 'conv2d_resample':
                item['w'] = (torch.randn(*c['w'], device=device) / np.sqrt(np.prod(c['w'][1:]))).to(dt)
                item['f'] = None if c['f'] is None else make_filter(c['f'], gen).to(device)
            self.items.append(item)
        # output shapes (and dy buffers) from one dry forward
        with torch.no_grad():
            for it in self.items:
                y = self._fwd(it, it['x'])
                it['dy'] = self._buf('dy', list(y.shape), y.dtype)
                it['bytes_fwd'] = (it['x'].numel() + y.numel()) * y.element_size()
                # bias_act: relu / lrelu keep 2-bit codes for the backward pass (x + y + n/4 forward with grad, dy + dx + n/4
                # backward); other activations re-read y in the backward pass (dy + y + dx)
                if it['c']['op'] in CONV_OPS + ('conv2d',) or (it['c']['op'] == 'conv2d_resample'):
                    it['flops_fwd'] = 2.0 * y.numel() * float(np.prod(it['w'].shape[1:]))
                coded = it['c']['op'] == 'bias_act' and it['c']['act'] in ('relu', 'lrelu')
                it['bytes_fwd_grad'] = it['bytes_fwd'] + (y.numel() // 4 if coded else 0)
                it['bytes_bwd'] = it['bytes_fwd'] + (y.numel() // 4 if coded else (y.numel() * y.element_size() if it['c']['op'] == 'bias_act' else 0))
                del y

    def _buf(self, kind, shape, dt):
        key = (kind, tuple(shape), dt)
        if key not in self.pool:
            self.pool[key] = torch.randn(*shape, device=self.device, dtype=dt)
        return self.pool[key]

    def _fwd(self, it, x):
        c = it['c']
        if c['op'] == 'bias_act':
            return self.ops['bias_act'].bias_act(x, it['b'], dim=c['dim'], act=c['act'], alpha=c['alpha'], gain=c['gain'], clamp=c['clamp'])
        if c['op'] == 'upfirdn2d':
            return self.ops['upfirdn2d'].upfirdn2d(x, it['f'], up=c['up'], down=c['down'], padding=c['padding'],
                                                   flip_filter=c['flip_filter'], gain=c['gain'])
        if c['op'] == 'filtered_lrelu':
            return self.ops['filtered_lrelu'].filtered_lrelu(x, fu=it['fu'], fd=it['fd'], b=it['b'], up=c['up'], down=c['down'],
                                                             padding=c['padding'], gain=c['gain'], slope=c['slope'],
                                                             clamp=c['clamp'], flip_filter=c['flip_filter'])
        if c['op'] == 'conv2d':
            return self.ops['conv2d'].conv2d(x, it['w'], padding=c['padding'], groups=it['groups'])
        if c['op'] in CONV_OPS:
            return self.ops[c['op']](x, it['w'], None, c['stride'], c['padding'], 1, c['groups'])
        return self.ops['conv2d_resample'].conv2d_resample(x, it['w'], f=it['f'], up=c['up'], down=c['down'], padding=c['padding'],
                                                           groups=c['groups'], flip_weight=c['flip_weight'], flip_filter=c['flip_filter'])

    def _keep(self, it, what, t):
        if self.sampler is not None:
            self.sampler.keep(f"{it['key']}.{what}", t)

    def forward_only(self):
        with torch.no_grad():
            for it in self.items:
                self.last_y = self._fwd(it, it['x'])
                self._keep(it, 'y_nograd', self.last_y)

    def forward_backward(self, timer=None, lo=0, hi=None):
        for it in self.items[lo:hi]:
            if it.get('nograd'):
                with torch.no_grad():
                    self.last_y = self._fwd(it, it['x'])
                self._keep(it, 'y', self.last_y)
                continue
            x = it['x'].detach().requires_grad_(True)
            leaves, names = [x], ['dx']
            b = it.get('b')
            if b is not None:
                b = b.detach().requires_grad_(True)
                leaves.append(b)
                names.append('db')
            saved_b = it.get('b')
            it['b'] = b
            saved_w = it.get('w')
            if saved_w is not None:
                it['w'] = saved_w.detach().requires_grad_(True)
                leaves.append(it['w'])
                names.append('dw')
            grads = ()
            if timer is not None and it['c']['op'] in timer.ops:
                flops = it.get('flops_fwd')
                timer.start()
                y = self._fwd(it, x)
                timer.stop(it['bytes_fwd_grad'] if flops is None else flops)
                if y.requires_grad:
                    timer.start()
                    grads = run_backward(y, leaves, it['dy'])
                    timer.stop(it['bytes_bwd'] if flops is None else 2.0 * flops)
            else:
                y = self._fwd(it, x)
                if y.requires_grad:
                    grads = run_backward(y, leaves, it['dy'])
            self.last_y = y.detach()
            self._keep(it, 'y', self.last_y)
            for name, g in zip(names, grads):
                self._keep(it, name, g)
            it['b'] = saved_b
            if saved_w is not None:
                it['w'] = saved_w


class KernelTimer:
    """CUDA-event timing of individual calls inside the timed region (events on the current stream)."""

    def __init__(self, op='bias_act'):
        self.ops = (op,) if isinstance(op, str) else tuple(op)      # which replayed ops get the event pairs (the step's dominant kernel)
        self.pairs = []
        self._cur = None

    def start(self):
        self._cur = torch.cuda.Event(enable_timing=True)
        self._cur.record()

    def stop(self, nbytes):
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        self.pairs.append((self._cur, e, nbytes))

    def summary(self):
        ms = sum(a.elapsed_time(b) for a, b, _ in self.pairs)
        nbytes = sum(n for _, _, n in self.pairs)
        return ms, nbytes, len(self.pairs)


class ClockSampler:
    """Samples SM clock and throttle reasons through NVML every 100 ms while the timed region runs."""
    REASONS = {0x8: 'hw_slowdown', 0x40: 'hw_thermal_slowdown', 0x20: 'sw_thermal_slowdown', 0x4: 'sw_power_cap'}

    def __init__(self, index):
        import threading
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nv = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()
        except Exception:
            self._thread = None

    def _run(self):
        nv = self._nv
        while not self._stop.is_set():
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM)))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self._h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
                for bit, name in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.1)

    def finish(self):
        if self._thread is None:
            return None
        self._stop.set()
        self._thread.join(timeout=2)
        if not self.samples:
            return None
        return {'sm_mhz': float(np.median(self.samples)), 'sm_max_mhz': self.max_mhz, 'reasons': sorted(self.reasons),
                'samples': len(self.samples)}


def measured_peak(kind='hbm'):
    try:
        mp = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
        if kind == 'hbm':
            return mp['hbm_gbs'], 'measured (MEASURED_PEAKS.json hbm_gbs)'
        return mp['bf16_tflops_sustained'], 'measured (MEASURED_PEAKS.json bf16_tflops_sustained: the kernel is timed inside a long step)'
    except Exception:
        return (6650.0, 'fallback (B200_PROFILING.md 6.65 TB/s)') if kind == 'hbm' else (1400.0, 'fallback (B200_PROFILING.md ~1.4 PFLOP/s sustained)')


def metric_name(scope):
    return ('frames/sec (G+D train step: every convolution and torch_utils.ops call of the forward/backward passes, replayed)' if scope == 'full'
            else 'frames/sec (G+D train step, hot-path operator trace)')


def reference_ops(ref):
    """The reference's side of the replay: its own ops modules; its convolutions are torch.nn.functional (cuDNN / CPU), fp32 with
    TF32 off as train_lres.py:269-270 sets it."""
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    return dict(bias_act=ref.bias_act, upfirdn2d=ref.upfirdn2d, filtered_lrelu=ref.filtered_lrelu, conv2d_resample=ref.conv2d_resample,
                conv2d=ref.conv2d_gradfix, conv3d=torch.nn.functional.conv3d, conv1d=torch.nn.functional.conv1d)


# ---------------------------------------------------------------------------------------------
# CPU arms (reported-only baselines, host cores of the box)

def _host_threads():
    """All host cores, whatever OMP_NUM_THREADS says (torchrun exports OMP_NUM_THREADS=1 to every rank)."""
    n = os.cpu_count() or 1
    torch.set_num_threads(n)
    return n


def cpu_sample_reference(workload, budget_s=20.0):
    """The REFERENCE'S OWN pure-PyTorch `_ref` op path (bias_act.py:91-120, upfirdn2d.py:167-211, filtered_lrelu.py:121-153,
    conv2d_resample.py over F.conv2d; staged unmodified at oracle/_ref/src) on CPU tensors, all host cores: forward AND
    backward (autograd) of the hot-path op calls of one G+D pass at batch 1, in trace order, until the time budget is
    used; the covered share of the pass's algorithmic bytes extrapolates to the whole pass. One training step = G ops
    2x forward + 1x backward, D ops 3x (forward + backward). -> (frames/s, description, threads, kind) or None."""
    from oracle import ref_cuda
    if not ref_cuda.available():
        return None
    threads = _host_threads()
    ref = ref_cuda.load()
    ops = reference_ops(ref)
    g_calls, d_calls, batch, frames = load_trace(workload)
    # groups = (network, op): sampled calls of a group extrapolate to the group's bytes (cost per byte differs by op);
    # calls are visited largest first within a fixed round-robin over the groups: a short budget samples every group and
    # measures the calls that carry most of the time directly
    groups = {}
    for net, calls in (('G', g_calls), ('D', d_calls)):
        for c in calls:
            groups.setdefault((net, c['op']), []).append(c)
    def weight(c):          # what a call's cost scales with inside its group: elements; multiply-adds for the convolutions
        if c['op'] in CONV_OPS:
            k = c['w'][2:]
            pad = c['padding'] if isinstance(c['padding'], (list, tuple)) else [c['padding']] * len(k)
            out = int(np.prod([s + 2 * p - kk + 1 for s, p, kk in zip(c['x'][2:], pad, k)]))
            return float(c['x'][0] * c['w'][0] * out) * float(np.prod(c['w'][1:]))
        return float(np.prod(c['x']))

    def bounded(c):
        """(call to run, factor): calls that would take many seconds on the host are cut along the time / plane axis (their cost
        is linear in it) and the measured time is scaled back by `factor` -- keeps every single sample, and so the arm, bounded."""
        cap = 4e9 if c['op'] in CONV_OPS else 2.5e7
        wgt = weight(c)
        if wgt <= cap:
            return c, 1.0
        xs = list(c['x'])
        axis = 2 if (c['op'] in CONV_OPS and len(xs) == 5) else max(range(min(3, len(xs))), key=lambda i: xs[i])
        lo = 4 * (c['w'][2] if c['op'] in CONV_OPS and len(xs) == 5 else 1)
        new = max(lo, min(xs[axis], int(xs[axis] * cap / wgt)))
        if c['op'] == 'bias_act' and axis == c.get('dim', 1):
            return c, 1.0                              # (the bias axis keeps its length)
        if new >= xs[axis]:
            return c, 1.0
        c2 = dict(c)
        xs2 = list(xs)
        xs2[axis] = new
        c2['x'] = xs2
        return c2, xs[axis] / float(new)

    for k in groups:
        groups[k].sort(key=lambda c: -weight(c))
    stat = {k: dict(tf=0.0, tb=0.0, done=0, total=sum(weight(c) for c in v)) for k, v in groups.items()}
    order, depth = [], 0
    while True:
        row = [(k, v[depth]) for k, v in groups.items() if depth < len(v)]
        if not row:
            break
        order += row
        depth += 1
    for key, v in groups.items():          # untimed: thread pool, primitive caches, allocator
        rp = Replay([v[-1]], 1, torch.device('cpu'), 'fp32', ops=ops)
        with torch.no_grad():
            rp._fwd(rp.items[0], rp.items[0]['x'])
    n_done = 0
    t_start = time.perf_counter()
    for key, c_full in order:
        if time.perf_counter() - t_start > budget_s:
            break
        c, factor = bounded(c_full)
        rp = Replay([c], 1, torch.device('cpu'), 'fp32', ops=ops)     # fp32 on CPU, as the reference's CPU path runs
        it = rp.items[0]
        x = it['x'].detach().requires_grad_(True)
        leaves = [x]
        if it.get('b') is not None:
            it['b'] = it['b'].detach().requires_grad_(True)
            leaves.append(it['b'])
        if it.get('w') is not None:
            it['w'] = it['w'].detach().requires_grad_(True)
            leaves.append(it['w'])
        t0 = time.perf_counter()
        y = rp._fwd(it, x)
        t1 = time.perf_counter()
        if y.requires_grad:
            torch.autograd.grad(y, leaves, it['dy'], allow_unused=True)
        t2 = time.perf_counter()
        st = stat[key]
        st['tf'] += (t1 - t0) * factor
        st['tb'] += (t2 - t1) * factor
        st['done'] += weight(c_full)
        n_done += 1
    for key, v in groups.items():          # a group the budget did not reach: its median call, so that every group has a rate
        if stat[key]['done'] == 0:
            c_full = v[len(v) // 2]
            c, factor = bounded(c_full)
            rp = Replay([c], 1, torch.device('cpu'), 'fp32', ops=ops)
            it = rp.items[0]
            x = it['x'].detach().requires_grad_(True)
            leaves = [x] + [it[k].detach().requires_grad_(True) for k in ('b', 'w') if it.get(k) is not None]
            for k in ('b', 'w'):
                if it.get(k) is not None:
                    it[k] = leaves[1 + [kk for kk in ('b', 'w') if it.get(kk) is not None].index(k)]
            t0 = time.perf_counter()
            y = rp._fwd(it, x)
            t1 = time.perf_counter()
            if y.requires_grad:
                torch.autograd.grad(y, leaves, it['dy'], allow_unused=True)
            stat[key]['tf'] += (t1 - t0) * factor
            stat[key]['tb'] += (time.perf_counter() - t1) * factor
            stat[key]['done'] += weight(c_full)
            n_done += 1
    est = 0.0
    for (net, _), st in stat.items():
        mult_f, mult_b = (2.0, 1.0) if net == 'G' else (3.0, 3.0)
        est += (mult_f * st['tf'] + mult_b * st['tb']) * st['total'] / st['done']
    done_bytes = {'all': sum(st['done'] for st in stat.values())}
    all_bytes = {'all': sum(st['total'] for st in stat.values())}
    fps = frames / est
    used = time.perf_counter() - t_start
    desc = (f"reference's own _ref ops (oracle/_ref/src, torch {torch.__version__} CPU, {threads} threads): forward+backward of {n_done} of "
            f"{len(order)} hot-path op calls of one G+D pass at batch 1 (of {batch}), {used:.1f} s, covering "
            f"{100.0 * sum(done_bytes.values()) / max(1, sum(all_bytes.values())):.0f} % of the pass's work (rest extrapolated per (network, op) group: by elements, by multiply-adds for convolutions; calls above 4e9 multiply-adds / 2.5e7 elements are cut along the time axis and scaled back); "
            f"step = G 2 fwd + 1 bwd, D 3 fwd + 3 bwd")
    return fps, desc, threads, 'reference'


def cpu_sample_port(workload, budget_s=20.0):
    """The CPU oracle (oracle/lvg_oracle.c, a float64 restatement) on a bounded sample of the same trace: repeated forward
    passes of every hot-path op call of one G+D pass at batch 1 until the time budget is used."""
    from oracle import oracle as orc
    threads = _host_threads()
    orc.set_num_threads(threads)
    g_calls, d_calls, batch, frames = load_trace(workload)
    gen = torch.Generator().manual_seed(0)
    rng = np.random.default_rng(0)
    calls = [c for c in g_calls + d_calls if c['op'] not in ('conv2d_resample', 'conv2d') + CONV_OPS]
    prepared = []
    for c in calls:
        item = {'c': c, 'x': rng.standard_normal(c['x'], dtype=np.float32)}
        if c['op'] == 'bias_act':
            item['b'] = np.zeros(c['x'][c['dim']], np.float32) if c['b'] else None
        elif c['op'] == 'upfirdn2d':
            item['f'] = None if c['f'] is None else make_filter(c['f'], gen).numpy()
        elif c['op'] == 'filtered_lrelu':
            item['fu'] = None if c['fu'] is None else make_filter(c['fu'], gen).numpy()
            item['fd'] = None if c['fd'] is None else make_filter(c['fd'], gen).numpy()
            item['b'] = np.zeros(c['x'][1], np.float32)
        prepared.append(item)
    t_used, passes = 0.0, 0
    while True:
        t0 = time.perf_counter()
        for it in prepared:
            c = it['c']
            if c['op'] == 'bias_act':
                orc.bias_act(it['x'], it['b'], c['dim'], c['act'], c['alpha'], c['gain'], c['clamp'])
            elif c['op'] == 'upfirdn2d':
                orc.upfirdn2d(it['x'], it['f'], c['up'], c['down'], c['padding'], c['flip_filter'], c['gain'])
            elif c['op'] == 'filtered_lrelu':
                orc.filtered_lrelu(it['x'], it['fu'], it['fd'], it['b'], c['up'], c['down'], c['padding'], c['gain'], c['slope'],
                                   c['clamp'], c['flip_filter'])
        t_used += time.perf_counter() - t0
        passes += 1
        if t_used >= budget_s or passes >= 64:
            break
    # one training step = (2 fwd + 1 bwd) of the G ops + 3 (fwd + bwd) of the D ops; a backward op costs about
    # a forward (same stencil transposed) -> ~4.5 forward-equivalents of the sampled G+D forward per step
    step_s_batch1 = (t_used / passes) * 4.5
    fps = frames / step_s_batch1
    desc = (f'{passes} forward passes of all {len(prepared)} hot-path op calls of one G+D pass at batch 1 (of {batch}) through the '
            f'CPU oracle (float64, {orc.num_threads()} OpenMP threads), {t_used:.1f} s; x4.5 forward-equivalents per training step')
    return fps, desc, orc.num_threads(), 'port'


def cpu_sample(workload, budget_s=20.0):
    """(frames/s, description, threads, kind): the reference's own CPU path when oracle/_ref is staged, else the port."""
    r = None
    try:
        r = cpu_sample_reference(workload, budget_s)
    except Exception as e:       # a broken stage must not take the bench down; say so
        sys.stderr.write(f'bench: reference _ref CPU arm unavailable ({type(e).__name__}: {e}); using the oracle port\n')
    return r if r is not None else cpu_sample_port(workload, budget_s)


# ---------------------------------------------------------------------------------------------
# multi-GPU: real Parameters + real autograd backward feeding lvg_dist.FlatGradSync(overlap=True)

class _InjectGrad(torch.autograd.Function):
    """Scalar node whose backward hands `g` to the parameter: what a weight-gradient kernel's output is to autograd."""

    @staticmethod
    def forward(ctx, p, g):
        ctx.save_for_backward(g)
        return p.new_zeros(())

    @staticmethod
    def backward(ctx, go):
        g, = ctx.saved_tensors
        return g, None


class UpdateTail:
    """The optimiser side of an update at the networks' parameter counts: FlatAdam over one flat fp32 buffer (+ the EMA copy
    for the generator, update_G_ema) -- sanitise, Adam and EMA in ONE kernel (lvg_adam_step) instead of the reference's
    ~900 per-tensor launches (utils.py:116-124, video_gan_lres.py:84-85,208-214). Gradients: the all-reduced flat buffer
    (several GPUs) or a synthetic one of the same size."""

    def __init__(self, n_elems, device, ema, params=None, grad_sync=None):
        from lvg_dist.flat_optim import FlatAdam
        if params is None:
            params = [torch.nn.Parameter(torch.randn(n_elems, device=device) * 0.02)]
        self.opt = FlatAdam(list(params), lr=3e-3, betas=(0.0, 0.99), grad_sync=grad_sync)
        if grad_sync is None:
            self.opt.flat_grads.normal_(0, 1e-3)
            for p, v in zip(self.opt.params, self.opt._grad_views):
                p.grad = v
        self.ema_flat = torch.zeros_like(self.opt.flat_params) if ema else None
        if ema:
            owner = self

            class _Ema:          # the parameters' EMA buffer, updated inside the optimiser kernel
                flat_params = owner.ema_flat

                @staticmethod
                def lerp_range(a, b, beta):
                    pass

                @staticmethod
                def update_buffers(beta):
                    pass
            self.opt._ema = _Ema

    def step(self, grad_scale=1.0):
        self.opt.step(grad_scale=grad_scale, ema_beta=0.999 if self.ema_flat is not None else None)


class GradExchange:
    """The gradient side of a network for the data-parallel step: `n_elems` fp32 parameters in tensors of the sizes a
    conv stack has, registered with FlatGradSync(overlap=True): each backward_bucket(k) runs a REAL autograd backward
    over the parameters of bucket k (AccumulateGrad -> post-accumulate hooks -> the bucket's asynchronous NCCL
    all-reduce starts while the remaining segments of the pass execute), finish() = FlatGradSync.sync()."""

    def __init__(self, n_elems, device, buckets, ema=False):
        from lvg_dist.grad_sync import FlatGradSync
        n_tensors = 96
        sizes = [n_elems // n_tensors] * n_tensors
        sizes[-1] += n_elems - sum(sizes)
        self.module = torch.nn.Module()
        self.module.ps = torch.nn.ParameterList([torch.nn.Parameter(torch.zeros(sz, device=device)) for sz in sizes])
        self.sync = FlatGradSync(self.module, overlap=True, buckets=buckets, backwards_per_sync=1)
        self.tail = UpdateTail(n_elems, device, ema, params=self.module.ps, grad_sync=self.sync)
        self.grads = [torch.randn(sz, device=device) * 1e-3 for sz in sizes]
        self.members = [[] for _ in range(len(self.sync._slices))]
        for i, b in self.sync._bucket_of.items():
            self.members[b].append(i)

    def backward_bucket(self, k):
        ps = self.sync.params
        outs = [_InjectGrad.apply(ps[i], self.grads[i]) for i in self.members[k]]
        torch.autograd.backward(outs)

    def finish(self, gain):
        # the tail of the update in ONE kernel: scale + nan_to_num of the all-reduced gradients, Adam, EMA (lvg_adam_step)
        self.sync.sync(gain=gain, postprocess=False)
        self.tail.step(self.sync.pending_scale)

    def begin(self):
        self.sync.zero_grad()


# ---------------------------------------------------------------------------------------------

def run_ours(args, workload, scope, steps, rank, world, local_rank, device, with_cpu, with_refcuda, dump=None):
    """One workload through this repository's ops on the GPU -> the JSON fields of its line. `dump` (a dict): receives
    the sampled outputs of the last step of the main timed region, keyed '<workload>.<scope>.<net><call>_<op>.<what>'."""
    global _scope
    import torch.distributed as dist
    from torch_utils import custom_ops
    _scope = scope
    torch.manual_seed(0)                     # the same inputs in every run with the same arguments
    g_calls, d_calls, batch, frames = load_trace(workload)
    policy = 'mixed' if workload == 'sres' else 'fp32'
    G = Replay(g_calls, batch, device, policy, tag='G')
    D = Replay(d_calls, batch, device, policy, tag='D')
    outputs = OutputSampler(f'{workload}.{scope}.') if dump is not None else None
    G.sampler = D.sampler = outputs
    kBuckets = 4
    ex_g = ex_d = None
    if world > 1:
        ng, nd = GRAD_ELEMS[workload]
        ex_g, ex_d = GradExchange(ng, device, kBuckets, ema=True), GradExchange(nd, device, kBuckets)
    else:
        ng, nd = GRAD_ELEMS[workload]
        tail_g, tail_d = UpdateTail(ng, device, ema=True), UpdateTail(nd, device, ema=False)

    # e2e: the step's real-video batch comes from pinned host memory and ENTERS the replay: lres -- the discriminator's
    # first layer (pad to 64x64, 1x1x1 conv 3->32, discriminator_lres.py:135-213; a library conv, row N1) is computed from
    # the copied video into the input buffer of the first replayed D op; sres -- the copied low-res clip IS the input of
    # the first replayed D op (upfirdn2d of (N, 3T, 36, 64), discriminator_sres.py:512). The value read back is the first
    # element of the last D op's output of that step (a computed result).
    entry = D.items[0]
    if workload == 'lres':
        host_video = torch.empty((batch, 3, frames, 36, 64), dtype=torch.float32).uniform_(-1, 1).pin_memory()
        dev_video = torch.empty_like(host_video, device=device)
        direct = entry['x'].shape[1] == 3        # --scope full: the first replayed D op IS that first conv3d on the padded video
        w_in = None if direct else torch.randn(entry['x'].shape[1], 3, 1, 1, 1, device=device) / 3 ** 0.5
        assert tuple(entry['x'].shape) == (batch, entry['x'].shape[1], frames, 64, 64), entry['x'].shape

        def ingest():
            dev_video.copy_(host_video, non_blocking=True)
            v = torch.nn.functional.pad(dev_video, (0, 0, 14, 14))
            entry['x'].copy_(v if direct else torch.nn.functional.conv3d(v, w_in))
    else:
        host_video = torch.empty(tuple(entry['x'].shape), dtype=torch.float32).uniform_(-1, 1).pin_memory()
        stage = torch.empty_like(host_video, device=device)

        def ingest():
            stage.copy_(host_video, non_blocking=True)
            entry['x'].copy_(stage)          # fp32 -> the layer's dtype
    host_out = torch.empty(1, dtype=torch.float32).pin_memory()

    # One step = update_G (G fwd+bwd, D fwd+bwd) then update_D (G fwd, D fwd+bwd on fakes, D fwd+bwd on reals).
    # Each half is a list of SEGMENTS. With one GPU a half is one segment. With several GPUs the network whose
    # gradients the half exchanges goes last and its second half is cut into kBuckets segments: after segment k a real
    # autograd backward over the parameters of bucket k runs, whose FlatGradSync hooks start that bucket's all-reduce
    # asynchronously (NCCL's own stream), overlapping the remaining segments; only the last bucket's exchange is exposed.
    def tail_cuts(n):
        half = n // 2
        return [half + (n - half) * k // kBuckets for k in range(kBuckets + 1)]

    if world == 1:
        # every update ends with its optimiser tail (G: Adam + EMA of the generator, D: Adam) at the networks' parameter counts
        segs_a = [lambda timer=None: (G.forward_backward(timer), D.forward_backward(timer), tail_g.step())]
        segs_b = [lambda timer=None: (G.forward_only(), D.forward_backward(timer), D.forward_backward(timer), tail_d.step())]
    else:
        ca, cb = tail_cuts(len(G.items)), tail_cuts(len(D.items))
        segs_a = [lambda timer=None: (D.forward_backward(timer), G.forward_backward(timer, 0, ca[0]))]
        segs_a += [(lambda timer=None, k=k: G.forward_backward(timer, ca[k], ca[k + 1])) for k in range(kBuckets)]
        segs_b = [lambda timer=None: (G.forward_only(), D.forward_backward(timer), D.forward_backward(timer, 0, cb[0]))]
        segs_b += [(lambda timer=None, k=k: D.forward_backward(timer, cb[k], cb[k + 1])) for k in range(kBuckets)]

    graphs = {}

    def run_half(name, segs, ex, timer, eager, prefill):
        if prefill:                          # see the roofline pass below
            torch.cuda._sleep(prefill)
        if ex is not None:
            ex.begin()
        for i, seg in enumerate(segs):
            if graphs and not eager:
                graphs[name][i].replay()
            else:
                seg(timer)
            if ex is not None and i >= 1:
                ex.backward_bucket(i - 1)
        if ex is not None:
            ex.finish(gain=1.0)

    def step(timer=None, e2e=False, eager=False, prefill=False):
        if e2e:
            ingest()
        run_half('a', segs_a, ex_g, timer, eager, prefill)
        run_half('b', segs_b, ex_d, timer, eager, prefill)
        if e2e:
            host_out.copy_(D.last_y.reshape(-1)[:1].float(), non_blocking=True)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(nsteps, e2e, timer=None, eager=False):
        barrier()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(nsteps):
            step(timer, e2e, eager)
        t1.record()
        barrier()
        ms = torch.tensor([t0.elapsed_time(t1)], device=device)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    warm = max(3, args.warmup)               # W >= 3 untimed steps, exactly as asked
    for _ in range(warm):
        step()
    torch.cuda.synchronize()
    dominant_op = ('conv3d' if scope == 'full' else 'bias_act') if workload == 'lres' else 'filtered_lrelu'
    launches_per_step = None
    if args.launch == 'graph':
        # Capture the two halves of the step (the gradient exchange stays outside: eager autograd + NCCL between the replays).
        # Launch counting happens while capturing: exactly one step's kernels.
        pool = None
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        launches0 = custom_ops.launch_count()
        with torch.cuda.stream(side):
            captured = {}
            for name, segs in (('a', segs_a), ('b', segs_b)):
                captured[name] = []
                for seg in segs:
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g, pool=pool, stream=side, capture_error_mode='thread_local'):
                        seg()
                    pool = g.pool()
                    captured[name].append(g)
            graphs.update(captured)
        torch.cuda.current_stream().wait_stream(side)
        launches_per_step = custom_ops.launch_count() - launches0
        step()                               # first replay (untimed)
        torch.cuda.synchronize()
    else:
        step(KernelTimer(dominant_op))       # untimed: same code path as the timed region (event pairs included)
    launches0 = custom_ops.launch_count()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    timer = KernelTimer(dominant_op)
    ms_total = timed(steps, e2e=False, timer=None if graphs else timer)
    if outputs is not None:
        # the optimiser's state after the last timed step (sampled outside the timed region), then everything kept so far
        tails = (tail_g, tail_d) if world == 1 else (ex_g.tail, ex_d.tail)
        for net, tail in zip('GD', tails):
            outputs.keep(f'{net}.adam.params', tail.opt.flat_params)
            outputs.keep(f'{net}.adam.ema', tail.ema_flat)
        dump.update(outputs.snapshot())
        G.sampler = D.sampler = None
    launches = launches_per_step * steps if graphs else custom_ops.launch_count() - launches0
    step(e2e=True)                           # untimed warm-up of the host-copy flavour
    ms_e2e = timed(steps, e2e=True)
    ms_e2e_eager = timed(steps, e2e=True, eager=True) if graphs else ms_e2e
    clocks = sampler.finish() if sampler is not None else None
    if graphs:
        # Per-kernel timing for the roofline: graph nodes cannot carry timing events, so one extra EAGER step is timed
        # with an event pair around every call of the dominant op. The stream is pre-filled with a ~30 ms spin kernel
        # before each half so that the host runs ahead and the pairs bracket kernel execution, not Python launch latency.
        spin = int(0.03 * 1.9e9)
        step(KernelTimer(dominant_op), eager=True, prefill=spin)
        torch.cuda.synchronize()
        step(timer, eager=True, prefill=spin)
        torch.cuda.synchronize()

    frames_per_step = batch * frames * world
    value = frames_per_step * steps / (ms_total / 1000.0)
    e2e_value = frames_per_step * steps / (ms_e2e / 1000.0)
    k_ms, k_bytes, k_n = timer.summary()
    tensor_bound = dominant_op == 'conv3d'
    peak, peak_src = measured_peak('tensor' if tensor_bound else 'hbm')
    achieved = k_bytes / (k_ms / 1000.0) / (1e12 if tensor_bound else 1e9) if k_ms > 0 else 0.0
    if graphs:
        k_share = k_ms / (ms_total / steps) if ms_total else None
        k_how = (f'CUDA events around every {dominant_op} call of one extra eager step (stream pre-filled by a spin kernel so that the '
                 'pairs bracket execution, not launch latency); the timed region itself replays CUDA graphs')
    else:
        k_share = k_ms / ms_total if ms_total else None
        k_how = f'CUDA events around every {dominant_op} call inside the timed region'

    traffic, traffic_note = None, None
    if workload == 'lres' and not tensor_bound:
        try:    # DRAM bytes of the dominant kernel from the committed ncu --set full capture (bench.py never runs under ncu)
            tr = json.load(open(os.path.join(ROOT, 'profiles', 'r01_traffic.json')))
            f, b = tr['bias_act_fwd'], tr['bias_act_bwd_fused_db']
            traffic = (f['dram_read'] + f['dram_write'] + b['dram_read'] + b['dram_write']) / 2.0
            traffic_note = (f"mean DRAM bytes per launch (one forward + one fused backward launch) at {tr['shape']}; algorithmic "
                            f"{(f['algorithmic'] + b['algorithmic']) / 2.0:.0f} B; {tr['source']}")
        except Exception:
            pass
    res = config = None
    if rank == 0:
        what = ('convolutions + torch_utils.ops calls of G+D update' if scope == 'full' else 'torch_utils.ops calls of G+D update')
        config = {'workload': f'{workload}: train_{workload} op trace ({what}), per-GPU batch {batch}, '
                              f'{frames} frames/sample, {"64x36" if workload == "lres" else "256x144 from 64x36"}',
                  'global_batch': batch * world, 'parallelism': f'dp{world}',
                  'l2': 'inputs and outputs of the replayed calls exceed L2 (largest tensors 0.75 GB); buffers shared per shape',
                  'launch': ('cuda_graph (step captured once, replayed' + ('; between the graph segments: real autograd backward over real Parameters -> lvg_dist.FlatGradSync(overlap=True) hooks -> bucketed NCCL all-reduces overlapping the rest of the pass)' if world > 1 else ')')) if args.launch == 'graph'
                            else 'eager (every call launched from Python)'}
        res = {'metric': metric_name(scope), 'value': value, 'unit': 'frames/s', 'n_gpus': world, 'steps': steps, 'warmup': warm,
               'ms_per_step': ms_total / steps,
               'dtype': 'f32' if policy == 'fp32' else 'f16/f32 mixed (fp16 layers as the reference config)',
               'config': config, 'gpu_launches': int(launches),
               'e2e': {'value': e2e_value, 'unit': 'frames/s', 'h2d_bytes_per_step': host_video.numel() * 4, 'd2h_bytes_per_step': 4,
                       'eager_value': frames_per_step * steps / (ms_e2e_eager / 1000.0),
                       'path': 'pinned host video -> device -> first replayed discriminator op; first element of the last discriminator output -> host'},
               'roofline': {'bound': 'tensor' if tensor_bound else 'hbm',
                            'kernel': {'bias_act': 'bias_act (vector kernel: forward writing 2-bit sign/clamp codes + backward from the codes with fused dx/db)',
                                       'filtered_lrelu': 'filtered_lrelu (fused up-FIR / lrelu / down-FIR; FP32-issue-bound, its HBM figure is shown for reference)',
                                       'conv3d': 'conv_igemm_kernel / conv_wgrad_v2_kernel (TMA-fed tcgen05 implicit GEMM; fp32 layers as bf16 hi/lo split: 3 tensor-core '
                                                 'products per algorithmic product, so the tensor pipe executes 3x the achieved figure) incl. its operand re-tiling passes'}[dominant_op],
                            'achieved': achieved,
                            'peak': peak, 'peak_source': peak_src, 'unit': 'TFLOP/s' if tensor_bound else 'GB/s', 'frac': achieved / peak if peak else None,
                            'launches_timed': k_n, 'share_of_step': k_share, 'traffic': traffic, 'traffic_note': traffic_note, 'timing': k_how},
               'clocks': clocks}
    # the same trace through the REFERENCE'S OWN CUDA ops on this GPU (oracle/_ref: its plugins built unmodified for sm_100a,
    # its Python wrappers, cuDNN for its convolutions) -- eager on both sides, N = 1 only: the "beat-this" baseline
    if rank == 0 and world == 1 and with_refcuda:
        try:
            from oracle import ref_cuda
            if ref_cuda.available():
                del G, D
                graphs.clear()
                torch.cuda.empty_cache()
                ref = ref_cuda.load()
                rops = reference_ops(ref)
                RG, RD = Replay(g_calls, batch, device, policy, ops=rops), Replay(d_calls, batch, device, policy, ops=rops)

                def rstep():
                    RG.forward_backward(); RD.forward_backward()
                    RG.forward_only(); RD.forward_backward(); RD.forward_backward()
                # one warm-up step, timed: a slow reference step (the super-res trace takes ~11 s on B200) gets 2 timed steps
                # without a second warm-up, a fast one a second warm-up and up to 5 -- the default run must end within minutes
                w0, w1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                w0.record()
                rstep()
                w1.record()
                torch.cuda.synchronize()
                if w0.elapsed_time(w1) > 1500.0:
                    nref = 2
                else:
                    nref = max(2, min(steps, 5))
                    rstep()
                    torch.cuda.synchronize()
                t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                t0.record()
                for _ in range(nref):
                    rstep()
                t1.record()
                torch.cuda.synchronize()
                rms = t0.elapsed_time(t1) / nref
                res['ref_cuda'] = {'value': batch * frames / (rms / 1000.0), 'unit': 'frames/s', 'ms_per_step': rms, 'steps': nref,
                                   'launch': 'eager', 'ours_eager_ms_per_step': ms_e2e_eager / steps,
                                   'what': "the same op trace through the reference's own CUDA plugins (built unmodified for sm_100a, "
                                           "oracle/_ref) and Python wrappers on this GPU; compare with ours_eager_ms_per_step (eager, incl. the e2e copies)"}
                del RG, RD
                torch.cuda.empty_cache()
        except Exception as e:
            res['ref_cuda'] = {'unavailable': f'{type(e).__name__}: {e}'}
    if rank == 0 and with_cpu:
        fps, desc, threads, kind = cpu_sample(workload, budget_s=args.cpu_budget)
        res['cpu_baseline'] = {'value': fps, 'unit': 'frames/s', 'cores': threads, 'kind': kind, 'sample': desc}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10,
                    help="timed steps of each of this repository's runs (lres, ops_only, sres); the ref_cuda comparison times 2..5 steps "
                         "and --impl reference samples up to K steps within a ~3-minute guard")
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--workload', default='both', choices=sorted(WORKLOADS) + ['both'],
                    help="both (default): the line's value is the lres step (BASELINE configs[1]); the sres step (configs[2]) is measured in the same run and reported under the key sres")
    ap.add_argument('--scope', default='full', choices=['full', 'ops'],
                    help='full (default): the F.conv3d / F.conv1d calls of the low-res networks are part of the replayed step (on the tensor-core engine); '
                         'ops: only the torch_utils.ops calls (the round-1 metric; also reported under ops_only in the default run)')
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--cpu-budget', type=float, default=4.0,
                    help='seconds of CPU sampling before every (network, op) group has been visited once (the whole sample takes ~30 s at 4: '
                         'every group is measured at least once; 12 gave 125 s on the 128-thread host of the B200 box)')
    ap.add_argument('--no-cpu', action='store_true')
    ap.add_argument('--no-ref-cuda', action='store_true')
    ap.add_argument('--launch', default='graph', choices=['graph', 'eager'],
                    help='graph: the step is captured once into CUDA graphs and replayed (default); eager: every call launched from Python')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write a fixed sample of what the last timed step computed (outputs, gradients, optimiser state) as DIR/*.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs needs --impl ours')

    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    local_rank = int(os.environ.get('LOCAL_RANK', 0))
    global _scope
    primary = 'lres' if args.workload == 'both' else args.workload
    _scope = args.scope
    metric = metric_name(args.scope)

    if args.impl == 'reference':
        # the reference's own CPU implementation of the path on the box's host cores (rank 0 only; all host threads)
        if rank != 0:
            return
        _, _, batch, frames = load_trace(primary)
        steps = max(1, args.steps)
        # the whole arm stays within ~3 minutes whatever K is: the per-step sample budget shrinks with K, and a wall-clock guard
        # stops sampling early (host contention can stretch a single CPU call far beyond its share of the budget)
        t_arm = time.perf_counter()
        budget = max(2.0, min(args.cpu_budget, 150.0 / (steps + 1)))
        for _ in range(max(0, min(args.warmup, 1))):
            cpu_sample(primary, budget_s=min(budget, 4.0))
        vals = []
        for _ in range(steps):
            fps, desc, threads, kind = cpu_sample(primary, budget_s=budget)
            vals.append(fps)
            if time.perf_counter() - t_arm > 170.0:
                desc += f' [time guard: {len(vals)} of {steps} steps sampled]'
                break
        v = float(np.mean(vals))
        what = ('convolutions + torch_utils.ops calls of G+D update' if args.scope == 'full' else 'torch_utils.ops calls of G+D update')
        config = {'workload': f'{primary}: train_{primary} op trace ({what}), per-GPU batch {batch}, '
                              f'{frames} frames/sample, {"64x36" if primary == "lres" else "256x144 from 64x36"}',
                  'global_batch': batch, 'parallelism': 'cpu'}
        print(json.dumps({'impl': 'reference', 'metric': metric, 'value': v, 'unit': 'frames/s', 'n_gpus': args.gpus, 'steps': steps,
                          'warmup': args.warmup, 'ms_per_step': 1000.0 * frames / v, 'higher_is_better': True, 'scaling': 'weak',
                          'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic', 'config': config,
                          'cpu_baseline': {'value': v, 'unit': 'frames/s', 'cores': threads, 'kind': kind, 'sample': desc},
                          'e2e': {'value': v, 'unit': 'frames/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}))
        return

    assert torch.cuda.is_available(), 'bench.py needs a CUDA device (the ops have no CPU fallback for the product path)'
    torch.cuda.set_device(local_rank)
    device = torch.device('cuda', local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group('nccl', device_id=device)
    from torch_utils import custom_ops
    custom_ops.load_library()

    dump = {} if args.dump_outputs else None
    res = run_ours(args, primary, args.scope, args.steps, rank, world, local_rank, device, with_cpu=not args.no_cpu, with_refcuda=not args.no_ref_cuda,
                   dump=dump)
    sres = ops_only = None
    if args.workload == 'both':
        torch.cuda.empty_cache()
        if args.scope == 'full':
            ops_only = run_ours(args, primary, 'ops', args.steps, rank, world, local_rank, device, with_cpu=False, with_refcuda=not args.no_ref_cuda,
                                dump=dump)
            torch.cuda.empty_cache()
        sres = run_ours(args, 'sres', 'ops', args.steps, rank, world, local_rank, device, with_cpu=False, with_refcuda=not args.no_ref_cuda,
                        dump=dump)
    if dump is not None and rank == 0:
        nbytes = sum(a.nbytes for a in dump.values())
        assert nbytes <= 64 << 20, f'--dump-outputs: {nbytes} bytes of samples, more than 64 MB'
        os.makedirs(args.dump_outputs, exist_ok=True)
        for k, a in dump.items():
            np.save(os.path.join(args.dump_outputs, k + '.npy'), a)
    if rank == 0:
        out = {'metric': metric, 'value': res['value'], 'unit': 'frames/s', 'n_gpus': world, 'steps': args.steps, 'warmup': res['warmup'],
               'ms_per_step': res['ms_per_step'], 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
               'dtype': res['dtype'], 'data': 'synthetic'}
        for k in ('config', 'gpu_launches', 'e2e', 'roofline', 'clocks', 'ref_cuda', 'cpu_baseline'):
            if k in res:
                out[k] = res[k]
        if ops_only is not None:
            out['ops_only'] = {k: ops_only[k] for k in ('metric', 'value', 'unit', 'steps', 'ms_per_step', 'gpu_launches', 'e2e', 'roofline', 'ref_cuda') if k in ops_only}
        if sres is not None:
            out['sres'] = {k: sres[k] for k in ('value', 'unit', 'steps', 'warmup', 'ms_per_step', 'dtype', 'config', 'gpu_launches', 'e2e',
                                                'roofline', 'ref_cuda') if k in sres}
        print(json.dumps(out))
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
