"""Generate tests/golden/refcuda_*.npz: the cases of tests/test_gpu_vs_refcuda.py run through the REFERENCE'S OWN CUDA ops
(its three plugins built unmodified for sm_100a into oracle/_ref by build_ref.py, its own Python wrappers) on a B200.
For every output tensor the file keeps its shape, max|ref|, L2 norm and the values at the test's fixed sample positions
(test_gpu_vs_refcuda.summarize), so that the test runs without the reference.

    python oracle/pin_refcuda.py [OUTDIR]        (default tests/golden)
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path[:0] = [os.path.join(ROOT, 'long-video-gan_b200'), ROOT, os.path.join(ROOT, 'tests')]

import test_gpu_vs_refcuda as cases  # noqa: E402
from oracle import ref_cuda  # noqa: E402


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, 'tests', 'golden')
    os.makedirs(out, exist_ok=True)
    ref = ref_cuda.load()
    assert ref.bias_act._init() and ref.upfirdn2d._init() and ref.filtered_lrelu._init()
    assert os.path.join('oracle', '_ref') in ref_cuda.load_plugin('bias_act_plugin').__file__
    for op, runs in cases.golden_cases().items():
        arrays = {}
        for key, run in runs:
            for name, t in run(ref).items():
                for field, v in cases.summarize(t).items():
                    arrays[f'{key}/{name}/{field}'] = v
        path = os.path.join(out, f'refcuda_{op}.npz')
        np.savez_compressed(path, **arrays)
        print(f'{path}: {len(runs)} cases, {os.path.getsize(path)} bytes')


if __name__ == '__main__':
    main()
