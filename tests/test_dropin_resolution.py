"""Drop-in rule (DESIGN.md section 1): with `long-video-gan_b200/` ahead of a LongVideoGAN checkout on PYTHONPATH,
`torch_utils.ops` resolves to this repository while the checkout's other `torch_utils` modules and `dnnlib` still
resolve to the checkout (torch_utils/__init__.py extends the package path). Checked against a minimal stand-in checkout."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, 'long-video-gan_b200')

PROBE = '''
import json
import dnnlib, torch_utils.misc, torch_utils.ops.bias_act, torch_utils.ops.upfirdn2d
print(json.dumps({m.__name__: m.__file__ for m in (dnnlib, torch_utils.misc, torch_utils.ops.bias_act, torch_utils.ops.upfirdn2d)}))
'''


def test_ops_from_here_the_rest_from_the_checkout(tmp_path):
    checkout = tmp_path / 'checkout'
    for rel in ('torch_utils/__init__.py', 'torch_utils/misc.py', 'torch_utils/ops/__init__.py', 'dnnlib/__init__.py'):
        (checkout / rel).parent.mkdir(parents=True, exist_ok=True)
        (checkout / rel).write_text('')
    (checkout / 'torch_utils/ops/bias_act.py').write_text('raise ImportError("the checkout\'s ops must not be imported")\n')
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([PKG, str(checkout)]), CUDA_VISIBLE_DEVICES='')
    r = subprocess.run([sys.executable, '-c', PROBE], env=env, cwd=str(tmp_path), stdout=subprocess.PIPE, stderr=subprocess.STDOUT,
                       text=True, timeout=300)
    assert r.returncode == 0, r.stdout[-3000:]
    where = json.loads(r.stdout.strip().splitlines()[-1])
    assert where['torch_utils.ops.bias_act'].startswith(PKG) and where['torch_utils.ops.upfirdn2d'].startswith(PKG)
    assert where['torch_utils.misc'].startswith(str(checkout)) and where['dnnlib'].startswith(str(checkout))
