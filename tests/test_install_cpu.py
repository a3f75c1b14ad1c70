"""`pgpp_b200.install()` -- the advertised drop-in switch -- exercised over a checkout laid out like the reference: model code
(`training/networks.py`) that imports `torch_utils.ops.*` gets this package's modules, `training.networks.modulated_conv2d` is
replaced, and on CPU tensors (reference dispatch rule, opt-in through `cpu_tensors='ref'`) the results reproduce the fixtures the
unmodified reference wrote.  The checkout is a stand-in written by the test: its own op modules and its own modulated_conv2d
raise, so every result has to come from this package.  Runs in a subprocess so the aliasing of `sys.modules` does not leak into
the test session."""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# The reference's import lines (training/networks.py imports the op modules from torch_utils.ops) and two callers written the way
# its layers call the ops (Conv2dLayer.forward: conv2d_resample, then bias_act).
STANDIN_NETWORKS = '''
from torch_utils.ops import conv2d_resample, upfirdn2d, bias_act, fma


def modulated_conv2d(*args, **kwargs):
    raise RuntimeError('the stand-in modulated_conv2d ran: install() did not replace it')


def conv_layer(x, w, f, up, down, padding, flip_weight):
    return conv2d_resample.conv2d_resample(x=x, w=w, f=f, up=up, down=down, padding=padding, flip_weight=flip_weight)


def act_layer(x, b, act, alpha, gain, clamp):
    return bias_act.bias_act(x, b, act=act, alpha=alpha, gain=gain, clamp=clamp)
'''
STANDIN_OP = 'raise ImportError("an op module of the stand-in checkout was imported: install() did not alias it")\n'

SCRIPT = r'''
import os, sys
import numpy as np
import torch
ROOT, STANDIN = sys.argv[1], sys.argv[2]
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'tests'))
from conftest import GOLDEN, load_pkg
from oracle.make_golden import CONV_CASES, MODCONV_CASES
pgpp = load_pkg()
torch.set_num_threads(4)
sys.path.insert(0, STANDIN)
pgpp.install(cpu_tensors='ref')                 # before the model modules are imported
import training.networks as networks            # the checkout's model code
import torch_utils.ops.bias_act as ba, torch_utils.ops.upfirdn2d as up, torch_utils.ops.conv2d_gradfix as cg
import torch_utils.custom_ops as co
for m in (ba, up, cg, co, networks.bias_act, networks.upfirdn2d, networks.conv2d_resample, networks.fma):
    assert m.__name__.startswith('pgpp_b200.'), m.__name__
pgpp.install()                                  # now that training.networks exists: swap its modulated_conv2d
mine = sys.modules['pgpp_b200.training.networks'].modulated_conv2d
assert networks.modulated_conv2d is mine
t = lambda a: torch.from_numpy(np.asarray(a))
opt = lambda v: None if v == 'None' else float(v)
# 1. the reference's modulated_conv2d call signature on CPU tensors reproduces the fixture of the unmodified reference
g = np.load(os.path.join(GOLDEN, 'modulated_conv2d.npz'))
for name, n, ic, oc, k, h, upf, demod, noise_kind, flipw in MODCONV_CASES:
    noise = t(g[f'{name}_noise']) if g[f'{name}_noise'].size else None
    for fused in (True, False):
        y = networks.modulated_conv2d(x=t(g[f'{name}_x']).clone(), weight=t(g[f'{name}_w']), styles=t(g[f'{name}_s']), noise=noise, up=upf,
                                      padding=k // 2, resample_filter=t(g['f']), demodulate=demod, flip_weight=flipw, fused_modconv=fused)
        err = float((y - t(g[f'{name}_y_fused'])).norm() / t(g[f'{name}_y_fused']).norm())
        assert err < 1e-5, (name, fused, err)
# 2. the checkout's layer code calling the aliased ops with their default impl on CPU tensors reproduces the op fixtures
g = np.load(os.path.join(GOLDEN, 'conv2d_resample.npz'))
for name, xs, ws, upf, down, pad, groups, flipw, usef in CONV_CASES:
    if groups != 1:
        continue
    y = networks.conv_layer(t(g[f'{name}_x']), t(g[f'{name}_w']), t(g['f']) if usef else None, upf, down, pad, flipw)
    np.testing.assert_allclose(y.numpy(), g[f'{name}_y'], rtol=1e-5, atol=1e-5, err_msg=name)
g = np.load(os.path.join(GOLDEN, 'bias_act.npz'))
for i in range(len([k for k in g.files if k.endswith('_meta')])):
    act, alpha, gain, clamp = g[f'case{i}_meta']
    y = networks.act_layer(t(g['x']), t(g['b']), str(act), opt(alpha), opt(gain), opt(clamp))
    np.testing.assert_allclose(y.numpy(), g[f'case{i}_y'], rtol=1e-6, atol=1e-6, err_msg=str(act))
# 3. without the opt-in a CPU tensor is refused (no silent path off the kernels)
co.cpu_tensors = 'raise'
try:
    ba.bias_act(torch.zeros(2, 3))
    raise SystemExit('impl=cuda accepted a CPU tensor')
except RuntimeError:
    pass
assert torch.equal(ba.bias_act(torch.ones(2, 3), impl='ref'), torch.ones(2, 3))
print('INSTALL_OK')
'''


def _write_standin(root):
    files = {'torch_utils/__init__.py': '', 'torch_utils/ops/__init__.py': '', 'torch_utils/custom_ops.py': STANDIN_OP,
             'training/__init__.py': '', 'training/networks.py': STANDIN_NETWORKS}
    for name in ('bias_act', 'upfirdn2d', 'conv2d_gradfix', 'conv2d_resample', 'fma', 'grid_sample_gradfix'):
        files[f'torch_utils/ops/{name}.py'] = STANDIN_OP
    for rel, text in files.items():
        path = root / rel
        path.parent.mkdir(parents=True, exist_ok=True)
        path.write_text(text)


def test_install_over_a_checkout_with_the_reference_layout(tmp_path):
    _write_standin(tmp_path)
    r = subprocess.run([sys.executable, '-c', SCRIPT, ROOT, str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and 'INSTALL_OK' in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]
