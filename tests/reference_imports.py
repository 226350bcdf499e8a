"""Test infrastructure: import modules of a checkout of the original GenIcoNet project UNCHANGED, with stand-ins for its
third-party packages.  The checkout is not part of this repository: the tests that need it run when the environment variable
GENICONET_REFERENCE names its directory and skip otherwise.  Nothing under geniconet_b200/ imports this.

Stand-ins (each only as far as the imported reference code touches it):
  natsort.natsorted      digit runs compare as integers (natsort's default algorithm), written independently of
                         geniconet_b200.data.natural_key
  kaolin, matplotlib.pyplot, torch_utils, python_utils, torchsummary      empty modules / no-op plotting
  icocnn, mesh           the oracle (oracle/install.py)
  numpy.Inf              removed in numpy 2; run.py:342 uses it as a default argument
"""
import contextlib
import importlib.util
import os
import re
import sys
import types

REF_ROOT = os.environ.get('GENICONET_REFERENCE', '')
SKIP_REASON = 'needs a checkout of the original GenIcoNet project (GENICONET_REFERENCE)'


def available():
    return bool(REF_ROOT) and os.path.isdir(REF_ROOT)


def _natsorted(seq, key=None):
    def k(v):
        s = key(v) if key else v
        return [(0, int(t), '') if t.isdigit() else (1, 0, t) for t in re.findall(r'\d+|\D+', s)]
    return sorted(seq, key=k)


class _Plot(types.ModuleType):
    def __getattr__(self, name):
        if name.startswith('__'):
            raise AttributeError(name)
        return lambda *a, **k: None


@contextlib.contextmanager
def reference_modules(*names):
    """Yields the imported reference modules (e.g. 'data', 'ico_utils', 'run'); sys.modules and sys.path are restored afterwards."""
    import numpy as np
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    from oracle.install import install_oracle_modules
    touched = ['natsort', 'kaolin', 'matplotlib', 'matplotlib.pyplot', 'torch_utils', 'python_utils', 'torchsummary',
               'ico_utils', 'data', 'losses', 'models', 'run', 'generate']
    before = {k: sys.modules.get(k) for k in touched}
    saved_oracle = install_oracle_modules()
    had_inf = hasattr(np, 'Inf')
    try:
        nat = types.ModuleType('natsort'); nat.natsorted = _natsorted
        mpl = types.ModuleType('matplotlib'); mpl.__path__ = []
        mpl.pyplot = _Plot('matplotlib.pyplot'); mpl.use = lambda *a, **k: None
        stubs = {'natsort': nat, 'kaolin': types.ModuleType('kaolin'), 'matplotlib': mpl, 'matplotlib.pyplot': mpl.pyplot,
                 'torch_utils': types.ModuleType('torch_utils'), 'python_utils': types.ModuleType('python_utils'),
                 'torchsummary': types.ModuleType('torchsummary')}
        stubs['kaolin'].__version__ = 'absent'
        for k, v in stubs.items():
            if before[k] is None:
                sys.modules[k] = v
        if not had_inf:
            np.Inf = np.inf
        sys.path.insert(0, REF_ROOT)
        cwd = os.getcwd()
        os.chdir(REF_ROOT)                      # models.py:4 appends '../IcosahedralCNN/' relative to the CWD
        try:
            mods = []
            for n in names:
                spec = importlib.util.spec_from_file_location(n, os.path.join(REF_ROOT, n + '.py'))
                m = importlib.util.module_from_spec(spec)
                sys.modules[n] = m
                spec.loader.exec_module(m)
                mods.append(m)
        finally:
            os.chdir(cwd)
        yield mods[0] if len(mods) == 1 else mods
    finally:
        from oracle.install import restore_modules
        restore_modules(saved_oracle)
        for k, v in before.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
        while REF_ROOT in sys.path:
            sys.path.remove(REF_ROOT)
        if not had_inf and hasattr(np, 'Inf'):
            del np.Inf
