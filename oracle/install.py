"""ORACLE (test infrastructure): expose the CPU restatement under the module names the
reference imports (icocnn.ico_conv, icocnn.utils.ico_geometry, mesh.utils) so that the
original project's models.py and losses.py can be imported UNCHANGED on top of it
(only where a checkout of it is given by the environment variable GENICONET_REFERENCE).
"""
import importlib
import sys
import types


def install_oracle_modules():
    """Bind the oracle under the reference's import names; returns the previous bindings."""
    from . import ico_geometry_ref, icocnn_ref, mesh_ref
    saved = {k: sys.modules.get(k) for k in
             ('icocnn', 'icocnn.ico_conv', 'icocnn.utils', 'icocnn.utils.ico_geometry', 'mesh', 'mesh.utils')}
    icocnn = types.ModuleType('icocnn'); icocnn.__path__ = []
    utils = types.ModuleType('icocnn.utils'); utils.__path__ = []
    icocnn.ico_conv = icocnn_ref
    icocnn.utils = utils
    utils.ico_geometry = ico_geometry_ref
    mesh = types.ModuleType('mesh'); mesh.__path__ = []
    mesh.utils = mesh_ref
    sys.modules.update({'icocnn': icocnn, 'icocnn.ico_conv': icocnn_ref, 'icocnn.utils': utils,
                        'icocnn.utils.ico_geometry': ico_geometry_ref, 'mesh': mesh, 'mesh.utils': mesh_ref})
    return saved


def restore_modules(saved):
    for k, v in saved.items():
        if v is None:
            sys.modules.pop(k, None)
        else:
            sys.modules[k] = v


def import_reference(name, ref_root=None):
    """Import <ref_root>/<name>.py (models / losses; default root: $GENICONET_REFERENCE) over the oracle modules."""
    import importlib.util
    import os
    ref_root = ref_root or os.environ.get('GENICONET_REFERENCE')
    if not ref_root:
        raise RuntimeError('import_reference: no checkout of the original project given (ref_root or GENICONET_REFERENCE)')
    path = os.path.join(ref_root, name + '.py')
    if not os.path.exists(path):
        raise FileNotFoundError(path)
    saved = install_oracle_modules()
    try:
        spec = importlib.util.spec_from_file_location('_reference_' + name, path)
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
    finally:
        restore_modules(saved)
    return mod
