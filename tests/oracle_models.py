"""Test tool: the ico2ico / ico2ico_vae graphs over the ORACLE layers (CPU), so model-level parity can be checked without
a checkout of the original project.  A thin adapter over oracle/models_ref.py: nothing here imports the product
package (the CPU arm of bench.py runs through this file and must not load libgeniconet_b200.so)."""
from oracle import models_ref

fill_params_deterministic = models_ref.fill_params_deterministic
ref_p2p_loss = models_ref.p2p_loss
ref_kld = models_ref.kld_loss


def build_oracle_model(name, params=None, level=None):
    """`params` is the slice of run.py's params dict the constructors read (geniconet_b200.models.default_params)."""
    if params is not None:
        level = int(params['ico'].get('subdivisions', 5)) if level is None else level
        corner_mode = params['ico']['corner_mode']
    else:
        level, corner_mode = (5 if level is None else level), 'average'
    return models_ref.build(name, level, corner_mode)
