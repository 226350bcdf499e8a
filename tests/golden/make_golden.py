"""Generates tests/golden/*.json from a checkout of the original GenIcoNet project:

    GENICONET_REFERENCE=<checkout> python tests/golden/make_golden.py

The reference's own models.py and losses.py are imported UNCHANGED on top of the oracle's icocnn / mesh
modules (oracle/install.py); weights are the name-keyed deterministic fill of tests/oracle_models.py, inputs come
from seeded CPU generators.  The stored numbers therefore pin "reference graph + reference loss code over the
oracle layers"; the GPU tests reproduce them through the CUDA path without needing the checkout.
"""
import json
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.join(ROOT, 'tests')]

import oracle_models as om                                   # noqa: E402
from oracle.install import import_reference, install_oracle_modules, restore_modules  # noqa: E402
from oracle import icocnn_ref                                # noqa: E402


def inputs(level, B, seed):
    g = torch.Generator().manual_seed(seed)
    n = 2 ** level
    x = torch.randn(B, 3, 5 * n, 2 * n, generator=g) * 0.3
    tgt = torch.randn(B, 9, 10 * 4 ** level + 2, generator=g) * 0.5
    return x, tgt


def sample(t, k=64):
    f = t.detach().flatten()
    idx = torch.linspace(0, f.numel() - 1, k).long()
    return [float(v) for v in f[idx]]


def params_for(name):
    p = {'ico': {'corner_mode': 'average', 'subdivisions': 5}, 'ico2ico': {'model': 'residualS2S'},
         'ico2ico_vae': {'model': 'residualS2S'}, 'model_name': name}
    return p


def build():
    """The fixture as a dict (needs GENICONET_REFERENCE)."""
    torch.set_num_threads(8)
    models = import_reference('models')
    saved = install_oracle_modules()
    try:
        losses = import_reference('losses')
    finally:
        restore_modules(saved)
    out = {}
    # ---- ico2ico (models.py:219-232) + P2P_Loss (losses.py:121-129), run.py:689-692 factors
    x, tgt = inputs(5, 2, 101)
    m = om.fill_params_deterministic(models.ico2ico(params_for('ico2ico')))
    crit = losses.P2P_Loss(5, 1., 0., 0.)
    y = m(x)
    loss = crit(y, tgt)
    loss.backward()
    out['ico2ico'] = {'input_seed': 101, 'batch': 2, 'loss': loss.item(), 'last_losses': [float(v) for v in crit.get_last_losses()],
                      'output_sample': sample(y), 'output_abs_sum': float(y.abs().sum()),
                      'grad_norms': {k: float(p.grad.norm()) for k, p in m.named_parameters()},
                      'state_dict': {k: list(v.shape) for k, v in m.state_dict().items()}}
    # ---- ico2ico_vae (models.py:254-300) + P2PKLD_Loss (losses.py:131-145), run.py:693-696 factors
    x, tgt = inputs(5, 2, 202)
    mv = om.fill_params_deterministic(models.ico2ico_vae(params_for('ico2ico_vae')))
    critv = losses.P2PKLD_Loss(5, 0.6, 0.2, 0.2, 1.0)
    torch.manual_seed(123)                       # eps = torch.randn_like(std) (models.py:91) on the CPU generator
    rec, mu, lv = mv(x)
    lossv = critv((rec, mu, lv), tgt)
    lossv.backward()
    out['ico2ico_vae'] = {'input_seed': 202, 'batch': 2, 'eps_seed': 123, 'loss': lossv.item(),
                          'last_losses': [float(v) for v in critv.get_last_losses()],
                          'mu_sample': sample(mu), 'logvar_sample': sample(lv), 'output_sample': sample(rec),
                          'grad_norms': {k: float(p.grad.norm()) for k, p in mv.named_parameters()},
                          'state_dict': {k: list(v.shape) for k, v in mv.state_dict().items()}}
    # ---- P2P loss alone with all three terms live
    x, tgt = inputs(3, 3, 303)
    xr = x.clone().requires_grad_(True)
    c3 = losses.P2P_Loss(3, 0.6, 0.2, 0.2)
    l3 = c3(xr, tgt)
    l3.backward()
    out['p2p_level3'] = {'input_seed': 303, 'batch': 3, 'loss': l3.item(), 'last_losses': [float(v) for v in c3.get_last_losses()],
                         'grad_sample': sample(xr.grad), 'grad_norm': float(xr.grad.norm())}
    # ---- single layers of the oracle (drift guard)
    layers = {}
    for (cin, cout, stride, level, cm) in [(3, 8, 1, 2, 'average'), (8, 8, 2, 3, 'average'), (4, 6, 1, 2, 'zeros')]:
        conv = om.fill_params_deterministic(icocnn_ref.IcoConvS2S(cin, cout, stride, True, level, cm), seed=5)
        g = torch.Generator().manual_seed(404)
        n = 2 ** level
        xi = torch.randn(2, cin, 5 * n, 2 * n, generator=g)
        layers['conv_%d_%d_s%d_l%d_%s' % (cin, cout, stride, level, cm)] = {'output_sample': sample(conv(xi)), 'input_seed': 404}
    for (c, level, cm) in [(4, 2, 'average'), (4, 1, 'zeros')]:
        up = icocnn_ref.IcoUpsampleS2S(c, level, cm)
        g = torch.Generator().manual_seed(505)
        n = 2 ** level
        xi = torch.randn(2, c, 5 * n, 2 * n, generator=g)
        layers['up_%d_l%d_%s' % (c, level, cm)] = {'output_sample': sample(up(xi)), 'input_seed': 505}
    out['layers'] = layers
    return out


def main():
    out = build()
    with open(os.path.join(HERE, 'reference_over_oracle.json'), 'w') as f:
        json.dump(out, f, indent=1)
    print('wrote', os.path.join(HERE, 'reference_over_oracle.json'))


if __name__ == '__main__':
    main()
