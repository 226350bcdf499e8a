"""The ico2ico / ico2ico_vae encoder-decoders of the reference, assembled over the CUDA layers.

Mirrors the module surface of /root/reference/models.py (class names, constructor arguments,
attribute names and therefore state-dict keys) so a reference user can switch imports:

    IcoUpS2S (models.py:9-20)            BasicIcoS2SDownBlock (:22-40)   BasicIcoS2SUpBlock (:42-62)
    Identity (:64-73)                    VAE (:75-97)
    createico2enc / createenc2ico (:101-160)   createico2enc_vae / createenc2ico_vae (:162-216)
    ico2ico (:219-232)  ico2enc (:234-241)  enc2ico (:243-252)
    ico2ico_vae (:254-300)  ico2enc_vae (:302-320)  enc2ico_vae (:322-340)

The reference hard-codes subdivision 5; here the graphs take the top level as an argument
(default 5) so the I6 configuration of BASELINE.json is the same code with levels shifted by one.
The unmodified reference file also runs on these layers (through the `icocnn` shim package).
"""
import torch

import os

from . import fused as _fused
from .ico_conv import IcoConvS2S, IcoUpsampleS2S
from .reparam import reparameterize as _reparameterize

# Fused execution of the encoder / decoder bodies (geniconet_b200/fused.py) in training mode; GIN_FUSED=0 or
# set_fused(False) runs every module on its own, exactly as the unmodified reference models.py does.
_FUSED = os.environ.get('GIN_FUSED', '1') != '0'
_HEAD = os.environ.get('GIN_HEAD', '1') != '0'           # the decoder head through gin_head_* (A/B: GIN_HEAD=0 keeps Conv2d + Tanh)
# Forward-only fused chains (fused.infer_chain) when grad is disabled (no_grad / inference_mode); opt-in: GIN_FUSED_INFER=1 or
# set_fused(True, inference=True).
_INFER = os.environ.get('GIN_FUSED_INFER', '0') == '1'
# Fused chains with every BatchNorm in eval mode and grad enabled (fused.run_frozen_chain: frozen-statistics fine-tuning, latent
# fitting, input gradients); opt-in: GIN_FUSED_FROZEN=1 or set_fused(True, frozen=True).
_FROZEN = os.environ.get('GIN_FUSED_FROZEN', '0') == '1'


def set_fused(flag, head=None, inference=None, frozen=None):
    global _FUSED, _HEAD, _INFER, _FROZEN
    _FUSED = bool(flag)
    if head is not None:
        _HEAD = bool(head)
    if inference is not None:
        _INFER = bool(inference)
    if frozen is not None:
        _FROZEN = bool(frozen)


def _bn_modes(tops):
    """The set of `training` flags of every BatchNorm2d or SyncBatchNorm inside the modules `tops`."""
    return {m.training for t in tops for m in t.modules() if isinstance(m, _fused._BN)}


def _route(mods, x, train_chain=True):
    """Which fused chain runs `mods` (a Sequential, whose own hooks count too, or a list of modules) on x: 'infer' (fused.infer_chain),
    'train' (fused.run_chain), 'frozen' (fused.run_frozen_chain), or None (the caller runs the modules).  A chain needs a CUDA fp32 x,
    no forward (pre-)hook and no `impl` override inside, a supported module list, and every BatchNorm inside in the same mode.  With
    grad disabled that is the forward-only chain (when switched on); with grad enabled the BatchNorms decide: train mode -> the
    training chain (unless train_chain is False: the split models never take it), eval mode -> the frozen chain (when switched on).
    SyncBatchNorm counts as BatchNorm; the training chain then synchronises the batch statistics (fused.sync_group)."""
    tops = [mods] if isinstance(mods, torch.nn.Module) else list(mods)
    mods = list(mods)
    if not (_FUSED and x.is_cuda and x.dtype == torch.float32):
        return None
    inner = [m for t in tops for m in t.modules()]
    if any(m._forward_hooks or m._forward_pre_hooks or (isinstance(m, IcoConvS2S) and getattr(m, 'impl', 0) != 0) for m in inner):
        return None
    modes = _bn_modes(tops)
    if not torch.is_grad_enabled():
        # train-mode SyncBatchNorm that synchronises keeps the module path: the forward-only chain has no exchange
        ok = _INFER and len(modes) == 1 and _fused.chain_supported(mods) and (modes == {False} or _fused.sync_group(mods) is None)
        return 'infer' if ok else None
    if modes == {True}:
        return 'train' if train_chain and _fused.chain_supported(mods) else None
    return 'frozen' if _FROZEN and modes == {False} and _fused.frozen_supported(mods) else None


def _apply(route, mods, x):
    """`mods` on x through the fused chain `route` (see _route), or for None through the modules themselves: a Sequential is
    called, a list runs in order."""
    if route is None:
        if isinstance(mods, torch.nn.Module):
            return mods(x)
        for m in mods:
            x = m(x)
        return x
    mods = list(mods)
    if route == 'infer':
        return _fused.infer_chain(x, mods)[0]
    return (_fused.run_chain if route == 'train' else _fused.run_frozen_chain)(x, mods)


def _run(mods, x):
    """nn.Sequential semantics over the module list, through a fused chain when one applies (_route)."""
    mods = list(mods)
    return _apply(_route(mods, x), mods, x)


def _body(seq, x):
    """A split model's body `seq` (a Sequential) on x: through the forward-only or the frozen chain where one applies, else module by
    module (the split models never take the training chain)."""
    return _apply(_route(seq, x, train_chain=False), seq, x)


def _infer_encode(encoder, mu, logvar, x):
    """A VAE encoder body on the forward-only chain: (its output map, (mu, logvar) or None).  The mu and logvar heads run as ONE GEMM
    on the body's operand copy (fused.infer_latent) where that is supported; None: the caller runs them."""
    h, h_b = _fused.infer_chain(x, list(encoder), want_operand=True)
    return h, (_fused.infer_latent(h_b, mu, logvar, x.shape[0]) if _fused.latent_supported(mu, logvar) else None)


BatchNorm2d = torch.nn.BatchNorm2d


class IcoUpS2S(torch.nn.Module):
    def __init__(self, in_features, out_features, bias=True, subdivisions=0, corner_mode='zeros'):
        super().__init__()
        self.up = IcoUpsampleS2S(in_features, subdivisions, corner_mode)
        self.conv = IcoConvS2S(in_features, out_features, 1, bias, subdivisions + 1, corner_mode=corner_mode)

    def forward(self, x):
        return self.conv(self.up(x))


class _ResidualBlock(torch.nn.Module):
    """Two-branch residual block: main = conv00-bn-relu-conv01-bn, skip = conv10-bn, out = relu(main+skip).

    `resample` is 'down' (conv00/conv10 have stride 2) or 'up' (an IcoUpsampleS2S precedes conv00/conv10).
    """

    def __init__(self, in_features, out_features, bias, in_subdivisions, corner_mode, resample):
        super().__init__()
        down = resample == 'down'
        lvl = in_subdivisions - 1 if down else in_subdivisions + 1
        first = dict(in_features=in_features, out_features=out_features, stride=2 if down else 1, bias=bias,
                     subdivisions=in_subdivisions if down else lvl, corner_mode=corner_mode)
        if not down:
            self.upsample00 = IcoUpsampleS2S(in_features, in_subdivisions, corner_mode)
        self.conv00 = IcoConvS2S(**first)
        self.icobn00 = BatchNorm2d(out_features)
        self.conv01 = IcoConvS2S(in_features=out_features, out_features=out_features, stride=1, bias=bias,
                                 subdivisions=lvl, corner_mode=corner_mode)
        self.icobn01 = BatchNorm2d(out_features)
        if not down:
            self.upsample10 = IcoUpsampleS2S(in_features, in_subdivisions, corner_mode)
        self.conv10 = IcoConvS2S(**first)
        self.icobn10 = BatchNorm2d(out_features)
        self._down = down

    def forward(self, x):
        relu = torch.nn.functional.relu
        a = x if self._down else self.upsample00(x)
        b = x if self._down else self.upsample10(x)
        main = self.icobn01(self.conv01(relu(self.icobn00(self.conv00(a)))))
        skip = self.icobn10(self.conv10(b))
        return relu(main + skip)


def _head(head, x):
    """The decoder head `Conv2d(64,3,1) -> Tanh` (models.py:151-154): one kernel each way instead of the stock modules."""
    if _FUSED and _HEAD and isinstance(head, torch.nn.Sequential) and _fused.head_supported(head, x):
        return _fused.run_head(head, x)
    return head(x)


class BasicIcoS2SDownBlock(_ResidualBlock):
    def __init__(self, in_features, out_features, bias, in_subdivisions, corner_mode):
        super().__init__(in_features, out_features, bias, in_subdivisions, corner_mode, 'down')


class BasicIcoS2SUpBlock(_ResidualBlock):
    def __init__(self, in_features, out_features, bias, in_subdivisions, corner_mode):
        super().__init__(in_features, out_features, bias, in_subdivisions, corner_mode, 'up')


class Identity(torch.nn.Module):
    """Debug network of the reference (models.py:64-73): x + (W - W)."""

    def __init__(self, subdivisions=5):
        super().__init__()
        n = 2 ** subdivisions
        self.W = torch.nn.Parameter(torch.randn(1, 3, 5 * n, 2 * n))

    def forward(self, x):
        w = self.W.expand(x.size(0), -1, -1, -1)
        return x + (w - w)


class VAE(torch.nn.Module):
    def __init__(self):
        super().__init__()
        self.encoder = self.mu = self.logvar = self.decoder = None

    def encode(self, input):
        raise NotImplementedError

    def decode(self, input):
        raise NotImplementedError

    def reparameterize(self, mu, logvar):
        return _reparameterize(mu, logvar)

    def forward(self, x):
        mu, logvar = self.encode(x)
        return self.decode(self.reparameterize(mu, logvar)), mu, logvar


# ------------------------------------------------------------------ graph factories
_ENC_WIDTHS = {'ae': (64, 128, 256, 256), 'vae': (64, 128, 256)}
_DEC_WIDTHS = {'ae': (256, 256, 128, 64), 'vae': (512, 256, 128, 64)}


def _encoder(kind, corner_mode, model, top):
    if model == 'identity':
        return torch.nn.Sequential(Identity(top))
    if model != 'residualS2S':
        raise ValueError('unknown model %r' % (model,))
    w = _ENC_WIDTHS[kind]
    layers = [IcoConvS2S(in_features=3, out_features=w[0], stride=1, bias=True, subdivisions=top, corner_mode=corner_mode),
              BatchNorm2d(w[0]), torch.nn.ReLU(inplace=False)]
    for d in range(len(w) - 1):
        layers.append(BasicIcoS2SDownBlock(in_features=w[d], out_features=w[d + 1], bias=True, in_subdivisions=top - d,
                                           corner_mode=corner_mode))
    return torch.nn.Sequential(*layers)


def _decoder(kind, corner_mode, model, top):
    if model == 'identity':
        return torch.nn.Sequential(Identity(top)), torch.nn.Sequential(torch.nn.Identity())
    if model != 'residualS2S':
        raise ValueError('unknown model %r' % (model,))
    w = _DEC_WIDTHS[kind]
    blocks = [BasicIcoS2SUpBlock(in_features=w[d], out_features=w[d + 1], bias=True, in_subdivisions=top - 3 + d,
                                 corner_mode=corner_mode) for d in range(3)]
    head = torch.nn.Sequential(torch.nn.Conv2d(in_channels=w[3], out_channels=3, kernel_size=(1, 1)), torch.nn.Tanh())
    return torch.nn.Sequential(*blocks), head


def createico2enc(corner_mode='average', model='simple', subdivisions=5):
    return _encoder('ae', corner_mode, model, subdivisions)


def createenc2ico(corner_mode='average', model='simple', subdivisions=5):
    return _decoder('ae', corner_mode, model, subdivisions)


def createico2enc_vae(corner_mode='average', model='simple', subdivisions=5):
    return _encoder('vae', corner_mode, model, subdivisions)


def createenc2ico_vae(corner_mode='average', model='simple', subdivisions=5):
    return _decoder('vae', corner_mode, model, subdivisions)


def _top(params):
    return int(params['ico'].get('subdivisions', 5))


class ico2ico(torch.nn.Module):
    def __init__(self, params):
        super().__init__()
        self.subdivisions = _top(params)
        self.encoder = createico2enc(params['ico']['corner_mode'], params['ico2ico']['model'], self.subdivisions)
        self.enc = torch.nn.Identity()
        self.decoder, self.enc2icoConv = createenc2ico(params['ico']['corner_mode'], params['ico2ico']['model'], self.subdivisions)

    def forward(self, x):
        whole = list(self.encoder) + list(self.decoder)
        # one fused chain through both halves, unless grad is enabled and the halves differ in BatchNorm mode (e.g. a frozen encoder
        # under a trained decoder): then each half is a chain of its own
        if isinstance(self.enc, torch.nn.Identity) and not self.enc._forward_hooks and (not torch.is_grad_enabled() or len(_bn_modes(whole)) < 2):
            return _head(self.enc2icoConv, _run(whole, x))
        return _head(self.enc2icoConv, _run(self.decoder, self.enc(_run(self.encoder, x))))


class ico2enc(torch.nn.Module):
    def __init__(self, params):
        super().__init__()
        self.encoder = createico2enc(params['ico']['corner_mode'], params['ico2ico']['model'], _top(params))

    def forward(self, x):
        return _body(self.encoder, x)


class enc2ico(torch.nn.Module):
    def __init__(self, params):
        super().__init__()
        self.subdivisions = _top(params)
        self.decoder, self.enc2icoConv = createenc2ico(params['ico']['corner_mode'], params['ico2ico']['model'], self.subdivisions)

    def forward(self, x):
        return _head(self.enc2icoConv, _body(self.decoder, x))


def _latent_head(params, level):
    return torch.nn.Sequential(IcoConvS2S(in_features=256, out_features=512, stride=2, bias=True, subdivisions=level,
                                          corner_mode=params['ico']['corner_mode']),
                               BatchNorm2d(512))


class ico2ico_vae(VAE):
    def __init__(self, params):
        super().__init__()
        self.params = params
        self.model = params[params['model_name']]['model']
        self.subdivisions = _top(params)
        self.encoder = createico2enc_vae(params['ico']['corner_mode'], self.model, self.subdivisions)
        self.mu = self.createMu()
        self.logvar = self.createLogvar()
        self.mu_hook = torch.nn.Identity()
        self.logvar_hook = torch.nn.Identity()
        self.reparameterize_hook = torch.nn.Identity()
        self.decoder, self.final_layer = createenc2ico_vae(params['ico']['corner_mode'], self.model, self.subdivisions)

    def createMu(self):
        return _latent_head(self.params, _top(self.params) - 2)

    def createLogvar(self):
        return _latent_head(self.params, _top(self.params) - 2)

    def encode(self, input):
        mods = list(self.encoder)
        route = _route(mods, input)
        if route == 'infer':
            h, lat = _infer_encode(mods, self.mu, self.logvar, input)
            if lat is not None:
                return self.mu_hook(lat[0]), self.logvar_hook(lat[1])
        else:
            h = _apply(route, mods, input)
        return self.mu_hook(self.mu(h)), self.logvar_hook(self.logvar(h))

    def decode(self, z):
        return _head(self.final_layer, _run(self.decoder, self.reparameterize_hook(z)))


class ico2enc_vae(VAE):
    def __init__(self, params):
        super().__init__()
        self.params = params
        self.model = params[params['model_name']]['model']
        self.encoder = createico2enc_vae(params['ico']['corner_mode'], self.model, _top(params))
        self.mu = _latent_head(params, _top(params) - 2)
        self.logvar = _latent_head(params, _top(params) - 2)

    def encode(self, input):
        route = _route(self.encoder, input, train_chain=False)
        if route == 'infer':
            h, lat = _infer_encode(self.encoder, self.mu, self.logvar, input)
            if lat is not None:
                return lat
        else:
            h = _apply(route, self.encoder, input)
        return self.mu(h), self.logvar(h)

    def forward(self, x):
        return self.encode(x)


class enc2ico_vae(VAE):
    def __init__(self, params):
        super().__init__()
        self.params = params
        self.model = params[params['model_name']]['model']
        self.subdivisions = _top(params)
        self.decoder, self.final_layer = createenc2ico_vae(params['ico']['corner_mode'], self.model, self.subdivisions)

    def createSample(self, batch_size, misc):
        trn_mean, trn_logvar = misc[0]['trn_mean'], misc[0]['trn_logvar']
        return torch.add(trn_mean, trn_logvar * torch.randn(trn_logvar.shape))

    def decode(self, z):
        return _head(self.final_layer, _body(self.decoder, z))

    def forward(self, x):
        return self.decode(x), torch.tensor([]), torch.tensor([])


def default_params(model_name='ico2ico', subdivisions=5, corner_mode='average'):
    """The slice of run.py's params dict (run.py:616-697) the model constructors and losses read."""
    p = {'model_name': model_name,
         'ico': {'corner_mode': corner_mode, 'subdivisions': subdivisions, 'width': 2 ** (subdivisions + 1)},
         'ico2ico': {'model': 'residualS2S', 'loss': 'p2p'},
         'ico2ico_vae': {'model': 'residualS2S', 'loss': 'p2pkld', 'factor_step_size': 25, 'factor_gamma': 0.9}}
    f = {'ico2ico': (1., 0., 0.), 'ico2ico_vae': (0.6, 0.2, 0.2)}[model_name]       # run.py:689-696
    p['ico']['factor_pos'], p['ico']['factor_nor'], p['ico']['factor_lap'] = f
    return p
