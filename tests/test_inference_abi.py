"""The eval-mode inference entry points reject bad arguments on the host, with a negative status, before any launch."""
from geniconet_b200 import _lib

L = _lib.lib
ARG, UNSUPPORTED = -1, -4


def _affine(**kw):
    a = dict(plan_host=None, plan_dev=None, xb=1, packed=1, scale=1, shift=1, relu_split=0, res=None, ld_res=0, res_fp16=0, split=64,
             out0_b=None, out0_f=1, out1_b=None, out1_f=None, ring=None, B=2, Cin=64, Cout=64)
    a.update(kw)
    return L.gin_hexconv_fwd_affine(*a.values(), None)


def test_affine_rejects_bad_arguments():
    assert L.gin_hexconv_affine_ring_bytes(2, 64) == 2 * 10 * 64 * 4
    assert L.gin_hexconv_affine_ring_bytes(0, 64) == 0
    assert _affine(xb=None) == ARG
    assert _affine(scale=None) == ARG
    assert _affine(B=0) == ARG
    assert _affine(relu_split=65) == ARG
    assert _affine(split=32) == ARG and b'split' in L.gin_last_error()
    assert _affine(split=128) == ARG
    assert _affine(out0_f=None) == ARG                                   # no output at all
    assert _affine(out1_f=1) == ARG                                      # split == Cout has one destination
    assert _affine(Cout=128, out1_f=None) == ARG                         # split < Cout needs a second one
    assert _affine(res=1, ld_res=32) == ARG and b'ld_res' in L.gin_last_error()
    assert _affine(out0_b=1) == ARG and b'ring_ws' in L.gin_last_error()
    assert _affine() == ARG and b'plan' in L.gin_last_error()            # arguments fine: the missing plan is reported


def test_eval_consts_rejects_bad_arguments():
    assert L.gin_bn_eval_consts(None, 0, 64, None) == 0                   # empty table: nothing to do
    assert L.gin_bn_eval_consts(None, 3, 64, None) == ARG
    assert L.gin_bn_eval_consts(1, -1, 64, None) == ARG
    assert L.gin_bn_eval_consts(1, 70000, 64, None) == ARG
    assert L.gin_bn_eval_consts(1, 3, 0, None) == ARG


def test_eval_table_layout():
    """fused._bn_table writes GinBnEvalEntry records: eight pointers, eps, C (72 bytes)."""
    import re
    import os
    src = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'include', 'geniconet_b200.h')).read()
    body = re.search(r'typedef struct \{([^}]*)\} GinBnEvalEntry;', src).group(1)
    fields = re.findall(r'(\w+\*?)\s+(\w+);', body)
    assert [t.endswith('*') for t, _ in fields] == [True] * 8 + [False, False]
    assert [n for _, n in fields][-2:] == ['eps', 'C']
