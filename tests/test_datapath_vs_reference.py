"""The data / checkpoint / helper mirrors (geniconet_b200/data.py, checkpoint.py, ico_utils.py) against what the original
project's own data.py, run.py, ico_utils.py and generate.py return on the same seeded inputs, stored in
tests/golden/reference_vectors.json (tests/golden/make_reference_vectors.py)."""
import json
import os

import numpy as np
import pytest
import torch

from geniconet_b200 import checkpoint as ck
from geniconet_b200 import data as gd
from geniconet_b200 import models as gm
from golden.make_reference_vectors import BEST_LOSSES, NORMALS_LEVEL, NORMALS_SAMPLE, POLE_SEED, digest
from test_datapath import LEVEL, N, P, _make_modelnet, _params

GOLD = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'reference_vectors.json')))


def test_datasets_match_reference_data_py(tmp_path):
    root = str(tmp_path)
    _make_modelnet(root)                                   # chair/bed x train/test, names that need natural ordering
    want = GOLD['data']
    for process in ('train', 'test'):
        params = _params(root, process=process)
        for inst in ('trn', 'val'):
            assert digest(gd.listFiles(params, 'ico', inst), root) == want[process]['listFiles'][inst]
        f0 = gd.listFiles(params, 'ico', 'trn')[0]
        assert digest(gd.loadIcoFile(params, f0), root) == want[process]['loadIcoFile']
        for cls in ('createico2icoDataset', 'createico2ico_vaeDataset'):
            ours = getattr(gd, cls)(params, 'val')
            assert len(ours) == len(want[process][cls]) == 6
            for i in range(len(ours)):
                assert digest(ours[i], root) == want[process][cls][i], (cls, process, i)
    # encodings: written with the original's save_to_file convention ('arr_0'), read back
    params = _params(root, process='test')
    enc = gd.createico2encDataset(params, 'val')
    assert [digest(enc[i], root) for i in range(len(enc))] == want['createico2encDataset']
    for i in range(len(enc)):
        np.savez_compressed(enc[i][1], np.full((2, 3), float(i), dtype=np.float32))
    assert digest(gd.loadEncFile(params, enc[2][1]), root) == want['loadEncFile']
    flat = dict(params, ico=dict(params['ico'], dataPthLvl=1, dataPth=os.path.join(root, 'ico', 'chair', 'test')))
    dec = gd.createenc2icoDataset(flat, 'val')
    assert len(dec) >= 1 and [digest(dec[i], root) for i in range(len(dec))] == want['createenc2ico_vaeDataset']
    with pytest.raises(ValueError):
        gd.loadEncFile(params, 'x.bin')


def test_pole_rule_matches_reference_ico_utils():
    # the original's pole rule (ico_utils.py:10-24) on the CPU against the plan the CUDA kernel walks (gin_pole_vertices_fwd)
    from geniconet_b200 import _lib
    x = torch.randn(2, 3, 5 * N, 2 * N, generator=torch.Generator().manual_seed(POLE_SEED))
    v_ref = torch.tensor(GOLD['pole']['vertices'])
    blob = _lib.plan_blob(_lib.PLAN_LOSS, LEVEL)
    assert int(blob[3]) == P and int(blob[4]) == P + 2                       # GinLossPlanHdr: magic, kind, level, P, V, total, ring, pole, flag
    ring = np.asarray(blob[int(blob[7]):int(blob[7]) + 10]).reshape(2, 5)    # pole_off: the five pixels averaged into each pole
    flat = x.reshape(2, 3, -1)
    assert tuple(v_ref.shape) == (2, P + 2, 3)
    assert torch.equal(v_ref[:, :P], flat.transpose(1, 2))
    for pole in (0, 1):
        assert torch.allclose(v_ref[:, P + pole], flat[:, :, torch.as_tensor(ring[pole]).long()].mean(-1), atol=1e-7)


def _model(seed):
    torch.manual_seed(seed)
    return gm.ico2ico(gm.default_params('ico2ico'))


def test_checkpoints_interoperate_with_reference_run_py(tmp_path):
    want = GOLD['checkpoint']
    # 1. the files and dict keys the original's saveModel writes, and their values
    p = _params(str(tmp_path / 'a'))
    m0 = _model(0)
    opt0 = torch.optim.Adam(m0.parameters(), lr=1e-3)
    ck.saveModel(p, m0, opt0, 'B4', 'ico2ico', 0.25, {'k': 1})
    files = sorted(os.path.relpath(os.path.join(d, f), p['logDir']) for d, _, fs in os.walk(p['logDir']) for f in fs)
    assert files == want['saveModel_files']
    saved = torch.load(os.path.join(p['logDir'], files[0]), weights_only=False)
    assert sorted(saved) == want['saveModel_keys'] and {k: saved[k] for k in ('epoch', 'loss', 'misc')} == want['saveModel_values']
    # 2. a file with exactly those keys and values (what the original writes) loads into ours
    m1 = _model(1)
    epoch, best, misc = [0], [np.inf], []
    assert ck.loadModel(p, m1, epoch, 'ico2ico', torch.optim.Adam(m1.parameters(), lr=1e-3), best, misc) is True
    assert epoch == [4] and best == [0.25] and misc == [{'k': 1}]
    assert all(torch.equal(a, b) for a, b in zip(m0.state_dict().values(), m1.state_dict().values()))
    assert os.path.basename(p['out']['dataPth']) == want['out_dataPth']
    # 3. the same sequence of validation losses leaves the same files behind (best-model rotation, run.py:317-328)
    pb, bb = _params(str(tmp_path / 'd')), [np.inf]
    for e, loss in enumerate(BEST_LOSSES, start=1):
        ck.saveBestModel(pb, m0, opt0, e, 'ico2ico', bb, [loss])
    assert sorted(os.listdir(os.path.join(pb['logDir'], 'savedModel'))) == want['best_files'] and bb == [want['best_loss']]
    # 4. no file: False; loadMultiModel: raises on a missing file, fills from two checkpoints
    assert ck.loadModel(_params(str(tmp_path / 'e')), m1, [3], 'ico2ico') is False
    ck.saveModel(p, _model(5), opt0, 2, 'other', 0.0, None)
    ma = _model(6)
    assert ck.loadMultiModel(p, ma, ['B4', 2], ['ico2ico', 'other'])
    with pytest.raises(ValueError):
        ck.loadMultiModel(p, ma, [77], ['ico2ico'])


def test_target_normals_against_reference_generate_py():
    """generate.py:20-43 mesh_vertexnormals made the dataset's normal targets.  Its fancy-index `+=` keeps one face per corner slot
    (numpy does not accumulate repeated indices), which data.vertex_normals(reference_semantics=True) reproduces; the
    default (true area-weighted accumulation, what the loss kernels compute for the OUTPUT mesh) differs measurably."""
    want = GOLD['normals']
    verts = gd.synthetic_mesh(NORMALS_LEVEL, NORMALS_SAMPLE)[1][:3].T.numpy().astype(np.float64)
    faces = gd._topology(NORMALS_LEVEL)[1]
    n_ref, c_ref, s_ref = np.asarray(want['normals']), np.asarray(want['center']), want['scale']
    assert n_ref.shape == (10 * 4 ** NORMALS_LEVEL + 2, 3)
    assert np.allclose(gd.vertex_normals(verts, faces, reference_semantics=True), n_ref, rtol=0, atol=1e-12)
    n_true = gd.vertex_normals(verts, faces)
    angle = np.degrees(np.arccos(np.clip((n_ref * n_true).sum(1), -1.0, 1.0)))
    assert 0.5 < angle.mean() < 10.0 and np.allclose(np.linalg.norm(n_true, axis=1), 1.0)
    assert np.allclose(c_ref, verts.mean(0)) and np.isclose(s_ref, np.linalg.norm(verts - verts.mean(0), axis=1).max())
