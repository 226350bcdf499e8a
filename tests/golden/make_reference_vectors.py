"""Generates tests/golden/reference_vectors.json: what the original GenIcoNet code returns on the seeded inputs of
tests/test_datapath_vs_reference.py and tests/test_models_host.py, so those tests compare without a checkout of it:

    python tests/golden/make_reference_vectors.py

  data        listFiles orders, loadIcoFile and every Dataset item of a synthetic ModelNet tree (data.py), as digests
  checkpoint  the files and dict keys saveModel writes and the best-model rotation of saveBestModel (run.py:317-409)
  pole        output2vertices on a seeded 2x3x(5N)x(2N) input (ico_utils.py:10-24)
  normals     mesh_vertexnormals / get_normalize_unitsphere of synthetic_mesh(3, 5) (generate.py:20-55)
  split_state_dicts   keys and shapes of ico2enc, enc2ico, ico2enc_vae, enc2ico_vae (models.py:234-252,302-340)
  adjacency   shape and non-zeros of the adjacency buffer losses.py:39-40 registers at level 5

The values are recorded through this project's restatements of those functions (geniconet_b200.data, checkpoint and models;
the oracle's pole rings and adjacency), which the suite held identical to the original's own files, imported unchanged, while a
checkout of the original was present.
"""
import hashlib
import json
import os
import sys
import tempfile

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.join(ROOT, 'tests')]

OUT = os.path.join(HERE, 'reference_vectors.json')
POLE_SEED = 0
NORMALS_LEVEL, NORMALS_SAMPLE = 3, 5
BEST_LOSSES = [1.0, 0.9, 0.95, 0.8, 0.7, 0.6, 0.65, 0.5, 0.4, 0.3]


def digest(obj, root):
    """A comparable summary of a Dataset item / loader result: arrays by dtype, shape and a hash of their bytes, paths below
    `root` relative to it."""
    if isinstance(obj, (tuple, list)):
        return [digest(v, root) for v in obj]
    if isinstance(obj, torch.Tensor):
        obj = obj.detach().cpu().numpy()
    if isinstance(obj, np.ndarray):
        a = np.ascontiguousarray(obj)
        return {'dtype': str(a.dtype), 'shape': list(a.shape), 'sha256': hashlib.sha256(a.tobytes()).hexdigest()}
    if isinstance(obj, str):
        return os.path.relpath(obj, root) if obj.startswith(root) else obj
    if isinstance(obj, (np.integer, np.floating)):
        return obj.item()
    return obj


def data_vectors(gd, root):
    from test_datapath import _make_modelnet, _params
    _make_modelnet(root)
    out = {}
    for process in ('train', 'test'):
        params = _params(root, process=process)
        rec = {'listFiles': {inst: digest(gd.listFiles(params, 'ico', inst), root) for inst in ('trn', 'val')}}
        rec['loadIcoFile'] = digest(gd.loadIcoFile(params, gd.listFiles(params, 'ico', 'trn')[0]), root)
        for cls in ('createico2icoDataset', 'createico2ico_vaeDataset'):
            ds = getattr(gd, cls)(params, 'val')
            rec[cls] = [digest(ds[i], root) for i in range(len(ds))]
        out[process] = rec
    params = _params(root, process='test')
    enc = gd.createico2encDataset(params, 'val')
    out['createico2encDataset'] = [digest(enc[i], root) for i in range(len(enc))]
    for i in range(len(enc)):
        np.savez_compressed(enc[i][1], np.full((2, 3), float(i), dtype=np.float32))      # save_to_file's 'arr_0' convention
    out['loadEncFile'] = digest(gd.loadEncFile(params, enc[2][1]), root)
    flat = dict(params, ico=dict(params['ico'], dataPthLvl=1, dataPth=os.path.join(root, 'ico', 'chair', 'test')))
    dec = gd.createenc2icoDataset(flat, 'val')
    out['createenc2ico_vaeDataset'] = [digest(dec[i], root) for i in range(len(dec))]
    return out


def checkpoint_vectors(ck, gm, root):
    from test_datapath import _params

    def listing(params):
        base = params['logDir']
        return sorted(os.path.relpath(os.path.join(d, f), base) for d, _, fs in os.walk(base) for f in fs)
    torch.manual_seed(0)
    m = gm.ico2ico(gm.default_params('ico2ico'))
    opt = torch.optim.Adam(m.parameters(), lr=1e-3)
    p = _params(os.path.join(root, 'save'))
    ck.saveModel(p, m, opt, 'B4', 'ico2ico', 0.25, {'k': 1})
    files = listing(p)
    saved = torch.load(os.path.join(p['logDir'], files[0]), weights_only=False)
    ck.loadModel(p, gm.ico2ico(gm.default_params('ico2ico')), [0], 'ico2ico')          # points params['out'] at the epoch's output
    pb = _params(os.path.join(root, 'best'))
    best = [np.inf]
    for e, loss in enumerate(BEST_LOSSES, start=1):
        ck.saveBestModel(pb, m, opt, e, 'ico2ico', best, [loss])
    return {'saveModel_files': files, 'saveModel_keys': sorted(saved), 'saveModel_values': {k: saved[k] for k in ('epoch', 'loss', 'misc')},
            'out_dataPth': os.path.basename(p['out']['dataPth']),
            'best_files': sorted(os.listdir(os.path.join(pb['logDir'], 'savedModel'))), 'best_loss': best[0]}


def pole_vectors():
    from oracle import ico_geometry_ref as geo
    from test_datapath import LEVEL, N
    x = torch.randn(2, 3, 5 * N, 2 * N, generator=torch.Generator().manual_seed(POLE_SEED))
    flat = x.reshape(2, 3, -1)
    rings = torch.from_numpy(np.asarray(geo.pole_rings(LEVEL))).long()
    poles = torch.stack([flat[:, :, rings[k]].mean(-1) for k in range(2)], 1)
    return {'seed': POLE_SEED, 'vertices': torch.cat([flat.transpose(1, 2), poles], 1).tolist()}


def normals_vectors(gd):
    verts = gd.synthetic_mesh(NORMALS_LEVEL, NORMALS_SAMPLE)[1][:3].T.numpy().astype(np.float64)
    faces = gd._topology(NORMALS_LEVEL)[1]
    c = verts.mean(0)
    return {'level': NORMALS_LEVEL, 'sample': NORMALS_SAMPLE, 'normals': gd.vertex_normals(verts, faces, reference_semantics=True).tolist(),
            'center': c.tolist(), 'scale': float(np.linalg.norm(verts - c, axis=1).max())}


def split_state_dicts(gm):
    out = {}
    for name in ('ico2enc', 'enc2ico', 'ico2enc_vae', 'enc2ico_vae'):
        base = 'ico2ico_vae' if name.endswith('_vae') else 'ico2ico'
        params = gm.default_params(base)
        params['model_name'] = name
        params[name] = dict(params[base])
        out[name] = [[k, list(v.shape)] for k, v in getattr(gm, name)(params).state_dict().items()]
    return out


def adjacency_vectors():
    from oracle import ico_geometry_ref as geo, mesh_ref
    faces = torch.from_numpy(geo.get_ico_faces(5))
    adj = mesh_ref.compute_adjacency_matrix_sparse(int(faces.max()) + 1, faces)
    return {'shape': list(adj.shape), 'nnz': int(adj._nnz()), 'faces_shape': list(faces.shape)}


def build():
    from geniconet_b200 import checkpoint as ck, data as gd, models as gm
    with tempfile.TemporaryDirectory() as tmp:
        root = os.path.realpath(tmp)
        return {'data': data_vectors(gd, os.path.join(root, 'data')), 'checkpoint': checkpoint_vectors(ck, gm, root),
                'pole': pole_vectors(), 'normals': normals_vectors(gd), 'split_state_dicts': split_state_dicts(gm),
                'adjacency': adjacency_vectors()}


if __name__ == '__main__':
    with open(OUT, 'w') as f:
        json.dump(build(), f, indent=0)
    print('wrote', OUT, os.path.getsize(OUT), 'bytes')
