"""ORACLE (test infrastructure, NOT product code) -- the normal and Laplacian terms of the Chamfer loss on the CPU, float64, given
the nearest-neighbour indices (the product kernels: geniconet_b200/csrc/gin_chamfer_terms.cuh).  Built on mesh_ref's
compute_vertex_normals and compute_laplacian_batch; the reference gradient is autograd through this restatement.
"""
_mesh_cache = {}


def _mesh(level):
    if level not in _mesh_cache:
        import torch
        from . import ico_geometry_ref as geo, mesh_ref
        faces = torch.from_numpy(geo.get_ico_faces(level))
        _mesh_cache[level] = (faces, mesh_ref.compute_adjacency_matrix_sparse(int(faces.max()) + 1, faces))
    return _mesh_cache[level]


def chamfer_terms(level, v, tn, tl, idx_xy, idx_yx, cos_eps=1e-8):
    """(nor_xy, nor_yx, lap_xy, lap_yx) as float64 torch scalars, differentiable in v [B,V,3] (float64 torch; the level-`level` output
    vertices).  n, L are mesh_ref.compute_vertex_normals / compute_laplacian_batch of v; tn, tl [B,M,3] the target's normals and
    Laplacians (None: those terms are 0); idx_xy [B,V], idx_yx [B,M] the nearest-neighbour indices (None: that direction is 0):

        nor_xy = mean_{b,i} (1 - cos(n_i, tn_{i_xy(i)}))        nor_yx = mean_{b,j} (1 - cos(tn_j, n_{i_yx(j)}))
        lap_xy = mean_{b,i,c} (L_i - tl_{i_xy(i)})_c^2           lap_yx = mean_{b,j,c} (tl_j - L_{i_yx(j)})_c^2

    with cos(a, b) = a.b / (max(|a|, eps) max(|b|, eps)) as in Point2Point_Loss."""
    import torch
    from . import mesh_ref
    faces, adj = _mesh(level)
    zero = v.new_zeros(())
    n = mesh_ref.compute_vertex_normals(v, faces) if tn is not None else None
    lap = mesh_ref.compute_laplacian_batch(v, adj) if tl is not None else None

    def gather(a, idx):
        return torch.gather(a, 1, torch.as_tensor(idx, dtype=torch.int64, device=a.device)[..., None].expand(-1, -1, 3))

    def one_minus_cos(a, b):
        return 1 - (a * b).sum(-1) / (a.norm(dim=-1).clamp_min(cos_eps) * b.norm(dim=-1).clamp_min(cos_eps))

    out = [zero, zero, zero, zero]
    for d, idx in ((0, idx_xy), (1, idx_yx)):
        if idx is None:
            continue
        if tn is not None:
            a, b = (n, gather(tn, idx)) if d == 0 else (tn, gather(n, idx))
            out[d] = one_minus_cos(a, b).mean()
        if tl is not None:
            a, b = (lap, gather(tl, idx)) if d == 0 else (tl, gather(lap, idx))
            out[2 + d] = ((a - b) ** 2).mean()
    return tuple(out)
