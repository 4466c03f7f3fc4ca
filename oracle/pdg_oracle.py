"""CPU ORACLE for the P-DivGNN hot path.  TEST INFRASTRUCTURE ONLY.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` /
``--impl reference`` legs may import this file; the product path
(``p-div-gnn_b200/``) never does and has no CPU fallback.

It is an independent pure-torch restatement of the reference's algorithm
(``/root/reference``; the reference itself cannot be imported on the GPU box and
needs ``torch_geometric``, which is not installed anywhere here).  Each function
cites the reference ``file:line`` it follows; third-party PyG semantics
(un-vendored, unpinned ``torch-geometric`` of ``pyproject.toml:38``) are restated
from SURVEY.md section 2.3.

Pinning status: the reference holds NO golden vectors or tests for this path
(``test/test_graph_utils.py`` only checks mesh<->graph bookkeeping).  The oracle is
pinned instead against outputs of the reference's *unmodified* modules executed in
the build container through the test-only PyG shim ``oracle/pyg_shim`` --
``oracle/make_golden.py`` wrote those outputs to ``tests/golden/*.npz`` and
``tests/test_oracle_golden.py`` replays them bit-for-bit on CPU.
Two restatements have no reference output to replay and are pinned by hand-derived known answers only -- **parity
unpinned** for them: ``compute_node_labels`` (the reference runs VTK filters; pyvista / VTK are absent) and
``is_periodic`` (``microgen.mesh.is_periodic``: an unpinned, un-vendored, absent dependency, restated from its
published algorithm).
"""
from __future__ import annotations

from collections import OrderedDict
from types import SimpleNamespace

import numpy as np
import torch
import torch.nn.functional as F

EPS_LN = 1e-5  # torch_geometric.nn.LayerNorm default eps

# --------------------------------------------------------------------------------------
# graph construction (datasets.py / convert_utils.py + PyG utils)
# --------------------------------------------------------------------------------------


def coalesce(edge_index: torch.Tensor, edge_attr, num_nodes: int):
    """PyG ``Data.coalesce()`` (datasets.py:119): sort columns by ``row*N+col``,
    merge duplicates by summing ``edge_attr`` (SURVEY 2.3c)."""
    row, col = edge_index[0].long(), edge_index[1].long()
    key = row * num_nodes + col
    uniq, inv = torch.unique(key, sorted=True, return_inverse=True)
    out_index = torch.stack([uniq // num_nodes, uniq % num_nodes], dim=0)
    if edge_attr is None:
        return out_index, None
    out_attr = torch.zeros(uniq.numel(), *edge_attr.shape[1:], dtype=edge_attr.dtype)
    out_attr.index_add_(0, inv, edge_attr)
    return out_index, out_attr


def to_undirected(edge_index: torch.Tensor, num_nodes: int) -> torch.Tensor:
    """PyG ``to_undirected`` (convert_utils.py:76-78): symmetrise then sort+unique."""
    row, col = edge_index[0], edge_index[1]
    both = torch.stack([torch.cat([row, col]), torch.cat([col, row])], dim=0)
    return coalesce(both, None, num_nodes)[0]


def face_to_edge(face: torch.Tensor, num_nodes: int) -> torch.Tensor:
    """PyG ``FaceToEdge`` on triangles (convert_utils.py:58-59):
    ``cat([face[:2], face[1:], face[::2]], 1)`` then ``to_undirected``."""
    assert face.shape[0] == 3
    ei = torch.cat([face[:2], face[1:], face[::2]], dim=1)
    return to_undirected(ei, num_nodes)


def quad_face_to_edge(face: torch.Tensor, num_nodes: int) -> torch.Tensor:
    """convert_utils.py:62-81 (quad meshes)."""
    assert face.shape[0] == 4
    ei = torch.cat([face[:2], face[1:3], face[2:], face[::3]], dim=1)
    return to_undirected(ei, num_nodes)


def edge_weights(pos: torch.Tensor, edge_index: torch.Tensor) -> torch.Tensor:
    """datasets.py:182-188 -- Euclidean length in the dtype of ``pos`` (float64 from
    pyvista); the caller casts ``.float()`` (datasets.py:254-256)."""
    d = pos[edge_index[0]] - pos[edge_index[1]]
    return torch.linalg.vector_norm(d, dim=1)


def compute_periodic_graph(pos: torch.Tensor, edge_index: torch.Tensor, edge_attr: torch.Tensor):
    """datasets.py:39-119.  ``pos`` is [N,3]; the last column is dropped (:40).
    Returns coalesced (edge_index, edge_attr) with periodic edges of weight 0."""
    p2 = pos[:, :-1].numpy()
    n = p2.shape[0]
    min_x, min_y = np.min(p2, axis=0)
    max_x, max_y = np.max(p2, axis=0)
    ids = np.arange(n)

    def side(mask):
        idx = np.where(mask)[0]
        return torch.from_numpy(idx[np.lexsort(p2[idx].T)])  # y-major, then x (:56)

    left = side(p2[:, 0] == min_x)
    right = side(p2[:, 0] == max_x)
    upper = side(p2[:, 1] == max_y)
    lower = side(p2[:, 1] == min_y)

    def corner(cx, cy):
        return ids[np.logical_and(p2[:, 0] == cx, p2[:, 1] == cy)]

    corners = torch.from_numpy(
        np.array([corner(min_x, min_y), corner(min_x, max_y), corner(max_x, min_y), corner(max_x, max_y)]).squeeze()
    )
    row, col = edge_index
    n_row = torch.cat((row, left, right, lower, upper, corners))
    n_col = torch.cat((col, right, left, upper, lower, corners.flip(dims=[0])))
    n_ei = torch.vstack([n_row, n_col]).long()
    attr = torch.zeros(n_ei.shape[1])
    attr[: edge_index.shape[1]] = edge_attr
    return coalesce(n_ei, attr, n)



def compute_node_labels(pos, faces):
    """``datasets.compute_node_labels`` (datasets.py:133-179) restated without VTK.

    The reference chains three VTK filters: ``extract_feature_edges(boundary_edges=True)`` (edges used by exactly
    one cell), ``connectivity()`` (connected regions of those edges) and ``cell_data_to_point_data()``; region 0 is
    taken as the external boundary and swapped with region 1 when its first point does not lie on the mesh bounds
    (``_regions_must_be_inverted``, :120-130).  For the plate-with-hole meshes this is: boundary loop touching
    the bounding box -> EXTERNAL_BOUNDARY (1), the other loop -> INTERNAL_BOUNDARY (-1), everything else
    INTERNAL (0).  Returns (labels [N] int64, number of regions).  pos [N,>=2], faces [3,F] or [4,F] (a cell side
    used by exactly one cell is a boundary edge whatever the cell type)."""
    import numpy as np
    pos = np.asarray(pos, dtype=np.float64)[:, :2]
    f = np.asarray(faces, dtype=np.int64)
    n = pos.shape[0]
    k = f.shape[0]
    e = np.concatenate([f[[i, (i + 1) % k]] for i in range(k)], axis=1)
    lo, hi = np.minimum(e[0], e[1]), np.maximum(e[0], e[1])
    keys, counts = np.unique(lo * n + hi, return_counts=True)
    bk = keys[counts == 1]
    ba, bb = bk // n, bk % n
    parent = np.arange(n)

    def find(x):
        while parent[x] != x:
            parent[x] = parent[parent[x]]
            x = parent[x]
        return x

    for a, b in zip(ba.tolist(), bb.tolist()):
        ra, rb = find(a), find(b)
        if ra != rb:
            parent[max(ra, rb)] = min(ra, rb)
    on_boundary = np.zeros(n, dtype=bool)
    on_boundary[ba] = True
    on_boundary[bb] = True
    xmin, ymin = pos.min(axis=0)
    xmax, ymax = pos.max(axis=0)
    labels = np.zeros(n, dtype=np.int64)
    roots = {}
    for i in np.nonzero(on_boundary)[0].tolist():
        r = find(i)
        touch = pos[i, 0] in (xmin, xmax) or pos[i, 1] in (ymin, ymax)
        roots[r] = roots.get(r, False) or touch
    for i in np.nonzero(on_boundary)[0].tolist():
        labels[i] = 1 if roots[find(i)] else -1
    return labels, len(roots)


def is_periodic(nodes_coords, tol: float = 1e-8, dim: int = 3) -> bool:
    """``microgen.mesh.is_periodic`` (== ``microgen.remesh.is_periodic``), asserted by the reference on every mesh it
    generates or benchmarks (generate_dataset.py:191, generate_dataset_hyperelast.py:160,237,
    benchmark_gnn_fem.py:195, plot_periodic_mesh.py:291; always called as ``is_periodic(shape.points[:, :-1])``,
    i.e. on the [N,2] in-plane coordinates with the default tolerance).

    ``microgen`` is an UNPINNED, un-vendored dependency (pyproject.toml:45) that is absent from this image, so this
    is a restatement of its published algorithm (the same routine ships as ``fedoo.Mesh.is_periodic``), **parity
    unpinned**: nodes within ``tol`` of the bounding-box minimum / maximum of an axis form the two opposite sides;
    each side is sorted along the other in-plane axis; the mesh is periodic when opposite sides hold the same number
    of nodes and no sorted coordinate of the max side exceeds its partner on the min side by more than ``tol``
    (the published test is one-sided: ``(crd[right, 1:] - crd[left, 1:] > tol).any()``, no absolute value).
    Axes beyond the columns present are not tested (2-D coordinates: x and y sides only)."""
    crd = np.asarray(nodes_coords, dtype=np.float64)
    ncol = crd.shape[1]
    dim = min(int(dim), ncol)
    if ncol > 2:
        raise NotImplementedError("3-D periodicity is outside the 2-D RVE path")
    for axis in range(dim):
        other = 1 - axis
        lo, hi = crd[:, axis].min(), crd[:, axis].max()
        side_lo = np.where(np.abs(crd[:, axis] - lo) < tol)[0]
        side_hi = np.where(np.abs(crd[:, axis] - hi) < tol)[0]
        side_lo = side_lo[np.argsort(crd[side_lo, other], kind="stable")]
        side_hi = side_hi[np.argsort(crd[side_hi, other], kind="stable")]
        if len(side_lo) != len(side_hi):
            return False
        if (crd[side_hi, other] - crd[side_lo, other] > tol).any():
            return False
    return True


def convert_mesh_to_graph(pos, faces, mean_stress) -> SimpleNamespace:
    """``benchmark_gnn_fem.convert_mesh_to_graph`` (benchmark_gnn_fem.py:388-415, the "with preprocessing" series):
    mesh_to_graph -> edge lengths -> periodic graph -> 2-D fp32 positions, broadcast mean stress, node labels as
    ``surfaces_nodes_for_div`` and ``nodes_types``.  pos [N,>=2] float64, faces [3,F] / [4,F]."""
    pos = torch.from_numpy(np.asarray(pos, dtype=np.float64))
    face = torch.from_numpy(np.asarray(faces, dtype=np.int64))
    n = pos.shape[0]
    ei = face_to_edge(face, n) if face.shape[0] == 3 else quad_face_to_edge(face, n)
    attr = edge_weights(pos, ei).float()
    ei, attr = compute_periodic_graph(pos, ei, attr)
    labels, _ = compute_node_labels(pos.numpy(), face.numpy())
    lab = torch.unsqueeze(torch.from_numpy(labels), 1)
    ms = torch.ones((n, 3)) * torch.Tensor(tuple(float(v) for v in mean_stress))
    return SimpleNamespace(pos=pos[:, :2].float(), face=face, edge_index=ei, edge_attr=attr, mean_stress=ms,
                           surfaces_nodes_for_div=lab, nodes_types=torch.clone(lab), is_periodic=True, num_nodes=n)


def init_op_div(row, col, data, shape) -> torch.Tensor:
    """datasets.py:191-213 -- coalesced fp32 sparse COO (N x 2N)."""
    idx = torch.vstack((torch.as_tensor(row, dtype=torch.long), torch.as_tensor(col, dtype=torch.long)))
    val = torch.as_tensor(np.asarray(data), dtype=torch.float32)
    return torch.sparse_coo_tensor(idx, val, torch.Size(tuple(int(s) for s in shape)), dtype=torch.float32).coalesce()


def build_graph(sample: dict, periodic: bool = True) -> SimpleNamespace:
    """One dataset item, following MeshStressFieldDatasetInMemory.__init__
    (datasets.py:240-281) on an in-memory sample (see ``synth.make_rve_mesh``)."""
    pos = torch.from_numpy(np.asarray(sample["pos"], dtype=np.float64))
    face = torch.from_numpy(np.asarray(sample["faces"], dtype=np.int64))
    n = pos.shape[0]
    ei = face_to_edge(face, n) if face.shape[0] == 3 else quad_face_to_edge(face, n)
    attr = edge_weights(pos, ei).float()
    org_ei = ei
    if periodic:
        ei, attr = compute_periodic_graph(pos, ei, attr)
    stress = torch.from_numpy(np.asarray(sample["stress_field"])).float()
    ms = np.asarray(sample["mean_stress"])
    mean_stress = torch.ones(stress.shape) * torch.Tensor((ms[0], ms[1], ms[2]))
    labels = torch.unsqueeze(torch.from_numpy(np.asarray(sample["labels"], dtype=np.int64)), 1)
    return SimpleNamespace(
        pos=pos[:, :2].float(),
        face=face,
        edge_index=ei,
        org_edge_index=org_ei,
        edge_attr=attr,
        mean_stress=mean_stress,
        local_stress=stress,
        op_div_matrix=init_op_div(sample["op_div_row"], sample["op_div_col"], sample["op_div_data"], sample["op_div_shape"]),
        surfaces_nodes_for_div=labels,
        nodes_types=labels,
        is_periodic=periodic,
        num_nodes=n,
    )


def collate(graphs) -> SimpleNamespace:
    """PyG ``Batch.from_data_list`` for the keys the hot path reads (SURVEY 2.3d):
    node-offset ``edge_index``; ``batch``/``ptr``; sparse ``op_div_matrix`` stacked
    along rows only (columns NOT offset, width = max 2N)."""
    ns = [g.num_nodes for g in graphs]
    ptr = torch.tensor([0] + list(np.cumsum(ns)), dtype=torch.long)
    rows, cols, vals = [], [], []
    for g, off in zip(graphs, ptr[:-1]):
        m = g.op_div_matrix
        rows.append(m.indices()[0] + off)
        cols.append(m.indices()[1])
        vals.append(m.values())
    width = max(int(g.op_div_matrix.shape[1]) for g in graphs)
    op = torch.sparse_coo_tensor(
        torch.vstack([torch.cat(rows), torch.cat(cols)]), torch.cat(vals), (int(ptr[-1]), width)
    ).coalesce()
    return SimpleNamespace(
        pos=torch.cat([g.pos for g in graphs]),
        edge_index=torch.cat([g.edge_index + off for g, off in zip(graphs, ptr[:-1])], dim=1),
        edge_attr=torch.cat([g.edge_attr for g in graphs]),
        mean_stress=torch.cat([g.mean_stress for g in graphs]),
        local_stress=torch.cat([g.local_stress for g in graphs]),
        nodes_types=torch.cat([g.nodes_types for g in graphs]),
        surfaces_nodes_for_div=torch.cat([g.surfaces_nodes_for_div for g in graphs]),
        op_div_matrix=op,
        batch=torch.repeat_interleave(torch.arange(len(graphs)), torch.tensor(ns)),
        ptr=ptr,
        batch_size=len(graphs),
        num_nodes=int(ptr[-1]),
    )


def batch_to(batch: SimpleNamespace, device) -> SimpleNamespace:
    """``Batch.to(device)`` (gnn_train.py:157): the same collated batch with every tensor moved -- used to run this
    restatement in the reference's own execution mode, eager torch on ``cuda`` (gnn_train.py:344)."""
    return SimpleNamespace(**{k: (v.to(device) if torch.is_tensor(v) else v) for k, v in vars(batch).items()})


def dataset_stats(graphs) -> dict:
    """datasets.py:283-291 -- 8 scalar stats; ``std`` is the unbiased torch default."""
    cat = lambda k: torch.cat([getattr(g, k) for g in graphs])  # noqa: E731
    pos, ms, ls, ew = cat("pos"), cat("mean_stress"), cat("local_stress"), cat("edge_attr")
    return dict(
        mean_pos=pos.mean(), std_pos=pos.std(),
        mean_mean_stress=ms.mean(), std_mean_stress=ms.std(),
        mean_local_stress=ls.mean(), std_local_stress=ls.std(),
        mean_edge_weight=ew.mean(), std_edge_weight=ew.std(),
    )


# --------------------------------------------------------------------------------------
# model (models.py)
# --------------------------------------------------------------------------------------

STATE_KEYS = [
    "node_encoder.0.weight", "node_encoder.0.bias", "node_encoder.2.weight", "node_encoder.2.bias",
    "node_encoder.4.weight", "node_encoder.4.bias",
    "edge_encoder.0.weight", "edge_encoder.0.bias", "edge_encoder.2.weight", "edge_encoder.2.bias",
    "edge_encoder.4.weight", "edge_encoder.4.bias",
    "processor.edge_net.0.weight", "processor.edge_net.0.bias", "processor.edge_net.2.weight",
    "processor.edge_net.2.bias", "processor.edge_net.4.weight", "processor.edge_net.4.bias",
    "processor.node_net.0.weight", "processor.node_net.0.bias", "processor.node_net.2.weight",
    "processor.node_net.2.bias", "processor.node_net.4.weight", "processor.node_net.4.bias",
    "node_decoder.0.weight", "node_decoder.0.bias", "node_decoder.2.weight", "node_decoder.2.bias",
]


def init_state_dict(latent: int = 128, in_nodes: int = 6, in_edges: int = 1, out_nodes: int = 3, seed=None):
    """Default-initialised parameters in the construction order of
    EncodeProcessDecode.__init__ (models.py:260-286) so that, under the same
    ``torch.manual_seed``, values equal the reference's."""
    if seed is not None:
        torch.manual_seed(seed)
    sd = OrderedDict()

    def mlp_ln(prefix, fin):
        l0, l2 = torch.nn.Linear(fin, latent), torch.nn.Linear(latent, latent)
        sd[prefix + ".0.weight"], sd[prefix + ".0.bias"] = l0.weight.detach(), l0.bias.detach()
        sd[prefix + ".2.weight"], sd[prefix + ".2.bias"] = l2.weight.detach(), l2.bias.detach()
        sd[prefix + ".4.weight"], sd[prefix + ".4.bias"] = torch.ones(latent), torch.zeros(latent)

    mlp_ln("node_encoder", in_nodes)
    mlp_ln("edge_encoder", in_edges)
    mlp_ln("processor.edge_net", 3 * latent)
    mlp_ln("processor.node_net", 2 * latent)
    d0, d2 = torch.nn.Linear(latent, latent), torch.nn.Linear(latent, out_nodes)
    sd["node_decoder.0.weight"], sd["node_decoder.0.bias"] = d0.weight.detach(), d0.bias.detach()
    sd["node_decoder.2.weight"], sd["node_decoder.2.bias"] = d2.weight.detach(), d2.bias.detach()
    assert list(sd.keys()) == STATE_KEYS
    return sd


def graph_layer_norm(x, weight, bias, eps: float = EPS_LN):
    """PyG ``LayerNorm(mode='graph')`` with ``batch=None`` (SURVEY 2.3a): ONE mean and
    ONE population std over every element of ``x``; eps is added to the std."""
    x = x - x.mean()
    out = x / (x.std(unbiased=False) + eps)
    return out * weight + bias


def _mlp_ln(x, sd, p):
    """Linear-ReLU-Linear-ReLU-LayerNorm (models.py:194-208, 260-274)."""
    h = F.relu(F.linear(x, sd[p + ".0.weight"], sd[p + ".0.bias"]))
    h = F.relu(F.linear(h, sd[p + ".2.weight"], sd[p + ".2.bias"]))
    return graph_layer_norm(h, sd[p + ".4.weight"], sd[p + ".4.bias"])


def processor_step(x, e, edge_index, sd):
    """Processor.forward / message / update (models.py:210-243) with PyG
    ``propagate`` semantics (SURVEY 2.3b): x_i = x[col] (target), x_j = x[row]."""
    row, col = edge_index[0], edge_index[1]
    msg = _mlp_ln(torch.cat([x[col], x[row], e], dim=-1), sd, "processor.edge_net")  # :233-238
    agg = torch.zeros(x.shape[0], msg.shape[1], dtype=msg.dtype, device=msg.device).index_add_(0, col, msg)
    upd = _mlp_ln(torch.cat([agg, x], dim=-1), sd, "processor.node_net")  # :240-243
    new_e = _mlp_ln(torch.cat([x[row], x[col], e], dim=-1), sd, "processor.edge_net")  # :219-222
    return upd + x, new_e + e  # :224-225


def format_node_features(batch, stats, scale: bool):
    """models.py:140-152."""
    ms, pos = batch.mean_stress, batch.pos
    if scale:
        ms = (ms - stats["mean_mean_stress"]) / stats["std_mean_stress"]
        pos = (pos - stats["mean_pos"]) / stats["std_pos"]
    return torch.hstack([ms, pos, batch.nodes_types])


def format_edge_features(batch, stats, scale: bool):
    """models.py:154-162."""
    ea = batch.edge_attr
    if scale:
        ea = (ea - stats["mean_edge_weight"]) / stats["std_edge_weight"]
    return ea


def forward(sd, batch, stats, steps: int = 10, scale_output: bool = True, scale_input: bool = True,
            dtype=torch.float32, return_latents: bool = False):
    """EncodeProcessDecode.forward (models.py:288-326) -> local_stress [N,3]."""
    if not torch.any(batch.mean_stress):  # :294-299
        return torch.zeros_like(batch.mean_stress)
    if dtype != torch.float32:
        sd = {k: v.to(dtype) for k, v in sd.items()}
        stats = {k: torch.as_tensor(v).to(dtype) for k, v in stats.items()}
        batch = SimpleNamespace(**{k: (v.to(dtype) if torch.is_tensor(v) and v.is_floating_point() and not v.is_sparse else v)
                                   for k, v in vars(batch).items()})
    x = format_node_features(batch, stats, scale_input)
    if x.dtype != dtype:
        x = x.to(dtype)
    ew = format_edge_features(batch, stats, scale_input).unsqueeze(1)
    x = _mlp_ln(x, sd, "node_encoder")
    e = _mlp_ln(ew, sd, "edge_encoder")
    lat = [(x, e)]
    for _ in range(steps):
        x, e = processor_step(x, e, batch.edge_index, sd)
        lat.append((x, e))
    h = F.relu(F.linear(x, sd["node_decoder.0.weight"], sd["node_decoder.0.bias"]))
    out = F.linear(h, sd["node_decoder.2.weight"], sd["node_decoder.2.bias"])
    if scale_output:
        out = out * stats["std_local_stress"] + stats["mean_local_stress"]
    return (out, lat) if return_latents else out


# --------------------------------------------------------------------------------------
# loss (gnn_train.py)
# --------------------------------------------------------------------------------------


def normalized_mse_loss_single(gt, pred):
    """gnn_train.py:41-57."""
    mean_gt = gt.mean(dim=0)
    mse = (gt - pred).square().sum(dim=0)
    norm = (gt - mean_gt).square().sum(dim=0)
    return (mse / norm).mean()


def _stack_stress(local_stress):
    """gnn_train.py:68-70: [[sxx; sxy], [sxy; syy]] as [2N, 2]."""
    a = local_stress[:, [0, 2]].T.reshape(-1)
    b = local_stress[:, [2, 1]].T.reshape(-1)
    return torch.stack([a, b], dim=1)


def compute_divergence(local_stress, op_div_rows_of_graph, labels):
    """gnn_train.py:60-92 -- the densify-and-slice path (:73-76) exactly as written.
    ``op_div_rows_of_graph`` is the (N_i x max2N) row block a PyG ``batch[i]`` yields."""
    s = _stack_stress(local_stress)
    n = op_div_rows_of_graph.shape[0]
    div = op_div_rows_of_graph.to_dense()[:, : n * 2] @ s
    lab = labels.squeeze()
    div[lab == 1] = 0
    div[lab == -1] = 0
    return torch.sum(torch.mean(torch.square(div), dim=0))


def compute_divergence_spmm(local_stress, row, col, val, labels):
    """Second opinion, compare_results.py:647-673: plain ``op_div @ S`` on the
    graph-local COO triplets, same masks and reduction."""
    s = _stack_stress(local_stress)
    n = local_stress.shape[0]
    div = torch.zeros(n, 2, dtype=s.dtype, device=s.device).index_add_(0, row, val.to(s.dtype)[:, None] * s[col])
    lab = labels.squeeze()
    div = div * ((lab != 1) & (lab != -1)).to(s.dtype)[:, None]
    return torch.sum(torch.mean(torch.square(div), dim=0))


def opdiv_entries(op_div_matrix, ptr):
    """The entries of a row-stacked batch operator that ``compute_divergence`` keeps, with the stacked-stress value
    each one multiplies.  The batch operator is coalesced first (fp32 sums of duplicates, as torch and the device
    path do); entry k of graph i multiplies S[col_k] of that graph, S[j] = (sxx, sxy)[j] for j < N_i and
    (sxy, syy)[j - N_i] below (gnn_train.py:68-70); columns outside [0, 2 N_i) are sliced away (:73-76).
    Returns (row, node, first, val): batch row, batch node of S[col], True where S[col] = (sxx, sxy), fp32 value."""
    m = op_div_matrix.coalesce()
    row, col = m.indices()[0], m.indices()[1]
    val = m.values()
    ptr = ptr.to(row.device)
    g = torch.searchsorted(ptr, row, right=True) - 1
    n0, ni = ptr[g], ptr[g + 1] - ptr[g]
    keep = (col >= 0) & (col < 2 * ni)
    row, col, val, n0, ni = row[keep], col[keep], val[keep], n0[keep], ni[keep]
    first = col < ni
    node = n0 + torch.where(first, col, col - ni)
    return row, node, first, val


def loss_fp64(pred, local_stress, mean_ls, std_ls, ptr, op_div_matrix=None, labels=None, divergence=True,
              penalty=1.0, upstream=(1.0, 1.0)):
    """Vectorised fp64 restatement of ``train_loss``'s loss assembly (gnn_train.py:162-202) and of its gradient, for
    any batch: segment sums instead of the per-graph loop and the dense operator blocks.

    The ground truth is standardised in fp32, ``(local_stress - mean) / std`` rounded as IEEE fp32 like the reference
    and the device kernel; everything after that is fp64 from the same fp32 ``pred``, ground truth and operator values.
    ``upstream`` = (g_nmse, g_div) weights the two outputs in ``grad`` = d(g_nmse*nmse + g_div*div)/d pred.
    Returns a namespace: gt (fp32), nmse_graph [B], div_node [N,2] (masked), div_graph [B] (before penalty),
    nmse, div (= penalty * mean div_graph, 0 without divergence), total, grad [N,3]."""
    dev = pred.device
    f64 = torch.float64
    ls = local_stress.to(torch.float32)
    # full-size operands: a scalar divisor may be turned into a multiplication by its reciprocal
    gt = (ls - torch.full_like(ls, float(mean_ls))) / torch.full_like(ls, float(std_ls))
    ptr = ptr.to(dev)
    b, n = ptr.numel() - 1, pred.shape[0]
    ni = (ptr[1:] - ptr[:-1]).to(f64)
    gid = torch.repeat_interleave(torch.arange(b, device=dev), ptr[1:] - ptr[:-1])
    seg = lambda x: torch.zeros(b, *x.shape[1:], dtype=f64, device=dev).index_add_(0, gid, x)  # noqa: E731
    p, t = pred.to(f64), gt.to(f64)
    mean = seg(t) / ni[:, None]
    norm = seg((t - mean[gid]).square())
    d = p - t
    nmse_graph = (seg(d.square()) / norm).mean(dim=1)
    g_nmse, g_div = (float(v) for v in upstream)
    grad = g_nmse * 2.0 * d / norm[gid] / (3.0 * b)
    div_node = torch.zeros(n, 2, dtype=f64, device=dev)
    div_graph = torch.zeros(b, dtype=f64, device=dev)
    if divergence:
        row, node, first, val = opdiv_entries(op_div_matrix, ptr)
        v = val.to(f64)[:, None]
        s = torch.where(first[:, None], p[node][:, [0, 2]], p[node][:, [2, 1]])
        div_node.index_add_(0, row, v * s)
        lab = labels.reshape(-1).to(dev)
        div_node *= ((lab != 1) & (lab != -1)).to(f64)[:, None]
        div_graph = seg(div_node.square()).sum(dim=1) / ni
        # d div_graph_i / d S[col] = 2 / N_i * sum over rows of v * div[row]
        ds = v * div_node[row] * (g_div * penalty * 2.0 / (ni[gid[row]] * b))[:, None]
        grad.index_add_(0, node, torch.where(first[:, None], torch.stack([ds[:, 0], 0 * ds[:, 0], ds[:, 1]], 1),
                                             torch.stack([0 * ds[:, 0], ds[:, 1], ds[:, 0]], 1)))
    nmse = nmse_graph.sum() / b
    div = penalty * div_graph.sum() / b if divergence else torch.zeros((), dtype=f64, device=dev)
    return SimpleNamespace(gt=gt, nmse_graph=nmse_graph, div_node=div_node, div_graph=div_graph, nmse=nmse, div=div,
                           total=nmse + div, grad=grad)


def op_div_row_block(op, start: int, end: int):
    """What PyG ``Batch.get_example`` returns for the row-stacked sparse attribute
    (SURVEY 2.3d): rows [start,end) narrowed, column count unchanged."""
    idx, val = op.indices(), op.values()
    sel = (idx[0] >= start) & (idx[0] < end)
    return torch.sparse_coo_tensor(
        torch.vstack([idx[0][sel] - start, idx[1][sel]]), val[sel], (end - start, op.shape[1])
    ).coalesce()


def train_loss(sd, batch, stats, steps: int = 10, divergence: bool = True, penalty: float = 10.0,
               dtype=torch.float32):
    """Loss assembly of ``train()`` (gnn_train.py:154-202):
    forward(scale_output=False) ; standardised GT ; per-graph NMSE and lambda*div ;
    both divided by the number of graphs.  Returns (total, nmse, div, pred)."""
    pred = forward(sd, batch, stats, steps, scale_output=False, scale_input=True, dtype=dtype)
    gt = (batch.local_stress.to(dtype) - stats["mean_local_stress"].to(dtype)) / stats["std_local_stress"].to(dtype)
    nmse = 0
    div = 0
    ptr = batch.ptr.tolist()
    for i in range(batch.batch_size):  # data_utils.py:25-33
        s, e_ = ptr[i], ptr[i + 1]
        nmse = nmse + normalized_mse_loss_single(gt[s:e_], pred[s:e_])
        if divergence:
            blk = op_div_row_block(batch.op_div_matrix, s, e_).to(dtype)
            div = div + compute_divergence(pred[s:e_], blk, batch.surfaces_nodes_for_div[s:e_]) * penalty
    nmse = nmse / batch.batch_size
    total = nmse
    if divergence:
        div = div / batch.batch_size
        total = nmse + div
    else:
        div = torch.zeros((), dtype=dtype, device=pred.device)
    return total, nmse, div, pred


def loss_and_grads(sd, batch, stats, steps: int = 10, divergence: bool = True, penalty: float = 10.0,
                   dtype=torch.float32):
    """fwd + bwd of one training batch; gradients in STATE_KEYS order."""
    p = OrderedDict((k, v.detach().clone().to(dtype).requires_grad_(True)) for k, v in sd.items())
    total, nmse, div, pred = train_loss(p, batch, stats, steps, divergence, penalty, dtype)
    grads = torch.autograd.grad(total, list(p.values()), allow_unused=True)
    grads = [g if g is not None else torch.zeros_like(v) for g, v in zip(grads, p.values())]
    return total.detach(), nmse.detach(), div.detach() if torch.is_tensor(div) else div, pred.detach(), \
        OrderedDict(zip(p.keys(), grads))
