"""Host-side graph construction for the pipe-network message-passing path.

Two jobs, both run ONCE per model (never per forward):

1. ``build_wdn_graph_from_inp`` -- EPANET ``.inp`` -> ``WDNGraph`` with the exact node
   numbering / ``edge_index`` / ``pipe_ends`` the reference produces
   (reference: models/utils.py:18-51 parse, :54-69 token helpers, :72-81 WDNGraph,
   :84-166 build).  Integer outputs are required to be bit-identical to the reference;
   tests/test_graph.py checks that against goldens minted by the reference's own code.

2. ``build_gcn_csr`` -- ``edge_index`` -> CSR (aggregate at edge target) plus its CSC
   transpose, carrying the symmetric GCN normalisation weights that
   ``torch_geometric.nn.conv.gcn_conv.gcn_norm`` would compute every forward
   (reference call sites: models/detector.py:162-164,199 with add_self_loops=True,
   normalize=True, cached=False).  The reference recomputes these for the B-times
   replicated graph in every conv of every step (SURVEY F4); here they are computed once
   for the single graph, with the same torch ops so the fp32 weights are bit-identical.
"""
from __future__ import annotations

import re
from dataclasses import dataclass
from pathlib import Path
from typing import Any, Dict, List, Sequence, Tuple

import numpy as np
import torch

__all__ = [
    "parse_epanet_inp",
    "WDNGraph",
    "build_wdn_graph_from_inp",
    "GCNCsr",
    "build_gcn_csr",
    "batchify_edge_index",
]

_HEADER = re.compile(r"^\s*\[(.+?)\]\s*$")


def parse_epanet_inp(inp_path: str | Path) -> Dict[str, List[str]]:
    """Split an EPANET ``.inp`` file into ``{SECTION_NAME_UPPER: [payload lines]}``.

    Behaviour follows reference models/utils.py:18-51: blank lines are dropped, a
    ``[name]`` line opens (or re-opens) a section, text after the first ``;`` is a
    comment, lines before the first header are ignored, payload lines are kept unsplit.
    """
    out: Dict[str, List[str]] = {}
    section: List[str] | None = None
    with Path(inp_path).open("r", encoding="utf-8", errors="ignore") as fh:
        for raw in fh:
            text = raw.strip()
            if not text:
                continue
            hdr = _HEADER.match(text)
            if hdr is not None:
                section = out.setdefault(hdr.group(1).strip().upper(), [])
                continue
            if section is None:
                continue
            text = text.partition(";")[0].strip()
            if text:
                section.append(text)
    return out


def _first_tokens(lines: Sequence[str]) -> List[str]:
    """IDs of a node section: first whitespace token of each line (utils.py:54-60)."""
    return [ln.split()[0] for ln in lines if ln.split()]


def _link_table(lines: Sequence[str]) -> Dict[str, Tuple[str, str]]:
    """``{link_id: (node1, node2)}`` for lines with >=3 tokens (utils.py:63-69).

    A repeated id keeps its FIRST position in iteration order but takes the LAST
    endpoints -- plain ``dict`` assignment semantics, which the edge order depends on.
    """
    table: Dict[str, Tuple[str, str]] = {}
    for ln in lines:
        tok = ln.split()
        if len(tok) >= 3:
            table[tok[0]] = (tok[1], tok[2])
    return table


@dataclass(frozen=True)
class WDNGraph:
    """Same fields as the reference dataclass (models/utils.py:72-81)."""

    node_names: List[str]
    node_to_idx: Dict[str, int]
    pipe_ids: List[str]
    pipe_to_idx: Dict[str, int]
    pipe_ends: np.ndarray  # (P, 2) int64
    edge_index: Any  # torch.LongTensor (2, E)


def build_wdn_graph_from_inp(
    inp_path: str | Path,
    sensor_node_ids: Sequence[str],
    pipe_ids_in_order: Sequence[str],
    *,
    include_all_nodes: bool = True,
    include_links: Sequence[str] = ("PIPES", "PUMPS", "VALVES"),
    add_self_loops: bool = True,
    make_undirected: bool = True,
) -> WDNGraph:
    """Drop-in for reference ``build_wdn_graph_from_inp`` (models/utils.py:84-166).

    * node set = sensors U (JUNCTIONS, RESERVOIRS, TANKS when ``include_all_nodes``)
      U every link endpoint; numbered by Python ``sorted()`` on the id strings
      (lexicographic: 'R1' < 'n100' < 'n11'), utils.py:113-125;
    * ``edge_index``: for each link of ``include_links`` in dict order, ``(u, v)``
      then ``(v, u)`` when ``make_undirected``; self loops appended last on request,
      utils.py:144-157;
    * ``pipe_ends`` only for ``pipe_ids_in_order`` and only looked up in ``[PIPES]``,
      utils.py:128-141; an unknown pipe id is a ``ValueError``.
    """
    sections = parse_epanet_inp(inp_path)

    links: Dict[str, Tuple[str, str]] = {}
    for name in include_links:
        links.update(_link_table(sections.get(name.upper(), ())))
    if not links:
        raise ValueError(f"No link endpoints found from sections {tuple(include_links)} in inp file.")

    names = set(sensor_node_ids)
    if include_all_nodes:
        for sec in ("JUNCTIONS", "RESERVOIRS", "TANKS"):
            names.update(_first_tokens(sections.get(sec, ())))
    for a, b in links.values():
        names.add(a)
        names.add(b)
    node_names = sorted(names)
    node_to_idx = {name: i for i, name in enumerate(node_names)}

    pipes = _link_table(sections.get("PIPES", ()))
    if not pipes:
        raise ValueError("No [PIPES] section found or empty; cannot map pipe_ids to endpoints.")
    pipe_ids = list(pipe_ids_in_order)
    pipe_to_idx = {pid: i for i, pid in enumerate(pipe_ids)}
    pipe_ends = np.zeros((len(pipe_ids), 2), dtype=np.int64)
    for i, pid in enumerate(pipe_ids):
        ends = pipes.get(pid)
        if ends is None:
            raise ValueError(f"Pipe id {pid} not found in inp [PIPES].")
        pipe_ends[i] = (node_to_idx[ends[0]], node_to_idx[ends[1]])

    uv = np.array([(node_to_idx[a], node_to_idx[b]) for a, b in links.values()], dtype=np.int64)
    if make_undirected:
        # interleave (u,v),(v,u) per link
        pairs = np.stack([uv, uv[:, ::-1]], axis=1).reshape(-1, 2)
    else:
        pairs = uv
    if add_self_loops:
        loops = np.arange(len(node_names), dtype=np.int64)
        pairs = np.concatenate([pairs, np.stack([loops, loops], axis=1)], axis=0)
    edge_index = torch.from_numpy(np.ascontiguousarray(pairs.T)).to(torch.long)

    return WDNGraph(node_names, node_to_idx, pipe_ids, pipe_to_idx, pipe_ends, edge_index)


def batchify_edge_index(edge_index_single: torch.Tensor, num_nodes: int, batch_size: int) -> torch.Tensor:
    """Disjoint union of ``batch_size`` copies (reference models/detector.py:105-114).

    Only the oracle and the PyG-signature compatibility path need this; the CUDA path
    treats the batch as a dense leading dimension and never materialises it.
    """
    e = edge_index_single.size(1)
    off = torch.arange(batch_size, device=edge_index_single.device).repeat_interleave(e) * num_nodes
    return edge_index_single.repeat(1, batch_size) + off.unsqueeze(0)


@dataclass(frozen=True)
class GCNCsr:
    """Normalised adjacency of ONE graph, in both orientations, on the host.

    ``rowptr/col/val``  : CSR of A_hat, row = message target (``edge_index[1]``),
                          ``col`` = message source (``edge_index[0]``); within a row the
                          entries keep ``edge_index`` order and the GCN self loop is last,
                          i.e. the order in which a sequential scatter-add over PyG's edge
                          list would add them.
    ``t_rowptr/t_col/t_val`` : CSR of A_hat^T (the "CSC transpose"): row = source,
                          entries ordered by edge position, used by every backward.
    ``t_perm``          : position in the forward arrays of each transposed entry.
    ``edge/t_edge``     : for every entry of the two orders, the position in the input ``edge_index`` of the edge it
                          comes from; an appended self loop holds the position of the self loop it replaces (the
                          last one, if a node had several), or -1 where the node had none (weight 1).  This is what
                          maps per-call ``edge_weight`` values (``num_edges`` of them) onto the entries.
    """

    num_nodes: int
    rowptr: np.ndarray  # int32 [N+1]
    col: np.ndarray  # int32 [nnz]
    val: np.ndarray  # float32 [nnz]
    t_rowptr: np.ndarray
    t_col: np.ndarray
    t_val: np.ndarray
    t_perm: np.ndarray  # int32 [nnz]
    edge: np.ndarray  # int32 [nnz]
    t_edge: np.ndarray  # int32 [nnz]
    num_edges: int

    @property
    def nnz(self) -> int:
        return int(self.col.shape[0])


def gcn_norm_edges(edge_index: torch.Tensor, num_nodes: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """PyG ``gcn_norm(edge_index, None, num_nodes, improved=False, add_self_loops=True)``.

    Published algorithm (torch_geometric/nn/conv/gcn_conv.py, 2.x): drop existing self
    loops, append one ``(i, i)`` per node at the END of the list with weight 1
    (``add_remaining_self_loops``); ``deg = scatter_add(w, col)``; ``dis = deg^-0.5``
    with ``inf -> 0``; ``norm = dis[row] * w * dis[col]``.  Computed with the same torch
    ops (``pow_(-0.5)``, two gathers, two multiplies) so the fp32 bits match what the
    reference's conv would see on CPU.
    """
    ei = edge_index.detach().to("cpu", torch.long)
    keep = ei[0] != ei[1]
    loops = torch.arange(num_nodes, dtype=torch.long).unsqueeze(0).repeat(2, 1)
    ei = torch.cat([ei[:, keep], loops], dim=1)
    w = torch.ones(ei.size(1), dtype=torch.float32)
    row, col = ei[0], ei[1]
    deg = torch.zeros(num_nodes, dtype=torch.float32).scatter_add_(0, col, w)
    dis = deg.pow_(-0.5)
    dis.masked_fill_(dis == float("inf"), 0.0)
    norm = dis[row] * w * dis[col]
    return ei, norm


def build_gcn_csr(edge_index: torch.Tensor, num_nodes: int) -> GCNCsr:
    """``edge_index`` (2,E) int64 of ONE graph -> ``GCNCsr`` (see class docstring)."""
    if edge_index.dim() != 2 or edge_index.size(0) != 2:
        raise ValueError(f"edge_index must be (2, E), got {tuple(edge_index.shape)}")
    if num_nodes <= 0:
        raise ValueError("num_nodes must be positive")
    if edge_index.numel() and (int(edge_index.min()) < 0 or int(edge_index.max()) >= num_nodes):
        raise ValueError("edge_index entries out of range for num_nodes")
    ei, norm = gcn_norm_edges(edge_index, num_nodes)
    # source edge of each normalised edge: kept non-loop edges in order, then per node its last removed loop or -1
    e_in = edge_index.detach().to("cpu", torch.long)
    pos = torch.arange(e_in.size(1), dtype=torch.long)
    is_loop = e_in[0] == e_in[1]
    loop_src = torch.full((num_nodes,), -1, dtype=torch.long)
    loop_src[e_in[0, is_loop]] = pos[is_loop]  # CPU index_put: the last duplicate wins, as PyG's loop_attr assignment
    ent_src_edge = torch.cat([pos[~is_loop], loop_src]).numpy()
    src = ei[0].numpy()
    dst = ei[1].numpy()
    w = norm.numpy()
    nnz = src.shape[0]

    def _csr(rows: np.ndarray, cols: np.ndarray):
        order = np.argsort(rows, kind="stable")  # stable: keeps edge order inside a row
        ptr = np.zeros(num_nodes + 1, dtype=np.int64)
        np.add.at(ptr, rows + 1, 1)
        ptr = np.cumsum(ptr)
        return ptr.astype(np.int32), cols[order].astype(np.int32), w[order].astype(np.float32), order

    rowptr, col, val, order_f = _csr(dst, src)
    t_rowptr, t_col, t_val, order_t = _csr(src, dst)
    # t_perm[k] = index in forward arrays holding the same edge as transposed entry k
    pos_in_fwd = np.empty(nnz, dtype=np.int64)
    pos_in_fwd[order_f] = np.arange(nnz)
    t_perm = pos_in_fwd[order_t].astype(np.int32)
    return GCNCsr(int(num_nodes), rowptr, col, val, t_rowptr, t_col, t_val, t_perm, ent_src_edge[order_f].astype(np.int32),
                  ent_src_edge[order_t].astype(np.int32), int(edge_index.size(1)))
