"""Seeded fixtures whose sizes sit on the tile boundaries of the layer kernels (tiles of kTM = 128 edges, nodes or
(node, channel) rows), shared by tests/test_gpu_tile_shapes.py and its CPU checks.

make_graph_case's conventions (seeded, self-loops and duplicate edges allowed, isolated rows, `gain` on the coordinate
heads), but E, the row layout and N*C are exact rather than random:

  ragged_1     N = 1, E = 1 (mod 128), C = 3: N*C is ragged too; gravity, Fe = 4 (the widest tensor-core edge kernel)
  ragged_127   N = 127, E = 127 (mod 128), C = 8, Fe = 0
  aligned      N, E and N*C multiples of 128, C = 1, Fe = 1, gravity
  tile_rows    a CSR built row by row: row starts at offsets 0, 1, 31, 32, 33, 126, 127 of an edge tile, a row of exactly
               128 edges that starts a tile, one of 129, one of 3 * 128 + 1, runs of isolated rows between them
  one_node     B = 1, N = 1, one self-loop
  many_graphs  about 400 graphs of 1-3 nodes: graph boundaries inside every node tile and (node, channel) tile
  no_edges     E = 0
"""
import torch

from tests.gpu_util import make_graph_case

TM = 128


def _exact_e(sizes, deg, e_mod):
    """heavy_row (extra edges of row 1) that makes E = sum(sizes) * deg + heavy_row land on e_mod (mod 128)."""
    return (e_mod - sum(sizes) * deg) % TM


def _tile_rows_layout():
    """Row lengths in CSR order (0 = isolated row) and the row starts the layout promises, as (start, length)."""
    lengths, marks = [], []
    pos = 0

    def iso(k):
        lengths.extend([0] * k)

    def row(n, mark=None):
        nonlocal pos
        if mark is not None:
            marks.append((pos, n, mark))
        lengths.append(n)
        pos += n

    def row_to(offset, mark=None):        # a row that ends where the next row starts at `offset` of a tile
        n = (offset - pos) % TM or TM
        row(n, mark)

    iso(3)
    row_to(1, "start@0")
    iso(2)
    row_to(31, "start@1")
    row_to(32, "start@31")
    iso(4)
    row_to(33, "start@32")
    row_to(126, "start@33")
    iso(1)
    row_to(127, "start@126")
    row_to(0, "start@127")
    iso(5)
    row(TM, "128@tile")
    iso(2)
    row(TM + 1, "129@tile")
    row_to(0)
    iso(3)
    row(3 * TM + 1, "3x128+1@tile")
    return lengths, marks


def _tile_rows_case(seed=41, C=3, Fe=1, tail_rows=560):
    lengths, _ = _tile_rows_layout()
    g = torch.Generator().manual_seed(seed + 500)
    # the rest of the graph: rows of degree 0-14 (about one in six isolated)
    tail = torch.randint(0, 15, (tail_rows,), generator=g)
    tail[torch.rand(tail_rows, generator=g) < 1 / 6] = 0
    lengths = lengths + tail.tolist() + [0, 0]
    N = len(lengths)
    sizes = [N // 3, N // 3, N - 2 * (N // 3)]
    cfg, params, inp = make_graph_case(seed, sizes, 0, C, Fe=Fe, L=2)
    batch = inp["data_batch"]
    gptr = torch.tensor([0, sizes[0], sizes[0] + sizes[1], N])
    rows = torch.repeat_interleave(torch.arange(N), torch.tensor(lengths))
    b = batch[rows]
    lo, hi = gptr[b], gptr[b + 1]
    cols = lo + (torch.rand(rows.numel(), generator=g) * (hi - lo).double()).long()     # same graph, self-loops allowed
    ei = torch.stack([rows, cols])
    ei = ei[:, torch.randperm(ei.size(1), generator=g)]        # unsorted: the CSR sort is exercised
    x = inp["node_loc"]
    dist = (x[ei[0]] - x[ei[1]]).norm(dim=1, keepdim=True)
    inp = dict(inp, edge_index=ei, edge_attr=torch.cat([dist] * Fe, dim=1) if Fe else torch.empty(ei.size(1), 0))
    return cfg, params, inp


def _many_graph_sizes(seed, B=400):
    g = torch.Generator().manual_seed(seed)
    return (torch.randint(1, 4, (B,), generator=g)).tolist()


# name -> (builder kwargs of make_graph_case, or None for the CSR-built fixture), grid-cap claims checked on the CPU
_R1 = [321, 320]                # N = 641 = 5 * 128 + 1
_R127 = [400, 367]              # N = 767 = 5 * 128 + 127
_AL = [768, 512, 256]           # N = 1536 = 12 * 128
TILE_CASES = {
    "ragged_1": dict(seed=51, sizes=_R1, deg=10, C=3, Fe=4, L=2, gravity=[0, -1, 0], heavy_row=_exact_e(_R1, 10, 1)),
    "ragged_127": dict(seed=52, sizes=_R127, deg=7, C=8, Fe=0, L=2, heavy_row=_exact_e(_R127, 7, 127)),
    "aligned": dict(seed=53, sizes=_AL, deg=8, C=1, Fe=1, L=2, gravity=[0, -1, 0], heavy_row=_exact_e(_AL, 8, 0)),
    "tile_rows": None,
    "one_node": dict(seed=54, sizes=[1], deg=1, C=8, Fe=4, L=2),
    "many_graphs": dict(seed=55, sizes=_many_graph_sizes(55), deg=2, C=8, Fe=0, L=2, gravity=[0, -1, 0]),
    "no_edges": dict(seed=56, sizes=[150, 120], deg=0, C=3, Fe=1, L=2),
}


def tile_case(name):
    """(cfg, params, inp) of one fixture, as make_graph_case returns them."""
    kw = TILE_CASES[name]
    if kw is None:
        return _tile_rows_case()
    return make_graph_case(**kw)


def tile_rows_marks():
    """[(start, length, label)] of the rows tile_rows places on tile offsets."""
    return _tile_rows_layout()[1]


def tiles_per_cta(N, E, C, sms):
    """Tiles (or tile pairs, for the two-group edge backward) that the busiest CTA of each persistent kernel runs, from
    the launch rules of the kernels (grid = min(tiles, CTAs per SM * sms)) with `sms` the grid_sms cap."""
    cdiv = lambda a, b: -(-a // b)
    ne, nn, nv = cdiv(E, TM), cdiv(N, TM), cdiv(N, TM // C)
    per = lambda nt, cap: cdiv(nt, min(nt, cap)) if nt else 0
    return {
        "edge_fwd_tc (mode 1, 3 CTAs/SM)": per(ne, 3 * sms),
        "edge_fwd_tc (mode 3, 1 CTA/SM)": per(ne, sms),
        "edge_fwd fp32 (2 CTAs/SM)": per(ne, 2 * sms),
        "edge_bwd_tc4 (mode 7, tiles per group)": per(cdiv(ne, 2), sms),
        "edge_bwd fp32": per(ne, sms),
        "virtual_fwd_tc (2 CTAs/SM)": per(nv, 2 * sms),
        "virtual_bwd_tc heads / trunk": per(nv, sms),
        "virtual_fwd / _bwd fp32": per(nv, sms),
        "node_pre_fwd_tc3": per(nn, sms),
        "node_h_fwd_tc": per(nn, sms),
        "dense_bwd_tc_rows (per range)": per(nn, sms),
    }


def row_starts(edge_index, N):
    """CSR row pointer of an edge list (the stable sort by row that fegnn_graph_prep does)."""
    deg = torch.bincount(edge_index[0], minlength=N)
    return torch.cat([torch.zeros(1, dtype=torch.long), deg.cumsum(0)])
