"""Element colouring (host set-up for the deterministic EBE scatter, round-2 work): no two elements of a colour
share a node; deterministic; few colours."""
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _check(colors, flat, owner, n_nodes, ncolors):
    for c in range(ncolors):
        sel = colors[owner] == c
        nodes = flat[sel]
        assert np.unique(nodes).size == nodes.size, f"colour {c}: two elements share a node"
    assert colors.max() == ncolors - 1 and colors.min() == 0


def test_hex_colouring():
    from pcg_mpi_solver_b200.coloring import color_elements, hex_parity_colors
    nx, ny, nz = 9, 7, 6
    ez, ey, ex = np.meshgrid(np.arange(nz), np.arange(ny), np.arange(nx), indexing="ij")
    ex, ey, ez = ex.ravel(), ey.ravel(), ez.ravel()
    nodes = np.stack([((ez + ((l >> 2) & 1)) * (ny + 1) + (ey + ((l >> 1) & 1))) * (nx + 1) + (ex + (l & 1)) for l in range(8)], axis=1)
    owner = np.repeat(np.arange(nodes.shape[0]), 8)
    colors, nc = color_elements(nodes)
    _check(colors, nodes.ravel(), owner, None, nc)
    assert nc <= 27                                   # greedy independent sets; the optimum is 8
    c2, n2 = color_elements(nodes)
    assert np.array_equal(colors, c2) and nc == n2    # deterministic
    pc, pn = hex_parity_colors(ex, ey, ez)
    _check(pc, nodes.ravel(), owner, None, pn)


def test_concrete_colouring():
    from pcg_mpi_solver_b200.coloring import color_elements
    from pcg_mpi_solver_b200.model import load_mdf
    zp = os.path.join(ROOT, "oracle", "_ref", "concrete.zip")
    if not os.path.exists(zp):
        pytest.skip("concrete.zip not staged")
    m = load_mdf(zp)
    ptr = np.concatenate([m.node_offset[:, 0], m.node_offset[-1:, 1] + 1])
    colors, nc = color_elements(m.node_flat, ptr, m.n_node)
    owner = np.repeat(np.arange(m.n_elem), np.diff(ptr))
    _check(colors, m.node_flat.astype(np.int64), owner, m.n_node, nc)
    assert nc <= 80
