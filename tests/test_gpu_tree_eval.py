"""The OCTREE primitive of an SDF program (what UnionSDF / SubtractSDF / IntersectSDF rebuild from) evaluates a tree one
point per thread; hpsdf_query evaluates it a warp at a time. Both must give the same bits, DBL_MAX outside the root, for
leaves of every degree a MemoryBlock may hold and for trees whose depth-4 level is not complete (no top table)."""
import numpy as np
import pytest

from cases import CASES, root_points
from common import product_cfg

NO_CHILD = np.uint64(0xFFFFFFFFFFFFFFFF)
NODE_DT = np.dtype({"names": ["child", "cstart", "deg", "depth"], "formats": ["<u8", "<u8", "u1", "u1"],
                    "offsets": [0, 32, 40, 48], "itemsize": 56})


def rewritten_block(hp, block, collapse, seed):
    """`block` with leaf i of degree i % 13 and seeded random coefficients. With `collapse`, every fifth depth-2 node
    becomes a leaf as well; its subtree stays in the block, unreachable, and the tree no longer reaches depth 4 everywhere."""
    block = bytes(block)
    b = hp.parse_block(block)
    off = 16 + 8 * b["n_coeffs"]
    nodes = np.frombuffer(bytearray(block[off:off + 56 * b["n_nodes"]]), NODE_DT)
    if collapse:
        cut = np.flatnonzero((nodes["depth"] == 2) & (nodes["child"] != NO_CHILD))[::5]
        assert len(cut)
        nodes["child"][cut] = NO_CHILD
    leaves = np.flatnonzero(nodes["child"] == NO_CHILD)
    deg = np.arange(len(leaves)) % 13
    count = np.array([hp.COEFF_COUNT[d] for d in deg], np.uint64)
    nodes["deg"][leaves] = deg
    nodes["cstart"][leaves] = np.concatenate(([0], np.cumsum(count)[:-1]))
    coeffs = np.random.default_rng(seed).standard_normal(int(count.sum()))
    return np.uint64(len(coeffs)).tobytes() + coeffs.tobytes() + np.uint64(len(nodes)).tobytes() + nodes.tobytes() + block[-80:]


@pytest.mark.gpu
@pytest.mark.parametrize("collapse", [False, True], ids=["top_table", "no_top_table"])
def test_octree_primitive_matches_query_bitwise(hp, collapse):
    cfg, prog = product_cfg(hp, "csg_small")
    src = hp.Octree()
    src.Create(cfg, prog)
    block = rewritten_block(hp, src.ToMemoryBlockBytes(), collapse, seed=7)
    t = hp.Octree()
    t.FromMemoryBlock(hp.MemoryBlock.frombytes(block))
    nodes = hp.parse_block(block)["nodes"]
    leaves = nodes["child"] == NO_CHILD
    assert set(nodes["deg"][leaves]) == set(range(13))
    assert (nodes["depth"][leaves] < 4).any() == collapse

    k = CASES["csg_small"]["cfg"]
    lo, hi = np.asarray(k["root_min"], np.float64), np.asarray(k["root_max"], np.float64)
    corners = np.array([[x, y, z] for x in (lo[0], hi[0]) for y in (lo[1], hi[1]) for z in (lo[2], hi[2])])
    pts = np.concatenate([root_points(k, 1 << 18, seed=3, margin=0.1), corners, corners * (1 + 1e-9), corners * (1 + 1e-6)])
    q = t.Query(pts)
    v = hp.SdfProgram([("octree", [], t)]).eval(pts)
    outside = q == hp.DBL_MAX
    assert outside.any() and (~outside).any()
    assert np.array_equal(v.view(np.uint64), q.view(np.uint64)), \
        "%d of %d points differ, largest difference %g" % ((v != q).sum(), len(q), np.abs(v - q)[~outside].max())
