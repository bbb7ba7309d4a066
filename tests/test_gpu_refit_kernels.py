"""The refit kernels of librbrt_gpu_update.so (csrc/update.cu) on buffers this test owns, against a numpy reference.

rbrt_update_refit(const RefitArgs*, scratch, stream) is called through ctypes on torch CUDA tensors: the raw vertices, the MeshDev record,
the triangle records, the normals, the 4-wide nodes and the BuildResult.  The trees are built here in the product's node format
(intersect.cuh): balanced ones with two to four children per node, chains thousands of nodes deep (long last-arriver chains in
k_upd_nodes), unused slots in every position, leaves of 1 to 8 triangles, the root as a leaf, N_eff = 0 and dropped tail triangles,
and 1.31 M and 5.24 M triangles (many blocks racing up the tree).

Checked bit for bit: the mesh AABB, MeshDev lo / hi / qorg / qstep (NaN where the step exceeds RBRT_QSTEP_MAX), the padding and the grid
in the scratch's RefitParams (with the 2^-21 * (mx + 1000) floor, and pad_rel = 0), the triangle records with the original index kept in
.w, the normals (norm3's float32 op sequence), the child refs, the unused-slot words and every node past live_nodes.

Checked in exact arithmetic: each quantised child bound, decoded as qorg + q * qstep, lies outside the union of its subtree's padded
triangle boxes by at least 63/64 of a grid step (the margin the traversal's slab test relies on) and at most 3 steps beyond it.  A leaf
whose triangles are NaN on an axis gets the build's [0, 0] words there."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from .bvh_exact import DUMMY_REF, NAN_BITS, QSTEP_MAX, UNUSED_WORD, BuildResultC, MeshDevC, RefitArgsC, bitseq, check_bounds, update_lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "rbrt_b200", "csrc")
F32_MAX = np.float32(3.4028235e38)


PARAMS_AT = 64                                 # RefitParams {pad, org[3], step[3]} at scratch + 64 (rbrt_update_refit)

LAYOUT_PROBE = r"""
#include "update.cuh"
#include <cstddef>
#include <cstdio>
using namespace rbrt;
int main() {
    printf("MeshDev %zu %zu %zu %zu %zu %zu %zu %zu %zu %zu\n", sizeof(MeshDev), offsetof(MeshDev, lo), offsetof(MeshDev, hi), offsetof(MeshDev, tri_base),
           offsetof(MeshDev, n_tris), offsetof(MeshDev, node_base), offsetof(MeshDev, root_ref), offsetof(MeshDev, nrm_base), offsetof(MeshDev, qorg),
           offsetof(MeshDev, qstep));
    printf("BuildResult %zu %zu %zu %zu\n", sizeof(BuildResult), offsetof(BuildResult, live_nodes), offsetof(BuildResult, depth), offsetof(BuildResult, error));
    printf("RefitArgs %zu %zu %zu %zu %zu %zu %zu %zu %zu %zu\n", sizeof(RefitArgs), offsetof(RefitArgs, raw), offsetof(RefitArgs, n_all),
           offsetof(RefitArgs, n_eff), offsetof(RefitArgs, pad_rel), offsetof(RefitArgs, mesh), offsetof(RefitArgs, tris), offsetof(RefitArgs, normals),
           offsetof(RefitArgs, nodes), offsetof(RefitArgs, res));
}
"""


def test_struct_layouts_match_the_headers(tmp_path):
    """The ctypes restatements above have the sizes and offsets the compiler gives the C++ structs (no GPU needed)."""
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    src, exe = tmp_path / "probe.cu", tmp_path / "probe"
    src.write_text(LAYOUT_PROBE)
    subprocess.run([nvcc, "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-I", CSRC, "-o", str(exe), str(src)], check=True)
    got = {ln.split()[0]: [int(x) for x in ln.split()[1:]] for ln in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines()}
    m = MeshDevC
    assert got["MeshDev"] == [C.sizeof(m), m.lo.offset, m.hi.offset, m.tri_base.offset, m.n_tris.offset, m.node_base.offset, m.root_ref.offset,
                              m.nrm_base.offset, m.qorg.offset, m.qstep.offset]
    b = BuildResultC
    assert got["BuildResult"] == [C.sizeof(b), b.live_nodes.offset, b.depth.offset, b.error.offset]
    a = RefitArgsC
    assert got["RefitArgs"] == [C.sizeof(a), a.raw.offset, a.n_all.offset, a.n_eff.offset, a.pad_rel.offset, a.mesh.offset, a.tris.offset,
                                a.normals.offset, a.nodes.offset, a.res.offset]


# ---------------------------------------------------------------- trees in the product's node format, built on the host
def leaf_ref(first, count):
    return (~((first << 3) | (count - 1))) & 0xFFFFFFFF


class Tree:
    """Nodes in creation order (children before parents, the root last) as CSR lists of child items: item < 0 is leaf -item - 1, item >= 0
    is node `item` (creation order); `levels` = ranges of creation ids whose children are all older.  `index` maps creation id -> node
    index in the buffer (the root is node 0, the others shuffled)."""

    def __init__(self, n_eff, leaf_max, rng, chain=False, fixed_leaf=False):
        sizes = np.full(n_eff, leaf_max) if fixed_leaf else rng.integers(1, leaf_max + 1, max(n_eff, 1))
        cut = np.cumsum(sizes)
        self.first = np.concatenate([[0], cut[cut < n_eff]]).astype(np.int64)
        self.count = np.diff(np.append(self.first, n_eff))
        items = -np.arange(len(self.first)) - 1
        ptr, kids, self.levels = [0], [], []
        n = 0
        if chain:                                                            # node k = {node k - 1} + 1..3 leaves: depth ~ leaves / 2
            cur, nxt = items[-1], len(items) - 1
            while nxt > 0:
                take = min(int(rng.integers(1, 4)), nxt)
                group = np.concatenate([[cur], items[nxt - take:nxt]])
                nxt -= take
                kids.append(group); ptr.append(ptr[-1] + len(group)); self.levels.append((n, n + 1))
                cur, n = n, n + 1
        else:
            while len(items) > 1:
                g = rng.integers(2, 5, len(items))
                starts = np.concatenate([[0], np.cumsum(g)])
                starts = starts[starts < len(items)]
                if len(items) - starts[-1] == 1 and len(starts) > 1:        # no one-child node: merge into, or borrow from, the previous group
                    if starts[-1] - starts[-2] <= 3:
                        starts = starts[:-1]
                    else:
                        starts[-1] -= 1
                sz = np.diff(np.append(starts, len(items)))
                kids.append(items); ptr.extend((ptr[-1] + np.cumsum(sz)).tolist())
                self.levels.append((n, n + len(starts)))
                items = n + np.arange(len(starts))
                n += len(starts)
        self.ptr = np.asarray(ptr, np.int64)
        self.kids = np.concatenate(kids).astype(np.int64) if kids else np.zeros(0, np.int64)
        self.n_nodes = n
        self.depth = len(self.levels)
        perm = rng.permutation(np.arange(1, n)) if n > 1 else np.zeros(0, np.int64)
        self.index = np.zeros(n, np.int64)
        if n:
            self.index[:n - 1] = perm
            self.index[n - 1] = 0
        nk = np.diff(self.ptr)
        self.slot_perm = rng.permuted(np.tile(np.arange(4), (n, 1)), axis=1)     # child i of a node sits in slot slot_perm[i]: unused slots anywhere
        self.child_node = np.repeat(np.arange(n), nk)
        self.child_slot = self.slot_perm[self.child_node, np.arange(len(self.kids)) - self.ptr[self.child_node]] if n else np.zeros(0, np.int64)

    def root_ref(self):
        return 0 if self.n_nodes else leaf_ref(0, int(self.count[0]))

    def node_words(self, n_alloc, rng):
        """[n_alloc, 16] uint32: random box words in the used slots (the refit overwrites them), the unused-slot pattern, the child refs;
        rows past the tree hold random words the refit must leave alone."""
        w = rng.integers(0, 2 ** 32, (n_alloc, 16), dtype=np.uint64).astype(np.uint32)
        if not self.n_nodes:
            return w
        j = self.index
        w[j, :12] = UNUSED_WORD
        w[j, 12:] = DUMMY_REF
        rows = j[self.child_node]
        ref = np.zeros(len(self.kids), np.uint64)
        leaf = self.kids < 0
        li = -self.kids[leaf] - 1
        ref[leaf] = leaf_ref(self.first[li], self.count[li])
        ref[~leaf] = j[self.kids[~leaf]]
        w[rows, 12 + self.child_slot] = ref.astype(np.uint32)
        for a in range(3):
            w[rows, 3 * self.child_slot + a] = rng.integers(0x10000, 2 ** 32, len(rows), dtype=np.uint64).astype(np.uint32)
        return w

    def node_boxes(self, leaf_lo, leaf_hi):
        """Float boxes of every leaf and node (creation order) from the padded triangle boxes: fminf / fmaxf, NaN ignored unless all are."""
        blo, bhi = np.fmin.reduceat(leaf_lo, self.first, axis=0), np.fmax.reduceat(leaf_hi, self.first, axis=0)
        nlo, nhi = np.zeros((self.n_nodes, 3), np.float32), np.zeros((self.n_nodes, 3), np.float32)

        def gather(items, src_leaf, src_node):
            return np.where((items < 0)[:, None], src_leaf[np.where(items < 0, -items - 1, 0)], src_node[np.where(items >= 0, items, 0)])
        for a, b in self.levels:
            s, e = self.ptr[a], self.ptr[b]
            it = self.kids[s:e]
            off = self.ptr[a:b] - s
            nlo[a:b] = np.fmin.reduceat(gather(it, blo, nlo), off, axis=0)
            nhi[a:b] = np.fmax.reduceat(gather(it, bhi, nhi), off, axis=0)
        return gather(self.kids, blo, nlo), gather(self.kids, bhi, nhi)                                                      # per child (CSR order)


# ---------------------------------------------------------------- the reference
def f2ord(x):
    b = np.ascontiguousarray(x, np.float32).view(np.int32).astype(np.int64)
    return np.where(b >= 0, b, b ^ 0x7FFFFFFF)


def ord2f(i):
    i = np.int64(i)
    b = i if i >= 0 else i ^ 0x7FFFFFFF
    return np.array([b], np.int64).astype(np.int32).view(np.float32)[0]


def reference(raw, n_eff, pad_rel, orig):
    """k_upd_aabb + k_upd_setup + k_upd_tris in numpy float32, op for op."""
    f = np.float32
    v = raw.reshape(-1, 3)
    lo, hi = np.zeros(3, f), np.zeros(3, f)
    for k in range(3):
        x = v[:, k][~np.isnan(v[:, k])]
        o = f2ord(x)
        lo[k] = ord2f(min([int(f2ord([F32_MAX])[0])] + ([int(o.min())] if len(o) else [])))       # k_upd_aabb_init: +-FLT_MAX
        hi[k] = ord2f(max([int(f2ord([-F32_MAX])[0])] + ([int(o.max())] if len(o) else [])))
    with np.errstate(all="ignore"):
        mx = f(0.0)
        for k in range(3):
            mx = np.fmax(mx, np.fmax(np.abs(lo[k]), np.abs(hi[k])))
            mx = np.fmax(mx, f(hi[k] - lo[k]))
        pad = np.fmax(f(pad_rel) * mx, f(4.7683716e-7) * f(mx + f(1000.0))) if f(pad_rel) > 0 else f(0.0)
        org, step = np.zeros(3, f), np.zeros(3, f)
        for k in range(3):
            ext = f(f(hi[k] + pad) - f(lo[k] - pad))
            s = f(ext / f(65500.0))
            if not s > f(1e-30):
                s = f(1e-30)
            step[k], org[k] = s, f(f(lo[k] - pad) - f(8.0) * s)
        qstep = np.where(step <= QSTEP_MAX, step, np.array([NAN_BITS], np.uint32).view(np.float32)[0]).astype(f)
        if not n_eff:
            qstep, qorg = np.zeros(3, f), np.zeros(3, f)
        else:
            qorg = org.copy()
        t = raw[orig].reshape(-1, 3, 3)
        a, b, c = t[:, 0], t[:, 1], t[:, 2]
        e1, e2 = b - a, c - a
        cx = e1[:, 1] * e2[:, 2] - e1[:, 2] * e2[:, 1]
        cy = e1[:, 2] * e2[:, 0] - e1[:, 0] * e2[:, 2]
        cz = e1[:, 0] * e2[:, 1] - e1[:, 1] * e2[:, 0]
        ln = np.sqrt((cx * cx + cy * cy) + cz * cz)
        nrm = np.stack([cx / ln, cy / ln, cz / ln], 1)
        leaf_lo = np.fmin(a, np.fmin(b, c)) - pad
        leaf_hi = np.fmax(a, np.fmax(b, c)) + pad
    return dict(lo=lo, hi=hi, pad=pad, org=org, step=step, qorg=qorg, qstep=qstep, a=a, e1=e1, e2=e2, nrm=nrm, leaf_lo=leaf_lo, leaf_hi=leaf_hi)


# ---------------------------------------------------------------- the driver
@pytest.fixture(scope="module")
def upd(gpu):
    return update_lib()


class Mesh:
    """The device buffers of one mesh (torch CUDA tensors), laid out as api.cu lays out a scene's mesh."""

    def __init__(self, tree, n_all, n_eff, rng, orig=None):
        import torch
        self.torch, self.tree, self.n_all, self.n_eff = torch, tree, n_all, n_eff
        self.orig = rng.permutation(n_eff).astype(np.uint32) if orig is None else orig          # tree position -> original triangle (Morton order)
        rec = rng.standard_normal((max(n_eff, 1) * 3, 4)).astype(np.float32)
        rec[0::3, 3] = self.orig.view(np.float32) if n_eff else 0
        self.n_alloc = max(n_eff - 1, 1) + 3
        self.words0 = tree.node_words(self.n_alloc, rng)
        md = MeshDevC()
        for k in range(3):
            md.lo[k] = md.hi[k] = md.qorg[k] = md.qstep[k] = 123.5
        md.tri_base, md.n_tris, md.node_base, md.root_ref, md.nrm_base, md.elem = 7, n_eff, 3, C.c_int32(tree.root_ref()).value, 5, 9
        self.md0 = bytes(md)
        res = BuildResultC(tree.n_nodes, tree.depth, 0, 0)
        dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
        self.mesh = dev(np.frombuffer(self.md0, np.uint8).copy())
        self.tris = dev(rec)
        self.normals = dev(rng.standard_normal((max(n_eff, 1), 4)).astype(np.float32))
        self.normals0 = self.normals.cpu().numpy()
        self.nodes = dev(self.words0.view(np.int32))
        self.res = dev(np.frombuffer(bytes(res), np.uint8).copy())

    def refit(self, lib, raw, pad_rel):
        torch = self.torch
        raw_d = torch.from_numpy(np.ascontiguousarray(raw, np.float32).reshape(-1)).cuda() if self.n_all else torch.zeros(9, device="cuda")
        scratch = torch.full((lib.rbrt_update_scratch_bytes(self.n_eff),), 0xA5, dtype=torch.uint8, device="cuda")
        a = RefitArgsC(raw_d.data_ptr(), self.n_all, self.n_eff, pad_rel, self.mesh.data_ptr(), self.tris.data_ptr(), self.normals.data_ptr(),
                       self.nodes.data_ptr(), self.res.data_ptr())
        torch.cuda.synchronize()
        assert lib.rbrt_update_refit(C.byref(a), scratch.data_ptr(), C.c_void_p(torch.cuda.current_stream().cuda_stream)) == 0
        torch.cuda.synchronize()
        md = MeshDevC.from_buffer_copy(self.mesh.cpu().numpy().tobytes())
        prm = scratch[PARAMS_AT:PARAMS_AT + 28].cpu().numpy().view(np.float32)
        return dict(md=md, pad=prm[0], org=prm[1:4], step=prm[4:7], tris=self.tris.cpu().numpy(), normals=self.normals.cpu().numpy(),
                    words=self.nodes.cpu().numpy().view(np.uint32))


def run_and_check(lib, mesh, raw, pad_rel):
    """One refit of `mesh` to `raw` [n_all, 3, 3], everything compared with the reference; returns the number of bounds checked."""
    out = mesh.refit(lib, raw, pad_rel)
    ref = reference(np.ascontiguousarray(raw, np.float32).reshape(-1, 9), mesh.n_eff, pad_rel, mesh.orig)
    md = out["md"]
    assert bitseq(np.array(md.lo), ref["lo"]) and bitseq(np.array(md.hi), ref["hi"]), (list(md.lo), list(md.hi), ref["lo"], ref["hi"])
    assert bitseq(np.array(md.qorg), ref["qorg"]) and bitseq(np.array(md.qstep), ref["qstep"]), (list(md.qorg), list(md.qstep), ref["qorg"], ref["qstep"])
    m0 = MeshDevC.from_buffer_copy(mesh.md0)
    assert (md.tri_base, md.n_tris, md.node_base, md.root_ref, md.nrm_base, md.elem) == (m0.tri_base, m0.n_tris, m0.node_base, m0.root_ref,
                                                                                          m0.nrm_base, m0.elem)
    assert bitseq(out["pad"], ref["pad"]), (out["pad"], ref["pad"])
    if mesh.n_eff:
        assert bitseq(out["org"], ref["org"]) and bitseq(out["step"], ref["step"]), (out["org"], out["step"], ref["org"], ref["step"])
        t = out["tris"].reshape(-1, 3, 4)
        assert bitseq(t[:, 0, :3], ref["a"]) and bitseq(t[:, 1, :3], ref["e1"]) and bitseq(t[:, 2, :3], ref["e2"])
        assert np.array_equal(t[:, 0, 3].view(np.uint32), mesh.orig) and not t[:, 1:, 3].view(np.uint32).any()     # orig kept, .w of e1 / e2 zero
        assert bitseq(out["normals"][mesh.orig, :3], ref["nrm"]) and not out["normals"][:, 3].view(np.uint32).any()
    w, w0 = out["words"], mesh.words0
    tr = mesh.tree
    assert np.array_equal(w[:, 12:], w0[:, 12:]), "child refs changed"
    if tr.n_nodes:
        used = np.zeros((mesh.n_alloc, 4), bool)
        used[tr.index[tr.child_node], tr.child_slot] = True
        idle = np.repeat(~used, 3, axis=1)
        live = np.zeros(mesh.n_alloc, bool)
        live[tr.index] = True
        assert np.array_equal(w[:, :12][live][idle[live]], w0[:, :12][live][idle[live]]), "unused-slot words changed"
        assert np.array_equal(w[~live], w0[~live]), "nodes past live_nodes changed"
        clo, chi = tr.node_boxes(ref["leaf_lo"], ref["leaf_hi"])
        return check_bounds(w, tr.index[tr.child_node], tr.child_slot, clo, chi, ref["step"], ref["org"])
    assert np.array_equal(w, w0), "a mesh without nodes had its node buffer written"
    return 0


def soup(n, rng, centre=(5.0, 1.4, -12.5), spread=4.0, size=0.3):
    c = rng.normal(size=(n, 1, 3)) * spread + np.asarray(centre)
    return (c + rng.normal(size=(n, 3, 3)) * size).astype(np.float32)


def deform(t, rng):
    return (t * np.float32(1.3) + rng.normal(size=t.shape).astype(np.float32) * np.float32(0.2) + np.float32([40.0, -3.0, 7.0])).astype(np.float32)



@pytest.mark.gpu
@pytest.mark.parametrize("leaf", [1, 2, 3, 4, 5, 6, 7, 8])
def test_balanced_trees_every_leaf_size(upd, leaf):
    rng = np.random.default_rng(leaf)
    n = 3001
    tree = Tree(n, leaf, rng, fixed_leaf=leaf > 4)
    mesh = Mesh(tree, n, n, rng)
    t = soup(n, rng)
    assert run_and_check(upd, mesh, t, 2e-5) > 3 * (n // leaf)
    assert run_and_check(upd, mesh, deform(t, rng), 2e-5) > 0                 # a second refit reads the words the first one wrote
    assert run_and_check(upd, mesh, t, 0.0) > 0                               # pad_rel = 0: no padding at all


@pytest.mark.gpu
@pytest.mark.parametrize("leaf_max", [1, 3, 8])
def test_chains_thousands_of_nodes_deep(upd, leaf_max):
    rng = np.random.default_rng(40 + leaf_max)
    n = 4000 * (leaf_max + 1)
    tree = Tree(n, leaf_max, rng, chain=True)
    assert tree.depth >= 2000 and tree.n_nodes == tree.depth, tree.depth   # one last-arriver walks the whole chain
    mesh = Mesh(tree, n, n, rng)
    t = soup(n, rng, spread=30.0)
    assert run_and_check(upd, mesh, t, 2e-5) > 2 * tree.n_nodes
    assert run_and_check(upd, mesh, deform(t, rng), 2e-5) > 0


@pytest.mark.gpu
def test_small_meshes_root_leaf_and_dropped_tail(upd):
    rng = np.random.default_rng(7)
    for n_all, n_eff, leaf in ((3, 0, 1), (5, 5, 8), (1, 1, 1), (2, 2, 1), (9, 8, 2), (43, 40, 4), (321, 320, 1)):
        tree = Tree(n_eff, leaf, rng, fixed_leaf=True)
        assert (tree.n_nodes == 0) == (n_eff <= leaf)
        mesh = Mesh(tree, n_all, n_eff, rng)
        t = soup(n_all, rng)
        t[n_eff:] += np.float32([300.0, -200.0, 400.0])                       # dropped by the tail rule: in the AABB, not in the tree
        run_and_check(upd, mesh, t, 2e-5)


@pytest.mark.gpu
def test_nan_and_collapsed_vertices(upd):
    rng = np.random.default_rng(11)
    n = 2000
    tree = Tree(n, 4, rng)
    mesh = Mesh(tree, n, n, rng)
    t = soup(n, rng)
    t[::7, 1, 0] = np.nan                                                     # one NaN corner
    t[::11, :, 2] = np.nan                                                    # NaN on a whole axis
    t[:64] = np.nan                                                           # whole leaves of NaN triangles, triangle 0 among them
    assert run_and_check(upd, mesh, t, 2e-5) > 0
    assert run_and_check(upd, mesh, np.broadcast_to(np.float32([5.0, 1.4, -12.5]), t.shape).copy(), 2e-5) > 0    # every vertex on one point
    assert run_and_check(upd, mesh, np.broadcast_to(np.float32([5.0, 1.4, -12.5]), t.shape).copy(), 0.0) > 0     # ... with no padding: step 1e-30
    assert run_and_check(upd, mesh, np.full(t.shape, np.nan, np.float32), 2e-5) == 0                             # nothing but NaN


@pytest.mark.gpu
@pytest.mark.parametrize("far", [1e11, 3e11, 1e12, 1e20, 1e30, 2e38, 3.4e38, np.inf, -np.inf])
def test_extreme_extents(upd, far):
    """The meshes of test_device_source_on_host.py::test_traversal_at_extreme_mesh_extents: the grid of the far axis (and from 1e20 on, of all
    three) exceeds RBRT_QSTEP_MAX and MeshDev.qstep must read NaN there; the other axes keep a grid whose bounds contain the boxes."""
    from . import scenes as S
    rng = np.random.default_rng(3)
    t = S.far_triangle_mesh(far, 0)
    n = len(t)
    tree = Tree(n, 4, rng)
    mesh = Mesh(tree, n, n, rng)
    run_and_check(upd, mesh, soup(n, rng), 2e-5)
    checked = run_and_check(upd, mesh, t, 2e-5)
    qstep = np.array(MeshDevC.from_buffer_copy(mesh.mesh.cpu().numpy().tobytes()).qstep, np.float32)
    assert np.isnan(qstep[0]) == (abs(far) >= 3e11) and (checked > 0) == (abs(far) < 1e20), (far, qstep, checked)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1310720, 5242880])
def test_c3_and_c5_scale(upd, n):
    """C3 / C5 triangle counts: thousands of blocks race up a balanced tree of ~0.4 M / 1.7 M nodes."""
    rng = np.random.default_rng(n)
    tree = Tree(n, 8, rng)
    assert tree.n_nodes > n // 16, tree.n_nodes
    mesh = Mesh(tree, n, n, rng)
    t = soup(n, rng, spread=40.0, size=0.05)
    assert run_and_check(upd, mesh, t, 2e-5) > 3 * tree.n_nodes
    assert run_and_check(upd, mesh, deform(t, rng), 2e-5) > 3 * tree.n_nodes
