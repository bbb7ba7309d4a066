"""The creation-time LBVH builder (csrc/bvh_build.cu) node by node against a host reference (host_device/lbvh_ref.cpp).

Hit parity cannot see a tree's shape: the traversal's answer does not depend on it as long as the boxes are conservative.  So here the
product's build_begin + build_mesh run, through a small test-owned shared object (host_device/lbvh_harness.cu linked with bvh_build.cu,
built with the Makefile's NVFLAGS), on buffers filled with sentinels, and everything they write is compared with a reference written from
the algorithm: Morton keys, a stable sort, the Karras 2012 radix tree, bottom-up boxes, one pass of Kensler rotations, the greedy 4-wide
collapse and the outward quantisation.  The device code is built without contraction, with IEEE division and sqrt and without FTZ, and min
and max are order-independent, so the tree is deterministic up to the slot numbers the collapse hands out with atomicAdd: trees are
compared after renumbering both breadth-first.

Checked bit for bit: the MeshDev fields, the permutation (tris[p].w is the stable Morton order), v0 / e1 / e2, the normals in original
order, every node's quantised words and child refs, and BuildResult.  Checked structurally: every node in [1, live_nodes) reached once,
nodes past the tree untouched, unused slots after the used ones, the leaves partition [0, n_eff) with counts <= leaf_size.  Checked in
exact arithmetic, independent of the reference's heuristics: each decoded bound lies outside the union of its subtree's padded triangle
boxes by >= 63/64 step and <= 3 steps.  And the refit (librbrt_gpu_update.so) of a built tree with unchanged vertices rewrites the same
bytes."""
import ctypes as C
import hashlib
import os
import re
import shlex
import subprocess

import numpy as np
import pytest

from .bvh_exact import DUMMY_REF, UNUSED_WORD, BuildResultC, MeshDevC, RefitArgsC, bitseq, check_bounds, update_lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "rbrt_b200", "csrc")
HD = os.path.join(ROOT, "tests", "host_device")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
SENT = 0xA5A5A5A5
PROTO_ROOT = 0x12345


def nvflags():
    """NVFLAGS of csrc/Makefile, with $(ARCH) expanded."""
    text = open(os.path.join(CSRC, "Makefile")).read().replace("\\\n", " ")
    var = dict(re.findall(r"^(\w+)\s*=\s*(.*)$", text, re.M))
    return shlex.split(re.sub(r"\$\((\w+)\)", lambda m: var[m.group(1)], var["NVFLAGS"]))


@pytest.fixture(scope="module")
def libs(tmp_path_factory):
    tuned = [v for v in ("RBRT_SAH_PASSES", "RBRT_SAH_MIN_LEAVES") if v in os.environ]
    if tuned:                                  # the reference restates the default build: one rotation pass at nodes of >= 16 triangles
        pytest.fail(f"{tuned} set: the builder would not build the default tree the reference restates")
    d = tmp_path_factory.mktemp("lbvh")
    ref, har = str(d / "liblbvh_ref.so"), str(d / "liblbvh_harness.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fno-fast-math", "-Wall", "-fPIC", "-shared", "-o", ref,
                    os.path.join(HD, "lbvh_ref.cpp")], check=True)
    flags = [f for f in nvflags() if f not in ("-Xptxas", "-v")]
    subprocess.run([NVCC] + flags + ["-Xcompiler", "-fvisibility=hidden", "-I", CSRC, "-shared", "-Xlinker", "-Bsymbolic", "-o", har,
                    os.path.join(HD, "lbvh_harness.cu"), os.path.join(CSRC, "bvh_build.cu")], check=True, capture_output=True)
    lib = C.CDLL(ref)
    lib.lbvh_ref_build.restype = C.c_int
    return dict(ref=lib, harness=har)


def ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def reference(lib, raw, n_eff, pad_rel, leaf, sah):
    raw = np.ascontiguousarray(raw, np.float32).reshape(-1, 9)
    n = n_eff
    grid, so, res, widths = np.zeros(13, np.float32), np.zeros(6, np.float32), np.zeros(4, np.uint32), np.zeros(4096, np.uint32)
    perm, tris, nrm = np.zeros(max(n, 1), np.uint32), np.zeros((max(n, 1), 12), np.float32), np.zeros((max(n, 1), 4), np.float32)
    nodes = np.zeros((max(n - 1, 1), 16), np.uint32)
    levels = lib.lbvh_ref_build(ptr(raw), C.c_uint64(len(raw)), C.c_uint32(n), C.c_float(pad_rel), C.c_uint32(leaf), C.c_int(int(sah)), ptr(grid),
                                ptr(so), ptr(perm), ptr(tris), ptr(nrm), ptr(nodes), ptr(res), ptr(widths), len(widths))
    return dict(lo=grid[0:3], hi=grid[3:6], qorg=grid[6:9], qstep=grid[9:12], pad=grid[12], step=so[:3], org=so[3:], perm=perm[:n], tris=tris[:n],
                nrm=nrm[:n], nodes=nodes[:res[3]], live=int(res[0]), depth=int(res[1]), error=int(res[2]), tail=int(res[3]), widths=widths[:levels])


def leaf_boxes(raw, perm, pad):
    t = np.ascontiguousarray(raw, np.float32).reshape(-1, 3, 3)[perm]
    with np.errstate(all="ignore"):
        return np.fmin(t[:, 0], np.fmin(t[:, 1], t[:, 2])) - pad, np.fmax(t[:, 0], np.fmax(t[:, 1], t[:, 2])) + pad


def decode_leaf(ref):
    x = (~ref.astype(np.uint32)).astype(np.int64)
    return x >> 3, (x & 7) + 1


# ---------------------------------------------------------------- the reference alone (no GPU)
def test_reference_karras_matches_the_papers_example(libs):
    """Karras 2012, figure 3: keys 00001 00010 00100 00101 10011 11000 11001 11110 (internal node i's children; ~j is leaf j); and four
    equal keys, split by position."""
    lib = libs["ref"]
    for keys, want in (([1, 2, 4, 5, 19, 24, 25, 30], [(3, 4), (~0, ~1), (~2, ~3), (1, 2), (~4, 5), (6, ~7), (~5, ~6)]),
                       ([7, 7, 7, 7], [(1, 2), (~0, ~1), (~2, ~3)])):
        k = np.asarray(keys, np.uint64)
        ch, rg = np.zeros(2 * (len(k) - 1), np.int32), np.zeros(2 * (len(k) - 1), np.int32)
        lib.lbvh_ref_karras(ptr(k), len(k), ptr(ch), ptr(rg))
        assert [tuple(int(x) for x in c) for c in ch.reshape(-1, 2)] == want


def test_reference_small_trees_by_hand(libs):
    """Four triangles along x, the last two larger, leaf_size 1: keys ascend with x, Karras gives ((0 1) (2 3)), and the collapse expands
    the larger half first, then the other: one 4-wide root with leaves 0, 2, 3, 1.  Two triangles: one node of two leaves and two unused
    slots.  One triangle, or n <= leaf_size: no node.  Four triangles at leaf_size 3: a root of two leaves of two."""
    lib = libs["ref"]
    t = np.zeros((4, 3, 3), np.float32)
    for i in range(4):
        s = 1.0 if i < 2 else 3.0
        t[i] = [[i * 10.0, 0, 0], [i * 10.0 + s, 0, s], [i * 10.0, s, 0]]
    r = reference(lib, t, 4, 2e-5, 1, True)
    assert list(r["perm"]) == [0, 1, 2, 3] and (r["tail"], r["depth"], r["live"], r["error"]) == (1, 1, 1, 0)
    assert [int(x) for x in r["nodes"][0, 12:]] == [(~(i << 3)) & 0xFFFFFFFF for i in (0, 2, 3, 1)]
    r2 = reference(lib, t[:2], 2, 2e-5, 1, True)
    assert r2["tail"] == 1 and [int(x) for x in r2["nodes"][0, 12:]] == [0xFFFFFFFF, (~(1 << 3)) & 0xFFFFFFFF, DUMMY_REF, DUMMY_REF]
    assert list(r2["nodes"][0, 6:12]) == [UNUSED_WORD] * 6
    for n, leaf in ((1, 1), (3, 4), (4, 4)):
        r3 = reference(lib, t[:n], n, 2e-5, leaf, True)
        assert (r3["tail"], r3["depth"], r3["error"]) == (0, 0, 0)
    r4 = reference(lib, t, 4, 2e-5, 3, True)
    f, c = decode_leaf(r4["nodes"][0, 12:14])
    assert r4["tail"] == 1 and sorted(zip(f.tolist(), c.tolist())) == [(0, 2), (2, 2)]


def test_reference_trees_are_sound(libs):
    """On random meshes the reference's own output passes the structural and exact-bound checks the GPU's output must pass."""
    rng = np.random.default_rng(5)
    for leaf, sah in ((1, True), (1, False), (3, False), (8, True)):
        t = soup(2000, rng)
        r = reference(libs["ref"], t, len(t), 2e-5, leaf, sah)
        structure_and_bounds(r["nodes"], r["tail"], t, r, len(t), leaf)


def test_harness_runs_the_products_machine_code(libs):
    """Every kernel of the harness (the builder's 12 and CUB's sort kernels) has, instruction for instruction, the SASS of the same
    function in librbrt_gpu.so: the audit below tests the shipped machine code.  Hashed per function: each instruction line and the
    line after it that holds the rest of its encoding (the scheduling and control bits); not the section headers between functions."""
    cuobjdump = os.path.join(os.path.dirname(NVCC), "cuobjdump")

    def bodies(path):
        out, name, got = subprocess.run([cuobjdump, "-sass", path], capture_output=True, text=True, check=True).stdout, None, {}
        for ln in out.splitlines():
            m = re.match(r"\s+Function : (\S+)", ln)
            if m:
                name = m.group(1)
                got.setdefault(name, []).append(hashlib.md5())
            elif name and (re.match(r"\s+/\*[0-9a-f]{4,}\*/", ln) or re.fullmatch(r"\s+/\* 0x[0-9a-f]{16} \*/\s*", ln)):
                got[name][-1].update(ln.strip().encode() + b"\n")
        return {k: {h.hexdigest() for h in v} for k, v in got.items()}
    har, prod = bodies(libs["harness"]), bodies(os.path.join(ROOT, "rbrt_b200", "librbrt_gpu.so"))
    assert len(har) == 17 and sum("rbrt" in k for k in har) == 12, sorted(har)
    diff = sorted(k for k in har if har[k] != prod.get(k))
    assert not diff, diff


# ---------------------------------------------------------------- structural and exact checks of a tree (GPU's or reference's)
def canonical(words, tail, root_internal=True):
    """Renumber a tree breadth-first (children in slot order), as the reference numbers it.  Asserts that every node in [1, tail) is
    reached exactly once.  Returns (renumbered words, level bounds)."""
    n_alloc = len(words)
    seen = np.zeros(n_alloc, np.int64)
    seen[0] = 1
    order, bounds, cur = [np.zeros(1, np.int64)], [(0, 1)], np.zeros(1, np.int64)
    while True:
        refs = words[cur, 12:].view(np.int32)
        nxt = refs[refs >= 0].astype(np.int64)
        if not len(nxt):
            break
        assert nxt.max() < tail, "a child ref points past the tree"
        np.add.at(seen, nxt, 1)
        assert seen[nxt].max() == 1, "a node is reached twice"
        a = bounds[-1][1]
        bounds.append((a, a + len(nxt)))
        order.append(nxt)
        cur = nxt
    assert seen[:tail].min() == 1 and not seen[tail:].any(), "not every node in [1, live_nodes) is reached"
    order = np.concatenate(order)
    canon = np.full(n_alloc, -1, np.int64)
    canon[order] = np.arange(len(order))
    w = words[order].copy()
    r = w[:, 12:].view(np.int32)
    r[r >= 0] = canon[r[r >= 0]]
    return w, bounds


def structure_and_bounds(w, tail, raw, ref, n, leaf):
    """w: canonical words [tail, 16].  Unused slots after used ones, >= 2 used, leaves partition [0, n) with counts <= leaf, and the
    exact-arithmetic bound check against the union of each subtree's padded triangle boxes."""
    _, bounds = canonical(w, tail)
    unused = (w[:, :12].reshape(-1, 4, 3) == UNUSED_WORD).all(axis=2) & (w[:, 12:] == DUMMY_REF)
    used = ~unused
    assert (used.sum(1) >= 2).all() and (used[:, 1:] <= used[:, :-1]).all(), "unused slots must follow the used ones"
    refs = w[:, 12:].view(np.int32)
    is_leaf = used & (refs < 0)
    first, count = decode_leaf(refs[is_leaf])
    o = np.argsort(first)
    first, count = first[o], count[o]
    assert first[0] == 0 and (first[1:] == first[:-1] + count[:-1]).all() and first[-1] + count[-1] == n, "leaves do not partition [0, n_eff)"
    assert count.max() <= leaf
    llo, lhi = leaf_boxes(raw, ref["perm"], ref["pad"])
    blo, bhi = np.fmin.reduceat(llo, first, axis=0), np.fmax.reduceat(lhi, first, axis=0)
    pos = np.full(n, -1, np.int64)
    pos[first] = np.arange(len(first))
    slo, shi = np.full((tail, 4, 3), np.nan, np.float32), np.full((tail, 4, 3), np.nan, np.float32)
    nlo, nhi = np.full((tail, 3), np.nan, np.float32), np.full((tail, 3), np.nan, np.float32)
    for a, b in reversed(bounds):
        for k in range(4):
            rr = refs[a:b, k]
            lf, nd = is_leaf[a:b, k], used[a:b, k] & (rr >= 0)
            fi, _ = decode_leaf(rr[lf])
            slo[a:b, k][lf], shi[a:b, k][lf] = blo[pos[fi]], bhi[pos[fi]]
            slo[a:b, k][nd], shi[a:b, k][nd] = nlo[rr[nd]], nhi[rr[nd]]
        with np.errstate(all="ignore"):
            nlo[a:b], nhi[a:b] = np.fmin.reduce(slo[a:b], axis=1), np.fmax.reduce(shi[a:b], axis=1)
    rows, slots = np.nonzero(used)
    return check_bounds(w, rows, slots, slo[rows, slots], shi[rows, slots], ref["step"], ref["org"])


# ---------------------------------------------------------------- the GPU build
class Build:
    """One mesh through the harness: sentinel-filled output buffers, then build_begin + build_mesh + synchronise."""

    def __init__(self, libs, raw, n_eff, pad_rel, leaf, sah, host_src=False):
        import torch
        self.torch = torch
        raw = np.ascontiguousarray(raw, np.float32).reshape(-1, 9)
        self.raw, self.n_all, self.n_eff, self.pad_rel = raw, len(raw), n_eff, pad_rel
        md = MeshDevC()
        for k in range(3):
            md.lo[k] = md.hi[k] = md.qorg[k] = md.qstep[k] = 123.5
        md.tri_base, md.n_tris, md.node_base, md.root_ref, md.nrm_base, md.elem = 7, n_eff, 3, PROTO_ROOT, 5, 9
        self.proto = md
        n1 = max(n_eff, 1)
        self.n_alloc = max(n_eff - 1, 1) + 2
        sent = lambda *shape: torch.full(shape, SENT - 2 ** 32, dtype=torch.int32, device="cuda")
        self.mesh, self.tris, self.normals, self.nodes, self.res = sent(C.sizeof(MeshDevC) // 4), sent(3 * n1, 4), sent(n1, 4), sent(self.n_alloc, 16), sent(4)
        self.raw_d = torch.from_numpy(raw.reshape(-1).copy()).cuda() if len(raw) else torch.zeros(9, device="cuda")
        self.raw_h = raw.reshape(-1).copy()
        h = C.CDLL(libs["harness"])
        h.lbvh_harness_build.restype = C.c_int
        h.lbvh_harness_build.argtypes = [C.c_int, C.c_void_p, C.c_uint64, C.c_uint32, C.c_float, C.c_uint32, C.c_int, C.c_void_p] + [C.c_void_p] * 5
        torch.cuda.synchronize()
        src = ptr(self.raw_h) if host_src else self.raw_d.data_ptr()
        rc = h.lbvh_harness_build(torch.cuda.current_device(), src, self.n_all, n_eff, pad_rel, leaf, int(sah), C.byref(md), self.mesh.data_ptr(),
                                  self.tris.data_ptr(), self.normals.data_ptr(), self.nodes.data_ptr(), self.res.data_ptr())
        assert rc == 0, rc
        self.out = self.read()

    def read(self):
        b = lambda t: t.cpu().numpy()
        return dict(md=MeshDevC.from_buffer_copy(b(self.mesh).tobytes()), res=BuildResultC.from_buffer_copy(b(self.res).tobytes()),
                    tris=b(self.tris).view(np.float32), normals=b(self.normals).view(np.float32), words=b(self.nodes).view(np.uint32))


def audit(libs, raw, n_eff=None, pad_rel=2e-5, leaf=1, sah=True, host_src=False, refit=True):
    """Build on the GPU, build on the host, compare everything; returns the reference (for phase assertions)."""
    raw = np.ascontiguousarray(raw, np.float32).reshape(-1, 9)
    n = len(raw) if n_eff is None else n_eff
    g = Build(libs, raw, n, pad_rel, leaf, sah, host_src)
    r = reference(libs["ref"], raw, n, pad_rel, leaf, sah)
    md, res = g.out["md"], g.out["res"]
    for f in ("lo", "hi", "qorg", "qstep"):
        assert bitseq(np.array(getattr(md, f)), r[f]), (f, list(getattr(md, f)), r[f])
    one_leaf = n and (n <= leaf or n == 1)
    bad = r["error"] == 1
    want_root = (C.c_int32(~((0 << 3) | (n - 1))).value if one_leaf else PROTO_ROOT if (not n or bad) else 0)
    assert (md.tri_base, md.n_tris, md.node_base, md.root_ref, md.nrm_base, md.elem) == (7, 0 if bad else n, 3, want_root, 5, 9)
    assert (res.live_nodes, res.depth, res.error, res.pad) == (r["live"], r["depth"], r["error"], 0)
    t = g.out["tris"].reshape(-1, 3, 4)
    if n:
        assert np.array_equal(t[:n, 0, 3].view(np.uint32), r["perm"]), "the permutation is not the stable Morton order"
        rt = r["tris"].reshape(-1, 3, 4)
        assert bitseq(t[:n, :, :3], rt[:, :, :3]) and not t[:n, 1:, 3].view(np.uint32).any()
        assert bitseq(g.out["normals"][:n], r["nrm"])
    else:
        assert (g.out["tris"].view(np.uint32) == SENT).all() and (g.out["normals"].view(np.uint32) == SENT).all()
    words = g.out["words"]
    tail = r["tail"]
    assert (words[tail:] == SENT).all(), "nodes past the tree were written"
    if tail:
        w, _ = canonical(words, tail)
        diff = np.nonzero((w != r["nodes"]).any(1))[0]
        assert not len(diff), (f"{len(diff)} of {tail} nodes differ; first (breadth-first) {diff[0]}:\n gpu {[hex(x) for x in w[diff[0]]]}\n"
                               f" ref {[hex(x) for x in r['nodes'][diff[0]]]}")
        structure_and_bounds(w, tail, raw, r, n, leaf)
    if refit and not bad:
        identity_refit(g)
    return r



def identity_refit(g):
    """rbrt_update_refit of the built tree with the same vertices rewrites the same bytes (DESIGN.md section 10)."""
    torch = g.torch
    lib = update_lib()
    scratch = torch.zeros(lib.rbrt_update_scratch_bytes(g.n_eff), dtype=torch.uint8, device="cuda")
    a = RefitArgsC(g.raw_d.data_ptr(), g.n_all, g.n_eff, g.pad_rel, g.mesh.data_ptr(), g.tris.data_ptr(), g.normals.data_ptr(),
                   g.nodes.data_ptr(), g.res.data_ptr())
    torch.cuda.synchronize()
    assert lib.rbrt_update_refit(C.byref(a), scratch.data_ptr(), C.c_void_p(torch.cuda.current_stream().cuda_stream)) == 0
    torch.cuda.synchronize()
    after = g.read()
    assert bytes(after["md"]) == bytes(g.out["md"]) and bytes(after["res"]) == bytes(g.out["res"])
    for k in ("tris", "normals", "words"):
        assert np.array_equal(after[k].view(np.uint32), g.out[k].view(np.uint32)), f"identity refit changed {k}"


# ---------------------------------------------------------------- meshes
def soup(n, rng, centre=(5.0, 1.4, -12.5), spread=4.0, size=0.3):
    c = rng.normal(size=(n, 1, 3)) * spread + np.asarray(centre)
    return (c + rng.normal(size=(n, 3, 3)) * size).astype(np.float32)


def x_chain(levels, copies, ratio=0.9):
    """Clusters of identical triangles at x = 2^-k, shrinking in y and z: every level of the chain is one Morton bit, and the larger
    cluster is expanded first, so the chain descends one 4-wide level per bit."""
    out = []
    for k in range(levels):
        s = ratio ** k
        out += [[[0.5 ** k, -s, -s], [0.5 ** k, s, -0.5 * s], [0.5 ** k, 0.2 * s, s]]] * copies
    return np.asarray(out, np.float32)


def boundary_soup():
    rng = np.random.default_rng(2048)
    return (rng.normal(size=(20000, 1, 3)) * 4.0 + rng.normal(size=(20000, 3, 3)) * 0.3).astype(np.float32)


def phases(widths, n):
    """Levels done by each collapse phase: the single block (levels of <= 2048 nodes), ceil(log2 n) + 2 whole-GPU launches, the final block."""
    b = next((i for i, x in enumerate(widths) if x > 2048), len(widths))
    n_multi = 2
    while (1 << (n_multi - 2)) < n:
        n_multi += 1
    d = len(widths)
    return b, min(n_multi, d - b), max(d - b - n_multi, 0)


# ---------------------------------------------------------------- GPU cases
@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 2, 3, 4, 5, 7, 8, 9])
@pytest.mark.parametrize("leaf", [1, 4, 8])
def test_small_sizes(gpu, libs, n, leaf):
    rng = np.random.default_rng(100 * n + leaf)
    audit(libs, soup(n, rng), leaf=leaf)


@pytest.mark.gpu
@pytest.mark.parametrize("sah", [True, False])
@pytest.mark.parametrize("leaf", [1, 2, 3, 4, 5, 6, 7, 8])
def test_every_leaf_size_with_and_without_sah(gpu, libs, leaf, sah):
    rng = np.random.default_rng(leaf + 10 * sah)
    r = audit(libs, soup(3001, rng), leaf=leaf, sah=sah)
    assert r["tail"] > 3000 // (4 * leaf)


@pytest.mark.gpu
def test_key_structure(gpu, libs):
    rng = np.random.default_rng(3)
    one = soup(1, rng)
    audit(libs, np.broadcast_to(one, (4096, 3, 3)), leaf=1)                   # every key equal: the tie-break builds the whole tree
    audit(libs, np.broadcast_to(one, (1000, 3, 3)), leaf=3)
    two = np.concatenate([np.broadcast_to(one, (700, 3, 3)), np.broadcast_to(one + np.float32(5.0), (900, 3, 3))])
    audit(libs, two[rng.permutation(len(two))], leaf=1)                      # two distinct keys, many duplicates, interleaved
    audit(libs, two, leaf=4, sah=False)
    flat = soup(2000, rng)
    flat[:, :, 2] = np.float32(2.5)                                           # zero extent on z: inv_ext = 0
    audit(libs, flat, leaf=1)
    line = flat.copy()
    line[:, :, 1] = np.float32(-7.25)                                         # ... and on y
    audit(libs, line, leaf=2)
    audit(libs, line, leaf=1, pad_rel=0.0)                                    # no padding: the grid's slack rounds away


@pytest.mark.gpu
def test_degenerate_vertices(gpu, libs):
    rng = np.random.default_rng(4)
    t = soup(3000, rng)
    t[::7, 1, 0] = np.nan                                                     # one NaN corner
    t[::11, :, 2] = np.nan                                                    # a whole axis NaN
    t[5:40:3] = np.nan                                                        # whole NaN triangles
    t[100:200, 1] = t[100:200, 0]                                             # needles
    t[200:300, 1:] = t[200:300, :1]                                           # points: zero area
    audit(libs, t, leaf=1)
    audit(libs, t, leaf=4)
    for v in (np.inf, -np.inf):                                               # an infinite vertex: the grid's step is inf, qstep NaN
        u = soup(500, rng)
        u[17, 2, 1] = v
        audit(libs, u, leaf=1)
    audit(libs, np.full((64, 3, 3), np.nan, np.float32), leaf=1)              # nothing but NaN


@pytest.mark.gpu
def test_coordinates(gpu, libs):
    rng = np.random.default_rng(6)
    far = soup(1500, rng)
    far[:, :, 0] *= np.float32(1e12)                                          # qstep NaN on x
    audit(libs, far, leaf=2)
    audit(libs, soup(1500, rng, centre=(1e5, -1e5, 3e5), spread=30.0), leaf=1)
    audit(libs, soup(1500, rng), leaf=4, pad_rel=0.0)


@pytest.mark.gpu
def test_tails_and_host_source(gpu, libs):
    rng = np.random.default_rng(8)
    t = soup(1003, rng)
    t[1000:] += np.float32([300.0, -200.0, 400.0])                            # dropped by the tail rule: in the AABB, not in the tree
    audit(libs, t, n_eff=1000, leaf=1)
    audit(libs, t, n_eff=1000, leaf=4, host_src=True)
    audit(libs, t[:3], n_eff=0, leaf=1)                                       # nothing left: the AABB only


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1310720, 5242880])
def test_c3_and_c5_sizes(gpu, libs, n):
    rng = np.random.default_rng(n)
    r = audit(libs, soup(n, rng, spread=40.0, size=0.05), leaf=1)
    assert r["tail"] > n // 3


@pytest.mark.gpu
@pytest.mark.parametrize("n,widest", [(13236, 2048), (13240, 2049)])
def test_first_collapse_phase_boundary(gpu, libs, n, widest):
    """A level of exactly 2048 nodes is the single block's; one of 2049 goes to the whole-GPU launches."""
    r = audit(libs, boundary_soup()[:n], leaf=1)
    w = r["widths"]
    b, multi, last = phases(w, n)
    assert max(w) == widest and (b == len(w) if widest == 2048 else w[b] == 2049 and multi > 0), (list(w), b, multi)


@pytest.mark.gpu
def test_all_three_collapse_phases(gpu, libs):
    """A wide soup (a level > 2048 ends the first phase early) plus a chain deeper than the ceil(log2 n) + 2 whole-GPU launches reach:
    the final single-block phase does real work."""
    rng = np.random.default_rng(9)
    t = np.concatenate([soup(16000, rng, centre=(3.0, 0.0, 0.0), spread=0.5, size=0.01), x_chain(40, 4)])
    r = audit(libs, t, leaf=1)
    first, multi, last = phases(r["widths"], len(t))
    assert first >= 1 and multi >= 2 and last >= 2, (list(r["widths"]), first, multi, last)


# ---------------------------------------------------------------- the depth limit: 3 * depth + 2 <= RBRT_STACK (192), depth <= 63
def deep_chain(end, bits=63, copies=4, ratio=0.9):
    """A mesh in the box [-1, 1]^3 whose 4-wide tree descends one level per Morton bit, then one per halving of a cluster of `end`
    identical triangles at the centre.  Bit p of the 63 gets 4 identical triangles whose box centre has only that bit (and the
    centre's) set; each such cluster is larger than everything below it, so the collapse expands it twice and keeps the rest of the
    chain one binary level down.  Two small triangles in opposite corners fix the mesh box.  end = 1024: depth 63, the deepest tree the
    traversal stack takes; end = 2048: depth 64, refused."""
    cell = 2.0 / 2 ** 21
    shape = np.array([[-1.0, -1.0, -1.0], [1.0, 1.0, 1.0], [1.0, -1.0, 0.3]])

    def tri(c, s):
        return (np.asarray(c) + s * shape).astype(np.float32)
    out = []
    for k, p in enumerate(range(62, 62 - bits, -1)):
        c = np.full(3, 0.5 * cell)
        axis, j = 2 - p % 3, p // 3                                           # bit 3j + 2: x, 3j + 1: y, 3j: z
        c[axis] = -0.5 if j == 20 else (2 ** j + 0.5) * cell
        out += [tri(c, 0.45 * ratio ** k)] * copies
    out += [tri(np.full(3, 0.5 * cell), 0.45 * ratio ** bits)] * end
    out += [np.float32([[-1, -1, -1], [-0.9, -0.9, -0.9], [-1, -0.9, -1]]), np.float32([[1, 1, 1], [0.9, 0.9, 0.9], [1, 0.9, 1]])]
    return np.asarray(out, np.float32)


DEEPEST, REFUSED = 1024, 2048                                                 # end-cluster sizes of the depth-63 and depth-64 meshes


@pytest.mark.parametrize("end,depth", [(DEEPEST, 63), (REFUSED, 64)])
@pytest.mark.parametrize("sah", [True, False])
def test_reference_depth_limit_meshes(libs, end, depth, sah):
    """The reference's depths of the two meshes: 63 is accepted (3 * 63 + 2 = 191 <= 192), 64 refused with live_nodes 0."""
    r = reference(libs["ref"], deep_chain(end), len(deep_chain(end)), 2e-5, 1, sah)
    assert (r["depth"], r["error"]) == (depth, int(depth > 63)) and (r["live"] == 0) == (depth > 63) and r["tail"] > 0


@pytest.mark.gpu
@pytest.mark.parametrize("end", [DEEPEST, REFUSED])
@pytest.mark.parametrize("leaf,sah", [(1, True), (1, False)])
def test_depth_limit_build(gpu, libs, end, leaf, sah):
    """The builder at the limit: depth 63 published, depth 64 refused by k_build_finish (error 1, live_nodes 0, n_tris 0, root not
    published) with the tree it collapsed still equal to the reference's."""
    r = audit(libs, deep_chain(end), leaf=leaf, sah=sah)
    assert r["depth"] == (63 if end == DEEPEST else 64)


def deep_scene(end):
    import rbrt_b200 as R
    from rbrt_b200.vec3 import Vec3
    from . import scenes as S
    scene = S.spheres_scene(leaf_size=1)
    scene.triangle_meshes.append(R.TriangleMesh.from_triangles(deep_chain(end), R.Lambertian(Vec3(0.6, 0.5, 0.4))))
    return scene


def deep_rays(n, seed):
    """Rays at the deepest leaves: from points around the centre at distances 1e-3 to 3 (log-uniform), aimed at the centre cluster
    with a jitter of its own size, plus rays in random directions from the same points.  The larger clusters' triangles pass through
    the centre too, so these rays hit the chain at every depth."""
    rng = np.random.default_rng(seed)
    cell = 2.0 / 2 ** 21
    d = rng.normal(size=(n, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    o = d * 10.0 ** rng.uniform(-3, 0.5, (n, 1)) + 0.5 * cell
    target = 0.5 * cell + rng.normal(size=(n, 3)) * 3e-4
    dirs = target - o
    dirs[n // 2:] = rng.normal(size=(n - n // 2, 3))
    dirs /= np.linalg.norm(dirs, axis=1, keepdims=True)
    return np.concatenate([o, dirs], 1).astype(np.float32)


def deep_camera(w, h):
    import rbrt_b200 as R
    from rbrt_b200.vec3 import Vec3
    return R.Camera.new(Vec3(0.012, 0.009, 0.02), Vec3(0.0, 0.0, 0.0), Vec3(0.0, 1.0, 0.0), h, w, 35.0)


@pytest.mark.gpu
def test_deepest_accepted_tree_through_every_traversal(gpu, oracle):
    """Depth 63 in a scene with spheres: the three trace modes (k_trace_rays, the renderer's stage A + k_trace), intersect_device and
    occluded_device (k_query's shared-memory stack), a render (k_trace, k_tail) and the AOVs (k_aov), bit for bit against the oracle."""
    import torch
    from rbrt_b200 import _abi
    import rbrt_b200 as R
    from . import aov_ref as A
    from .test_gpu_aov import assert_passes
    from .test_gpu_query import check_closest, check_occluded
    from .test_gpu_trace import MODES, assert_same
    from .test_gpu_update import assert_images_equal
    scene = deep_scene(DEEPEST)
    assert scene.info()["num_bvh_nodes"] > 0
    rays = deep_rays(20000, 1)
    want = oracle.OracleScene.from_scene(scene).hit(rays)
    mesh_hits = want["kind"] == _abi.HIT_MESH
    assert mesh_hits.sum() > 10000, mesh_hits.sum()
    for mode in MODES:
        assert_same(scene.hit(rays, mode), want, f"depth 63, mode {mode}")
    # rays from within 2e-4 of the centre start inside the boxes of every level: each visits >= 63 nodes, pushing siblings on the way
    rng = np.random.default_rng(4)
    near = np.concatenate([rng.normal(size=(2000, 3)) * 1e-4 + 2.0 ** -21, rng.normal(size=(2000, 3))], 1).astype(np.float32)
    near[:, 3:] /= np.linalg.norm(near[:, 3:], axis=1, keepdims=True)
    st, sq = {}, {}
    assert_same(scene.hit(near, _abi.TRACE_BVH, stats=st), oracle.OracleScene.from_scene(scene).hit(near), "depth 63, rays from the centre")
    scene.intersect_device(torch.from_numpy(near).cuda(), stats=sq)
    assert st["node_visits"] >= 63 * len(near) and sq["node_visits"] >= 63 * len(near), (st["node_visits"], sq["node_visits"])
    rays = np.concatenate([rays, near])
    hits = check_closest(scene, rays, "depth 63", oracle)
    check_occluded(scene, rays, hits, "depth 63")
    torch.cuda.synchronize()
    cam = deep_camera(40, 30)
    ref = oracle.OracleScene.from_scene(scene).render_hdr(cam.to_c(), 2, _abi.RenderOptsC(seed=5))
    assert_images_equal(R.render_scene_hdr(cam, 2, scene, seed=5), ref, "depth 63 render")
    assert_passes(R.render_aovs(cam, 2, scene, seed=5), A.expected(cam, 2, scene, seed=5, oracle=oracle), "depth 63 AOVs")


@pytest.mark.gpu
def test_refused_tree_through_the_product(gpu):
    """Depth 64: the mesh is left out and every call that reads the scene reports it — scene info, render, trace_rays, AOVs, both
    queries, and a refit of the refused mesh.  A mesh rebuilt into a too-deep tree (RBRT_UPDATE_REBUILD) is reported the same way."""
    import torch
    import rbrt_b200 as R
    from rbrt_b200 import _abi
    msg = "mesh 0: BVH deeper than the traversal stack allows"
    rays = deep_rays(256, 2)
    cam = deep_camera(8, 6)
    deep = deep_chain(REFUSED)

    def refused(call, exc=_abi.RbrtGpuError):
        with pytest.raises(exc, match=msg) as e:
            call()
        assert not isinstance(e.value, _abi.RbrtGpuError) or e.value.code == _abi.E_INVALID

    scene = deep_scene(REFUSED)
    refused(scene.info)
    refused(lambda: R.render_scene_hdr(cam, 1, scene, seed=1))
    refused(lambda: scene.hit(rays))
    refused(lambda: R.render_aovs(cam, 1, scene, seed=1))
    t = torch.from_numpy(rays).cuda()
    refused(lambda: scene.intersect_device(t), ValueError)
    refused(lambda: scene.occluded_device(t), ValueError)
    refused(lambda: scene.update_mesh(0, deep))
    refused(lambda: scene.update_mesh(0, deep, rebuild=True))
    scene.close()
    rng = np.random.default_rng(3)
    shallow = soup(len(deep), rng, centre=(0.0, 0.0, 0.0), spread=0.3, size=0.05)
    scene = deep_scene(DEEPEST)
    scene.triangle_meshes[0] = R.TriangleMesh.from_triangles(shallow, scene.triangle_meshes[0].material)
    scene.info()
    scene.hit(rays)
    scene.update_mesh(0, deep, rebuild=True)                                  # enqueued: the depth is known when the rebuild completes
    refused(scene.info)
    refused(lambda: scene.hit(rays))
    refused(lambda: R.render_scene_hdr(cam, 1, scene, seed=1))
    scene.close()
