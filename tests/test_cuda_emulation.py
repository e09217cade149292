"""CPU-side check of CUDA kernel LOGIC without a GPU: the kernel source of csrc/bvh.cu, csrc/bvh.cuh and
csrc/datacosts.cu is compiled unchanged by g++ against tests/cpp/cuda_emul.h (threads run one after the other)
and compared with the oracle.

Why: none of the smooth sphere / terrain scenes produces a single occluded (face, view) pair, so on those the
visibility rays only ever prove "no false hits".  The `occ` scenes (floating plates in front of a displaced
sphere) make ~30 % of the candidates fail the geometric visibility test; this file checks the device LBVH build,
the any-hit traversal and the candidate / ray-bitmap / quality / compaction kernels on them.  It proves nothing
about races or memory ordering -- tests/test_zz_gpu_occlusion.py runs the same scenes on the real device.

Kernels that synchronise (csrc/mrf.cu: cooperative k_forest with grid.sync, the k_up / k_down dataflow sweeps over
per-node flags; csrc/seam.cu: the persistent cooperative PCG) run on tests/cpp/cuda_fiber.h: one ucontext fiber per
CUDA thread, barriers / shuffles / grid.sync as yield points, deterministic round-robin scheduling.  `occ` adds what
the smooth scenes lack there too: 37 faces no view sees (label 0) and ten separate mesh components.
"""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import reference_golden as G  # noqa: E402

CSRC = os.path.join(ROOT, "mvs-texturing_b200", "csrc")
OUT = os.path.join(ROOT, "tests", "cpp", "_emul")
CUDA_INC = "/usr/local/cuda/include"

pytestmark = pytest.mark.skipif(not os.path.exists(os.path.join(CUDA_INC, "cuda_runtime.h")),
                                reason="CUDA headers not installed")


def _kernel_part(cu_file, host_entry, drop=None, remove_line=None, close=1):
    """Text of a .cu file up to its first host entry point (the part that holds the kernels), unchanged except for
    the CUB include and, optionally, a span [drop[0], drop[1]) that cannot be compiled for the host (CUB calls, inline
    PTX) and one line (`extern __shared__`).  `close` = number of namespaces still open at the cut."""
    src = open(os.path.join(CSRC, cu_file)).read()
    head = src.split(host_entry)[0].replace("#include <cub/cub.cuh>", "")
    for span in ([drop] if drop and isinstance(drop[0], str) else (drop or [])):
        a, b = head.index(span[0]), head.index(span[1])
        head = head[:a] + head[b:]
    if remove_line:
        assert remove_line in head
        head = head.replace(remove_line, "")
    return head + "}  // namespace\n" * close


@pytest.fixture(scope="module")
def emul():
    os.makedirs(OUT, exist_ok=True)
    with open(os.path.join(OUT, "bvh_kernels.inc"), "w") as f:
        f.write(_kernel_part("bvh.cu", "int build_bvh("))
    with open(os.path.join(OUT, "datacosts_kernels.inc"), "w") as f:
        f.write(_kernel_part("datacosts.cu", "static int finish_candidates(", ("int cub_exclusive_sum_u64", "namespace {")))
    with open(os.path.join(OUT, "mrf_kernels.inc"), "w") as f:
        f.write(_kernel_part("mrf.cu", "Mrf make_mrf(b2tex_ctx",
                             [("// ---- shared-memory / async-copy primitives", "// ---- end of primitives ----"),
                              ("// ---- system-scope flag primitives", "// ---- end of flag primitives ----")],
                             "    extern __shared__ __align__(16) unsigned char tree_dyn[];\n", close=2))
    with open(os.path.join(OUT, "seam_kernels.inc"), "w") as f:
        f.write(_kernel_part("seam.cu", "int seam_run(b2tex_ctx"))
    with open(os.path.join(OUT, "seam_mg_kernels.inc"), "w") as f:
        f.write(_kernel_part("seam_mg.cu", "// ---- host side: peer block management and launch",
                             ("__device__ __forceinline__ void st_release_sys", "__device__ __forceinline__ void mg_block_reduce6"))
                .replace("    __shared__ double smem[(MG_THREADS / 32) * 6 + 1];\n",
                         "    double *smem = (double *)emul::block_shared(sizeof(double) * ((MG_THREADS / 32) * 6 + 1));\n"))
    with open(os.path.join(OUT, "patches_kernels.inc"), "w") as f:
        f.write(_kernel_part("patches.cu", "void patches_free(b2tex_ctx"))
    with open(os.path.join(OUT, "localseam_kernels.inc"), "w") as f:
        f.write(_kernel_part("localseam.cu", "int local_seam_run(b2tex_ctx"))
    libs = {}
    cpp = os.path.join(ROOT, "tests", "cpp")
    names = ("emul_bvh", "emul_datacosts", "emul_mrf", "emul_seam", "emul_seam_mg", "emul_patches", "emul_localseam")

    def compile_one(name):
        so = os.path.join(OUT, name + ".so")
        subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared", "-w",
                               "-I" + os.path.join(cpp, "emul_include"), "-I" + cpp, "-I" + CUDA_INC, "-I" + CSRC,
                               "-I" + os.path.join(ROOT, "oracle"), "-I" + OUT, os.path.join(cpp, name + ".cpp"), "-o", so])
        return so

    import concurrent.futures as cf
    with cf.ThreadPoolExecutor(max_workers=len(names)) as ex:
        for name, so in zip(names, ex.map(compile_one, names)):
            libs[name] = C.CDLL(so)
    return libs


@pytest.mark.parametrize("name", ["tiny", "occ", "C2s"])
def test_device_bvh_build_and_traversal(emul, orc, scene_mod, name):
    """k_morton / k_hierarchy / k_refit give a well-formed tree (every triangle in exactly one leaf, boxes nest) and
    bvh_occluded() answers every vertex->camera ray like the oracle's BVH (itself checked against brute force)."""
    s = scene_mod.config(name, with_images=False)
    L, OL = emul["emul_bvh"], orc.lib()
    nv, K = s.verts.shape[0], s.num_views
    occ = np.zeros((K, nv), np.uint8)
    rays = np.zeros((K, nv, 8), np.float32)
    stats = np.zeros(4, np.int32)
    rc = L.emul_bvh_trace(orc._p(s.verts), C.c_uint32(nv), orc._p(s.faces), C.c_uint32(s.num_faces),
                          orc._p(np.ascontiguousarray(s.pos)), C.c_uint32(K), orc._p(occ), orc._p(rays), orc._p(stats))
    assert rc == 0, f"malformed tree (code {rc})"
    assert 0 < stats[0] <= 64                                  # traversal stack holds 100 entries
    OL.orc_bvh_build.restype = C.c_void_p
    b = C.c_void_p(OL.orc_bvh_build(orc._p(s.verts), orc._p(s.faces), C.c_uint32(s.num_faces)))
    fl = rays.reshape(-1, 8)
    base = fl.ctypes.data
    ref = np.zeros(len(fl), np.uint8)
    for i in range(len(fl)):
        p = base + 32 * i
        ref[i] = OL.orc_bvh_occluded(b, C.c_void_p(p), C.c_void_p(p + 12), C.c_float(fl[i, 6]), C.c_float(fl[i, 7]))
    OL.orc_bvh_free(b)
    assert ref.sum() > 0 and np.array_equal(ref, occ.ravel())


@pytest.mark.parametrize("name,data_term,vis", [("tiny", 1, True), ("occ", 1, True), ("occ", 0, True), ("occ", 1, False),
                                                ("occ2", 1, True), ("C2s", 1, True), ("messy", 1, True)])
def test_device_data_cost_kernels(emul, orc, get_scene, name, data_term, vis):
    """cull -> ray bitmaps -> rays -> quality -> compaction (csrc/datacosts.cu) vs orc_data_costs: identical
    (face, view) set and bit-identical qualities, with real occlusion in the `occ` scenes."""
    s = get_scene(name)
    L = emul["emul_datacosts"]
    views, keep = orc.make_views(s)
    grads = [orc.gradient_magnitude(s.images[k]) for k in range(s.num_views)]
    gp = (C.c_void_p * s.num_views)(*[g.ctypes.data for g in grads])
    F = s.num_faces
    ptr = np.zeros(F + 1, np.uint64)
    vw, ql = C.c_void_p(), C.c_void_p()
    stats = np.zeros(4, np.int64)
    rc = L.emul_data_costs(orc._p(s.verts), C.c_uint32(s.verts.shape[0]), orc._p(s.faces), orc._p(s.face_normals), C.c_uint32(F),
                           views, C.c_uint32(s.num_views), gp, data_term, 1 if vis else 0, orc._p(ptr), C.byref(vw), C.byref(ql),
                           orc._p(stats))
    assert rc == 0
    n = int(ptr[-1])
    view = np.ctypeslib.as_array(C.cast(vw, C.POINTER(C.c_uint16)), (max(n, 1),))[:n].copy()
    qual = np.ctypeslib.as_array(C.cast(ql, C.POINTER(C.c_float)), (max(n, 1),))[:n].copy()
    L.emul_free(vw); L.emul_free(ql)
    o = orc.data_costs(s, data_term=data_term, visibility=vis)
    assert np.array_equal(ptr, o["face_ptr"]) and np.array_equal(view, o["view"])
    assert np.array_equal(qual.view(np.uint32), o["quality"].view(np.uint32))
    if name.startswith("occ") and vis:
        assert stats[2] > 500                                  # occluded (vertex, view) rays
        assert n < stats[0] * 0.9                              # >10 % of the candidates are occluded
    if not vis:
        assert stats[1] == 0


@pytest.mark.parametrize("name,kw", [("tiny", {}), ("occ", {}), ("occ", dict(root_div=0, rounds=200)), ("occ", dict(num_parts=2)),
                                     ("occ", dict(group=32)), ("messy", {}), ("occ", dict(cap=16)), ("occ", dict(cap=16, group=8)),
                                     ("occ", dict(rounds=32, root_div=256, cap=32))])
def test_device_view_selection_kernels(emul, orc, scene_mod, get_scene, name, kw):
    """csrc/mrf.cu on fibers vs orc_view_selection: identical forest levels in iteration 1, identical iteration count,
    identical labels (=> identical energy).  `occ`: unseen faces (label 0, excluded from the graph), ten components,
    single-root mode, two partitions, 32 lanes per node instead of alloc_mrf's choice."""
    s = get_scene(name)
    adj = scene_mod.face_adjacency(s.faces)
    dc = orc.data_costs(s)
    P = dict(orc.DEFAULT_MRF)
    okw = {k: v for k, v in kw.items() if k not in ("group", "cap")}
    P.update(okw)
    o = orc.view_selection(adj[0], adj[1], dc["face_ptr"], dc["view"], dc["cost"], threads=1, **okw)
    F = s.num_faces
    params = np.array([P["max_iterations"], P["rounds"], P["root_div"], P["seed"], P["window"], P["num_parts"], kw.get("group", 0),
                       kw.get("cap", 0), 0], np.uint32)
    stats = np.zeros(4, np.uint64)
    labels = np.zeros(F, np.uint32)
    trace = np.full(P["max_iterations"] + 1, np.nan)
    lvl = np.zeros(F, np.uint32)
    it = emul["emul_mrf"].emul_view_selection(C.c_uint32(F), C.c_uint32(s.num_views), orc._p(adj[0]), orc._p(adj[1]), orc._p(dc["face_ptr"]),
                                              orc._p(dc["view"]), orc._p(dc["cost"]), orc._p(params), C.c_float(P["ratio"]), orc._p(labels),
                                              orc._p(trace), orc._p(lvl), orc._p(stats))
    assert it >= 0, "a kernel launch did not terminate (protocol hang)" if it == -1 else "bad parameters"
    assert np.array_equal(lvl, orc.mrf_sample_forest(adj[0], adj[1], dc["face_ptr"], 1, **okw))
    assert it == o["iterations"]
    assert np.array_equal(labels, o["labels"])
    assert abs(trace[it] - o["energy"]) <= 1e-6 * max(1.0, o["energy"])
    if name == "occ":
        assert (o["labels"] == 0).sum() > 10
    maxn = int(np.diff(dc["face_ptr"]).max())
    if "cap" in kw and maxn > kw["cap"]:
        assert stats[0] > 0          # trees with a label list longer than the scratch took the global-memory recursion
    elif name != "messy":
        assert stats[0] == 0, stats  # every tree of these scenes (manifold, lists within the scratch) is solved by k_tree proper


@pytest.mark.parametrize("name,ranks,kw", [("occ", 2, {}), ("occ", 3, dict(cap=16)), ("C2s", 4, {}), ("tiny", 8, {}), ("messy", 2, {})])
def test_device_multi_gpu_view_selection(emul, orc, scene_mod, get_scene, name, ranks, kw):
    """The multi-GPU view selection on `ranks` emulated devices: every rank owns a contiguous face range, runs k_forest /
    k_tree on it, stores the labels of its boundary faces into the label arrays of the ranks that own a neighbour
    (k_halo_push) and meets the others at epoch-flag barriers (k_mg_sync, all ranks alive at once under
    emul::launch_ranks, epochs crossing the 32-bit wrap); partial energies travel through per-rank slots and are summed in
    rank order.  Result: the labels, iteration count and energy of the oracle run with num_parts = ranks, identical stop
    decisions and energy traces on every rank, and every halo copy equal to its owner's label."""
    s = get_scene(name)
    adj = scene_mod.face_adjacency(s.faces)
    dc = orc.data_costs(s)
    P = dict(orc.DEFAULT_MRF)
    o = orc.view_selection(adj[0], adj[1], dc["face_ptr"], dc["view"], dc["cost"], threads=1, num_parts=ranks)
    F = s.num_faces
    params = np.array([P["max_iterations"], P["rounds"], P["root_div"], P["seed"], P["window"], ranks, 0, kw.get("cap", 0), ranks], np.uint32)
    stats = np.zeros(4, np.uint64)
    labels = np.zeros(F, np.uint32)
    trace = np.full(P["max_iterations"] + 1, np.nan)
    it = emul["emul_mrf"].emul_view_selection(C.c_uint32(F), C.c_uint32(s.num_views), orc._p(adj[0]), orc._p(adj[1]), orc._p(dc["face_ptr"]),
                                              orc._p(dc["view"]), orc._p(dc["cost"]), orc._p(params), C.c_float(P["ratio"]), orc._p(labels),
                                              orc._p(trace), None, orc._p(stats))
    assert it >= 0, {-1: "a launch hung (barrier protocol)", -4: "the ranks disagree", -5: "barrier timeout"}.get(it, it)
    assert it == o["iterations"] and np.array_equal(labels, o["labels"])
    assert abs(trace[it] - o["energy"]) <= 1e-6 * max(1.0, o["energy"])
    assert 0 < stats[3] < F / 2 or name == "tiny"      # only boundary faces travel


@pytest.mark.parametrize("name", ["tiny", "occ", "messy"])
def test_device_seam_leveling_kernels(emul, orc, scene_mod, get_scene, name):
    """csrc/seam.cu on fibers vs orc_global_seam_leveling: identical unknown numbering, identical Laplacian, bit-identical
    right-hand side, same CG iteration counts, solution within 1e-4 relative (the reductions are ordered differently)."""
    import scipy.sparse as sp
    s = get_scene(name)
    adj = scene_mod.face_adjacency(s.faces)
    rings = scene_mod.vertex_rings(s.faces, s.verts.shape[0])
    dc = orc.data_costs(s)
    labels = orc.view_selection(adj[0], adj[1], dc["face_ptr"], dc["view"], dc["cost"], threads=1)["labels"]
    o = orc.global_seam_leveling(s, rings, labels)
    views, keep = orc.make_views(s)
    Vn = s.verts.shape[0]
    row_ptr = np.zeros(Vn + 1, np.uint32)
    sizes = np.zeros(3, np.uint32)
    status = np.zeros(8, np.uint32)
    ptrs = [C.c_void_p() for _ in range(6)]
    L = emul["emul_seam"]
    rc = L.emul_seam(orc._p(s.verts), C.c_uint32(Vn), orc._p(s.faces), C.c_uint32(s.num_faces), orc._p(rings[0]), orc._p(rings[1]),
                     orc._p(rings[2]), orc._p(rings[3]), orc._p(np.ascontiguousarray(labels, np.uint32)), views, C.c_uint32(s.num_views),
                     orc._p(row_ptr), *[C.byref(p) for p in ptrs], orc._p(sizes), orc._p(status))
    assert rc == 0
    R, A, nnz = (int(v) for v in sizes)
    def grab(p, ct, n):
        a = np.ctypeslib.as_array(C.cast(p, C.POINTER(ct)), (max(n, 1),))[:n].copy()
        L.emul_seam_free(p)
        return a
    row_label, cp, cc, cv = grab(ptrs[0], C.c_uint32, R), grab(ptrs[1], C.c_uint32, R + 1), grab(ptrs[2], C.c_uint32, nnz), grab(ptrs[3], C.c_float, nnz)
    rhs, x = grab(ptrs[4], C.c_float, 3 * R).reshape(R, 3), grab(ptrs[5], C.c_float, 3 * R).reshape(R, 3)
    assert np.array_equal(row_ptr, o["row_ptr"]) and np.array_equal(row_label, o["row_label"]) and A == o["num_a_rows"]
    G = sp.csr_matrix((cv, cc, cp), shape=(R, R)); G.sum_duplicates()
    ocp, occ_, ocv = o["csr"]
    Om = sp.csr_matrix((ocv, occ_, ocp), shape=(R, R)); Om.sum_duplicates()
    assert (G != Om).nnz == 0
    assert np.array_equal(rhs.view(np.uint32), o["rhs"].view(np.uint32))
    assert status[:3].tolist() == list(o["iterations"])
    assert np.linalg.norm(x - o["x"]) / np.linalg.norm(o["x"]) < 1e-4


# ---- texture patches + adjust_colors (csrc/patches.cu, csrc/patches_host.h) -----------------------------------------
def _emul_patches(emul, orc, s, adj, labels, seam=None):
    L = emul["emul_patches"]
    views, keep = orc.make_views(s)
    ptrs = [C.c_void_p() for _ in range(6)]
    sizes = np.zeros(3, np.uint64)
    labels = np.ascontiguousarray(labels, np.uint32)
    if seam is not None:
        x = np.ascontiguousarray(seam["x"], np.float32)
        args = (orc._p(seam["row_ptr"]), orc._p(seam["row_label"]), orc._p(x), C.c_uint32(len(seam["row_label"])))
    else:
        args = (None, None, None, C.c_uint32(0))
    rc = L.emul_texture_patches(orc._p(s.verts), C.c_uint32(s.verts.shape[0]), orc._p(s.faces), C.c_uint32(s.num_faces), orc._p(adj[0]),
                                orc._p(adj[1]), orc._p(labels), views, C.c_uint32(s.num_views), *args, *[C.byref(p) for p in ptrs],
                                orc._p(sizes))
    assert rc == 0
    n, T, Pn = (int(v) for v in sizes)
    def grab(p, ct, k):
        a = np.ctypeslib.as_array(C.cast(p, C.POINTER(ct)), (max(k, 1),))[:k].copy()
        L.emul_patches_free(p)
        return a
    desc = grab(ptrs[0], C.c_int32, 8 * n).reshape(n, 8)
    faces, tex = grab(ptrs[1], C.c_uint32, T), grab(ptrs[2], C.c_float, 6 * T).reshape(-1, 2)
    img, val, bl = grab(ptrs[3], C.c_float, 3 * Pn).reshape(-1, 3), grab(ptrs[4], C.c_uint8, Pn), grab(ptrs[5], C.c_uint8, Pn)
    out, off = [], 0
    for q in range(n):
        label, mx, my, w, h, first, nf, _ = (int(v) for v in desc[q])
        out.append(dict(label=label, min_x=mx, min_y=my, faces=faces[first:first + nf].tolist(), texcoords=tex[3 * first:3 * (first + nf)],
                        image=img[off:off + w * h].reshape(h, w, 3), validity=val[off:off + w * h].reshape(h, w),
                        blending=bl[off:off + w * h].reshape(h, w)))
        off += w * h
    return out


def _same_patch(a, label, faces, texcoords, image, validity, blending):
    return (a["label"] == label and a["faces"] == list(faces)
            and np.array_equal(a["texcoords"].view(np.uint32), np.asarray(texcoords, np.float32).view(np.uint32))
            and a["image"].shape == image.shape and np.array_equal(a["image"].view(np.uint32), image.view(np.uint32))
            and np.array_equal(a["validity"], validity) and np.array_equal(a["blending"], blending))


@pytest.mark.parametrize("name,adjust", [("tiny", False), ("tiny", True), ("occ", True), ("messy", True)])
def test_device_texture_patch_kernels(emul, orc, scene_mod, get_scene, name, adjust):
    """csrc/patches.cu vs oracle/patches.py (itself pinned to the reference TUs): same patches, face order, bit-identical
    texcoords, images after adjust_colors (zero and solved offsets), validity and blending masks."""
    import patches as P
    s = get_scene(name)
    adj = scene_mod.face_adjacency(s.faces)
    rings = scene_mod.vertex_rings(s.faces, s.verts.shape[0])
    dc = orc.data_costs(s)
    labels = orc.view_selection(adj[0], adj[1], dc["face_ptr"], dc["view"], dc["cost"], threads=1)["labels"]
    seam = orc.global_seam_leveling(s, rings, labels) if adjust else None
    ep = _emul_patches(emul, orc, s, adj, labels, seam)
    pp, _ = P.generate_texture_patches(orc, s, adj, labels)
    assert len(ep) == len(pp) > 0
    if adjust:
        pa = P.apply_adjust_values(s, pp, seam["row_ptr"], seam["row_label"], seam["x"])
        exp = [(q.label, q.faces, q.texcoords, q.image, q.validity, q.blending) for q in pa]
    else:
        exp = [(q.label, q.faces, q.texcoords) + P.adjust_colors(q, np.zeros((3 * len(q.faces), 3), np.float32)) for q in pp]
    for a, e, q in zip(ep, exp, pp):
        assert _same_patch(a, *e)
        assert [a["min_x"], a["min_y"]] == list(q.bbox[:2])


def test_device_texture_patches_merge_like_reference_tu(emul, orc, scene_mod, get_scene):
    """Candidate merging (generate_texture_patches.cpp:484-508): label islands whose bounding box lies inside the box of
    another component of the same label are absorbed.  Crafted on `small` (six one-face islands); compared with what the
    reference's own translation units return on it (tests/golden/reference_tu.json)."""
    import patches as P
    s = get_scene("small")
    adj, rings, labels = G.seam_inputs(orc, scene_mod, s)
    labels, islands = G.island_labels(orc, s, adj, labels)
    assert islands >= 3
    ncomp = sum(len(P.get_subgraphs(adj[0], adj[1], labels, lab)) for lab in range(1, s.num_views + 1))
    ep = _emul_patches(emul, orc, s, adj, labels, None)
    assert len(ep) <= ncomp - islands                          # the islands (at least) were absorbed
    g = G.load()[0]["texture_patches_with_islands/small"]
    assert g["islands"] == islands and g["labels"] == [a["label"] for a in ep]
    for field, d in G.patch_digests(ep, ("faces", "texcoords", "image", "validity", "blending")).items():
        assert g[field] == d, field


def test_patch_plan_merge_chains(emul):
    """plan_patches() on random rectangles vs a literal transcription of the reference's std::list loop (:484-508),
    including chains (a candidate that absorbed others is absorbed itself later: offsets accumulate in order)."""
    L = emul["emul_patches"]
    rng = np.random.RandomState(4)
    chains_seen = 0
    for trial in range(60):
        Cn = int(rng.randint(2, 14))
        labels = np.sort(rng.randint(1, 4, size=Cn)).astype(np.uint32)
        x0, y0 = rng.randint(0, 40, size=Cn), rng.randint(0, 40, size=Cn)
        w, h = rng.randint(1, 45, size=Cn), rng.randint(1, 45, size=Cn)
        if trial % 3 == 0:                                     # nested boxes, small first -> chains (the harness reports <= 8 offsets)
            Cn = min(Cn, 8); labels = labels[:Cn]
            x0, y0, w, h = 20 - np.arange(Cn), 20 - np.arange(Cn), 2 + 2 * np.arange(Cn), 2 + 2 * np.arange(Cn)
            labels[:] = 1
        bbox = np.stack([x0, y0, x0 + w, y0 + h], 1).astype(np.int32)
        # transcription: candidates in order, Rect(min - border, max), list erase semantics
        cands = [dict(r=[int(b[0]) - 1, int(b[1]) - 1, int(b[2]), int(b[3])], members=[(c, [])], label=int(labels[c])) for c, b in enumerate(bbox)]
        out = []
        for lab in sorted(set(labels.tolist())):
            lst = [c for c in cands if c["label"] == lab]
            i = 0
            while i < len(lst):
                it = lst[i]
                j = 0
                while j < len(lst):
                    sit = lst[j]
                    if sit is not it and sit["r"][0] >= it["r"][0] and sit["r"][2] <= it["r"][2] and sit["r"][1] >= it["r"][1] and sit["r"][3] <= it["r"][3]:
                        off = (float(sit["r"][0] - it["r"][0]), float(sit["r"][1] - it["r"][1]))
                        it["members"] += [(c, ch + [off]) for c, ch in sit["members"]]
                        del lst[j]
                        if j < i:
                            i -= 1
                    else:
                        j += 1
                i += 1
            out += lst
        comp_patch, comp_pos, cnt = np.zeros(Cn, np.uint32), np.zeros(Cn, np.uint32), np.zeros(Cn, np.uint32)
        chain = np.zeros((Cn, 16), np.float32)
        desc = np.zeros((Cn, 8), np.int32)
        n = L.emul_plan_patches(C.c_uint32(Cn), labels.ctypes.data_as(C.c_void_p), bbox.ctypes.data_as(C.c_void_p),
                                comp_patch.ctypes.data_as(C.c_void_p), comp_pos.ctypes.data_as(C.c_void_p), cnt.ctypes.data_as(C.c_void_p),
                                chain.ctypes.data_as(C.c_void_p), desc.ctypes.data_as(C.c_void_p))
        assert n == len(out)
        for q, cand in enumerate(out):
            assert desc[q, 0] == cand["label"] and desc[q, 1] == cand["r"][0] and desc[q, 2] == cand["r"][1]
            assert desc[q, 3] == cand["r"][2] - cand["r"][0] + 2 and desc[q, 4] == cand["r"][3] - cand["r"][1] + 2
            for pos, (c, ch) in enumerate(cand["members"]):
                assert comp_patch[c] == q and comp_pos[c] == pos and cnt[c] == len(ch)
                assert chain[c, :2 * len(ch)].tolist() == [v for o in ch for v in o]
                chains_seen += len(ch) >= 2
    assert chains_seen > 10


# ---- local seam leveling (csrc/localseam.cu) ---------------------------------------------------------------------------
def _emul_pipeline(emul, orc, s, adj, labels, seam, stage):
    L = emul["emul_localseam"]
    views, keep = orc.make_views(s)
    ptrs = [C.c_void_p() for _ in range(6)]
    sizes = np.zeros(8, np.uint64)
    labels = np.ascontiguousarray(labels, np.uint32)
    if seam is not None:
        x = np.ascontiguousarray(seam["x"], np.float32)
        sargs = (orc._p(seam["row_ptr"]), orc._p(seam["row_label"]), orc._p(x), C.c_uint32(len(seam["row_label"])))
    else:                                                      # no global leveling: zero offsets (texrecon.cpp:174-183)
        sargs = (None, None, None, C.c_uint32(0))
    rc = L.emul_texture_pipeline(orc._p(s.verts), C.c_uint32(s.verts.shape[0]), orc._p(s.faces), C.c_uint32(s.num_faces), orc._p(adj[0]),
                                 orc._p(adj[1]), orc._p(labels), views, C.c_uint32(s.num_views), *sargs, stage,
                                 *[C.byref(p) for p in ptrs], orc._p(sizes))
    assert rc == 0, "the Poisson CG launch did not terminate" if rc == -1 else rc
    n, T, Pn = (int(v) for v in sizes[:3])
    def grab(p, ct, k):
        a = np.ctypeslib.as_array(C.cast(p, C.POINTER(ct)), (max(k, 1),))[:k].copy()
        L.emul_local_free(p)
        return a
    desc = grab(ptrs[0], C.c_int32, 8 * n).reshape(n, 8)
    faces, tex = grab(ptrs[1], C.c_uint32, T), grab(ptrs[2], C.c_float, 6 * T).reshape(-1, 2)
    img, val, bl = grab(ptrs[3], C.c_float, 3 * Pn).reshape(-1, 3), grab(ptrs[4], C.c_uint8, Pn), grab(ptrs[5], C.c_uint8, Pn)
    out, off = [], 0
    for q in range(n):
        label, mx, my, w, h, first, nf, _ = (int(v) for v in desc[q])
        out.append(dict(label=label, faces=faces[first:first + nf].tolist(), image=img[off:off + w * h].reshape(h, w, 3),
                        validity=val[off:off + w * h].reshape(h, w), blending=bl[off:off + w * h].reshape(h, w)))
        off += w * h
    return out, sizes


@pytest.fixture(scope="module")
def local_inputs(orc, scene_mod, get_scene):
    cache = {}
    def _get(name):
        if name not in cache:
            import patches as P
            s = get_scene(name)
            adj = scene_mod.face_adjacency(s.faces)
            rings = scene_mod.vertex_rings(s.faces, s.verts.shape[0])
            dc = orc.data_costs(s)
            labels = orc.view_selection(adj[0], adj[1], dc["face_ptr"], dc["view"], dc["cost"], threads=1)["labels"]
            seam = orc.global_seam_leveling(s, rings, labels)
            pp, pvpi = P.generate_texture_patches(orc, s, adj, labels)
            cache[name] = (s, adj, rings, labels, seam, pp, pvpi)
        return cache[name]
    return _get


@pytest.mark.parametrize("name", ["tiny", "occ", "messy", "C2s"])
def test_device_seam_colours_stamping_and_blending_mask(emul, orc, local_inputs, name, monkeypatch):
    """csrc/localseam.cu up to the Poisson solve vs oracle/patches.local_seam_leveling with the solve switched off: the
    images with the mean seam / vertex colours stamped in ("last writer wins" by atomicMax on the write order) and the
    blending masks after prepare_blending_mask (breadth-first layering, 20 px strip) are bit-identical.  The harness also runs
    the seam planning twice -- host bookkeeping (patches_host.h) and the device kernels (k_seam_edges / k_plan_edges /
    k_plan_vertices) -- and fails unless every planning array is identical (error codes -7 .. -15)."""
    import patches as P
    s, adj, rings, labels, seam, pp, pvpi = local_inputs(name)
    pa = P.apply_adjust_values(s, pp, seam["row_ptr"], seam["row_label"], seam["x"])
    monkeypatch.setattr(P, "poisson_blend", lambda *a, **k: None)
    P.local_seam_leveling(s, adj, labels, pa, pvpi)
    ep, sizes = _emul_pipeline(emul, orc, s, adj, labels, seam, 1)
    assert len(ep) == len(pa) and sizes[3] > 20 and sizes[5] > 20
    for a, b in zip(ep, pa):
        assert np.array_equal(a["blending"], b.blending)
        assert np.array_equal(a["image"].view(np.uint32), b.image.view(np.uint32))
    assert sum(int((a["blending"] == 128).sum()) for a in ep) > 100 and sum(int((a["blending"] == 255).sum()) for a in ep) > 100


@pytest.mark.parametrize("name", ["tiny", "occ", "messy"])
def test_device_local_seam_leveling(emul, orc, local_inputs, name):
    """Full tex::local_seam_leveling on the device kernels (one batched CG over all patches, on fibers) vs the oracle
    (scipy splu per patch) and vs what the reference's own translation units return (SparseLU shim, tests/golden):
    same validity masks, images within 5e-5 (CG tolerance 1e-5 relative residual; 8-bit quantisation is 4e-3)."""
    import patches as P
    s, adj, rings, labels, seam, pp, pvpi = local_inputs(name)
    pa = P.apply_adjust_values(s, pp, seam["row_ptr"], seam["row_label"], seam["x"])
    before = [q.image.copy() for q in pa]
    P.local_seam_leveling(s, adj, labels, pa, pvpi)
    ep, sizes = _emul_pipeline(emul, orc, s, adj, labels, seam, 2)
    assert sizes[6] > 500 and 10 < sizes[7] < 1000                # unknowns, CG iterations
    worst = 0.0
    for a, b, b0 in zip(ep, pa, before):
        assert np.array_equal(a["validity"], b.validity)
        worst = max(worst, float(np.abs(a["image"] - b.image).max()))
    print(f"local seam leveling {name}: max |device - oracle| = {worst:.2e}, unknowns {sizes[6]}, CG iterations {sizes[7]}")
    assert worst < 2e-5                                           # the bar of the oracle <-> reference pin
    assert max(float(np.abs(b.image - b0).max()) for b, b0 in zip(pa, before)) > 0.01
    golden = G.load()
    key = f"local_seam_leveling/{name}"
    assert golden[0][key]["validity"] == G.patch_digests(ep, ("validity",))["validity"]
    assert G.image_error(golden, key, [a["image"] for a in ep]) < 5e-5


def _random_mrf_problem(rng, n, extra_edges, K, max_labels, unseen_frac=0.03):
    """ring + random chords: node degrees up to ~8 (face graphs of non-manifold meshes exceed 3)"""
    edges = set((i, (i + 1) % n) for i in range(n))
    while len(edges) < n + extra_edges:
        a, b = rng.randint(n, size=2)
        if a != b:
            edges.add((min(a, b), max(a, b)))
    adj = [[] for _ in range(n)]
    for a, b in sorted(edges):
        adj[a].append(b); adj[b].append(a)
    ap = np.zeros(n + 1, np.uint32)
    ap[1:] = np.cumsum([len(x) for x in adj])
    ai = np.array([w for x in adj for w in x], np.uint32)
    ptr, view, cost = [0], [], []
    for i in range(n):
        k = 0 if rng.rand() < unseen_frac else rng.randint(1, max_labels + 1)
        view += np.sort(rng.choice(K, size=k, replace=False)).tolist()
        cost += rng.uniform(0, 1, size=k).astype(np.float32).tolist()
        ptr.append(len(view))
    return ap, ai, np.array(ptr, np.uint64), np.array(view, np.uint16), np.array(cost, np.float32)


@pytest.mark.parametrize("case", ["degree>3", "degree>3, no label masks", "3000 views, binary search", "64 labels per node"])
def test_device_view_selection_generic_paths(emul, orc, case):
    """Code paths of k_up / k_down / k_energy no mesh-derived test reaches: neighbour lists longer than 3 (CSR fallback
    instead of the packed adjacency), more than 2047 views (no label bitmasks: binary search in the sorted label lists),
    long label lists (several strides of the lane loop)."""
    rng = np.random.RandomState(7)
    n, extra, K, maxl, Kdev, group = {"degree>3": (600, 500, 12, 6, 12, 0), "degree>3, no label masks": (600, 500, 12, 6, 5000, 0),
                                      "3000 views, binary search": (500, 0, 3000, 40, 3000, 32),
                                      "64 labels per node": (400, 300, 70, 64, 70, 0)}[case]
    ap, ai, ptr, view, cost = _random_mrf_problem(rng, n, extra, K, maxl)
    o = orc.view_selection(ap, ai, ptr, view, cost, threads=1)
    P = dict(orc.DEFAULT_MRF)
    params = np.array([P["max_iterations"], P["rounds"], P["root_div"], P["seed"], P["window"], P["num_parts"], group, 0, 0], np.uint32)
    labels = np.zeros(n, np.uint32)
    trace = np.full(P["max_iterations"] + 1, np.nan)
    it = emul["emul_mrf"].emul_view_selection(C.c_uint32(n), C.c_uint32(Kdev), orc._p(ap), orc._p(ai), orc._p(ptr), orc._p(view), orc._p(cost),
                                              orc._p(params), C.c_float(P["ratio"]), orc._p(labels), orc._p(trace), None, None)
    assert it == o["iterations"] and np.array_equal(labels, o["labels"])
    if extra:
        assert int(np.diff(ap).max()) > 3


# ---- multi-GPU seam solve: compute + exchange in one kernel per GPU (csrc/seam_mg.cu) ------------------------------------
@pytest.mark.parametrize("ranks,grid", [(2, 2), (3, 1)])
def test_device_multi_gpu_seam_solve(emul, orc, scene_mod, get_scene, ranks, grid):
    """k_pcg_mg on `ranks` emulated devices at once (emul::launch_ranks: one grid.sync scope per device, peer blocks =
    each other's host buffers): the rows are split across the ranks, z = M^-1 r of the halo rows travels by peer stores (the readers update their own copy of p),
    dot products go through per-rank slots summed in rank order, barriers are epoch flags in peer memory (started 16 below
    the 32-bit wrap-around).  Every rank must end with the SAME complete solution, with the single-GPU iteration counts,
    within 1e-4 of the oracle, and no barrier may time out."""
    s = get_scene("tiny")
    adj = scene_mod.face_adjacency(s.faces)
    rings = scene_mod.vertex_rings(s.faces, s.verts.shape[0])
    dc = orc.data_costs(s)
    labels = orc.view_selection(adj[0], adj[1], dc["face_ptr"], dc["view"], dc["cost"], threads=1)["labels"]
    o = orc.global_seam_leveling(s, rings, labels)
    views, keep = orc.make_views(s)
    L = emul["emul_seam_mg"]
    R, xp = C.c_uint32(), C.c_void_p()
    status = np.zeros(16 * ranks, np.uint32)
    rc = L.emul_seam_mg(orc._p(s.verts), C.c_uint32(s.verts.shape[0]), orc._p(s.faces), C.c_uint32(s.num_faces), orc._p(rings[0]),
                        orc._p(rings[1]), orc._p(rings[2]), orc._p(rings[3]), orc._p(np.ascontiguousarray(labels, np.uint32)), views,
                        C.c_uint32(s.num_views), C.c_uint32(ranks), C.c_uint32(grid), C.byref(R), C.byref(xp), orc._p(status))
    assert rc == 0, "a rank never left the kernel (barrier protocol hang)" if rc == -1 else rc
    Rn = R.value
    x = np.ctypeslib.as_array(C.cast(xp, C.POINTER(C.c_float)), (ranks * Rn * 3,)).copy().reshape(ranks, Rn, 3)
    L.emul_seam_mg_free(xp)
    st = status.reshape(ranks, 16)
    assert Rn == len(o["row_label"]) and not st[:, 7].any()
    assert 0 < st[0, 15] < Rn          # only the halo rows of the search direction travel
    for k in range(ranks):
        assert np.array_equal(x[k].view(np.uint32), x[0].view(np.uint32))
        assert st[k, :3].tolist() == list(o["iterations"])
    assert np.linalg.norm(x[0] - o["x"]) / np.linalg.norm(o["x"]) < 1e-4


def test_device_multi_gpu_seam_solve_survives_a_dead_peer(emul, orc, scene_mod, get_scene):
    """A peer that never arrives (process died, GPU fell off the bus) must not hang the healthy ranks: every wait in k_pcg_mg
    has a poll limit, the verdict is taken once per block, and after the first timeout nobody waits any more.  Rank 1 of 2 never
    enters the kernel; rank 0 (two blocks) must leave it with barrier timeouts recorded in status[7]."""
    s = get_scene("tiny")
    adj = scene_mod.face_adjacency(s.faces)
    rings = scene_mod.vertex_rings(s.faces, s.verts.shape[0])
    dc = orc.data_costs(s)
    labels = orc.view_selection(adj[0], adj[1], dc["face_ptr"], dc["view"], dc["cost"], threads=1)["labels"]
    views, keep = orc.make_views(s)
    L = emul["emul_seam_mg"]
    ranks, grid = 2, 2
    R, xp = C.c_uint32(), C.c_void_p()
    status = np.zeros(16 * ranks, np.uint32)
    L.emul_set_dead_rank(C.c_int(1), C.c_uint64(300))
    try:
        rc = L.emul_seam_mg(orc._p(s.verts), C.c_uint32(s.verts.shape[0]), orc._p(s.faces), C.c_uint32(s.num_faces), orc._p(rings[0]),
                            orc._p(rings[1]), orc._p(rings[2]), orc._p(rings[3]), orc._p(np.ascontiguousarray(labels, np.uint32)), views,
                            C.c_uint32(s.num_views), C.c_uint32(ranks), C.c_uint32(grid), C.byref(R), C.byref(xp), orc._p(status))
    finally:
        L.emul_set_dead_rank(C.c_int(-1), C.c_uint64(0))
    assert rc == 0, "the healthy rank never left the kernel"
    L.emul_seam_mg_free(xp)
    st = status.reshape(ranks, 16)
    assert st[0, 7] > 0          # barrier timeouts reported (seam_mg_solve turns them into B2TEX_ERR_CUDA)


def test_device_local_seam_leveling_without_global_leveling(emul, orc, local_inputs):
    """texrecon --skip_global_seam_leveling: zero-offset adjust_colors pass (texrecon.cpp:174-183), then local seam leveling on
    the raw patch colours (larger seam differences to blend away).  Against what the reference's own translation units
    return (tests/golden/reference_tu.json)."""
    s, adj, rings, labels, seam, pp, pvpi = local_inputs("tiny")
    ep, sizes = _emul_pipeline(emul, orc, s, adj, labels, None, 2)
    golden = G.load()
    key = "local_seam_leveling_without_global/tiny"
    assert golden[0][key]["validity"] == G.patch_digests(ep, ("validity",))["validity"]
    assert G.image_error(golden, key, [a["image"] for a in ep]) < 1e-4   # raw gain/bias differences are ~10x larger than after global leveling


@pytest.mark.parametrize("seed", [0x9E3779B97F4A7C15, 12345])
def test_protocols_do_not_depend_on_the_thread_schedule(emul, orc, scene_mod, get_scene, seed):
    """Hardware promises no execution order between warps, blocks or GPUs.  The fiber scheduler can visit the live threads in
    a fresh pseudo-random order on every pass; the dataflow sweeps of the MRF (flags), the cooperative PCG (grid.sync) and
    the multi-GPU solve (epoch flags in peer memory) must give the very same results as under round robin."""
    s = get_scene("tiny")
    adj = scene_mod.face_adjacency(s.faces)
    rings = scene_mod.vertex_rings(s.faces, s.verts.shape[0])
    dc = orc.data_costs(s)
    o = orc.view_selection(adj[0], adj[1], dc["face_ptr"], dc["view"], dc["cost"], threads=1)
    os_ = orc.global_seam_leveling(s, rings, o["labels"])
    views, keep = orc.make_views(s)
    F = s.num_faces
    for lib in ("emul_mrf", "emul_seam_mg"):
        emul[lib].emul_set_schedule(C.c_uint64(seed))
    try:
        P = dict(orc.DEFAULT_MRF)
        params = np.array([P["max_iterations"], P["rounds"], P["root_div"], P["seed"], P["window"], P["num_parts"], 0, 0, 0], np.uint32)
        labels = np.zeros(F, np.uint32)
        trace = np.full(P["max_iterations"] + 1, np.nan)
        it = emul["emul_mrf"].emul_view_selection(C.c_uint32(F), C.c_uint32(s.num_views), orc._p(adj[0]), orc._p(adj[1]), orc._p(dc["face_ptr"]),
                                                  orc._p(dc["view"]), orc._p(dc["cost"]), orc._p(params), C.c_float(P["ratio"]), orc._p(labels),
                                                  orc._p(trace), None, None)
        assert it == o["iterations"] and np.array_equal(labels, o["labels"])
        ranks = 2
        R, xp = C.c_uint32(), C.c_void_p()
        status = np.zeros(16 * ranks, np.uint32)
        L = emul["emul_seam_mg"]
        rc = L.emul_seam_mg(orc._p(s.verts), C.c_uint32(s.verts.shape[0]), orc._p(s.faces), C.c_uint32(F), orc._p(rings[0]), orc._p(rings[1]),
                            orc._p(rings[2]), orc._p(rings[3]), orc._p(np.ascontiguousarray(o["labels"], np.uint32)), views,
                            C.c_uint32(s.num_views), C.c_uint32(ranks), C.c_uint32(1), C.byref(R), C.byref(xp), orc._p(status))
        assert rc == 0
        x = np.ctypeslib.as_array(C.cast(xp, C.POINTER(C.c_float)), (ranks * R.value * 3,)).copy().reshape(ranks, R.value, 3)
        L.emul_seam_mg_free(xp)
        st = status.reshape(ranks, 16)
        assert not st[:, 7].any() and st[0, :3].tolist() == list(os_["iterations"])
        assert np.array_equal(x[0].view(np.uint32), x[1].view(np.uint32))
        assert np.linalg.norm(x[0] - os_["x"]) / np.linalg.norm(os_["x"]) < 1e-4
    finally:
        for lib in ("emul_mrf", "emul_seam_mg"):
            emul[lib].emul_set_schedule(C.c_uint64(0))
