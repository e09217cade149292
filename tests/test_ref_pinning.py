"""Pins the oracle against the reference's own translation units.

oracle/_ref/libtexref.so is built from the reference's libs/tex/*.cpp (unmodified, compiled where they lie) and the
dependency shims in oracle/refshim/ (MVE / rayint / Eigen / mapMAP are not vendored in the reference, see
oracle/refshim/README.md).  Everything written in libs/tex -- cull rules, projection, validity mask, footprint
integral, histogram, normalisation -- runs as the reference wrote it; the oracle has to agree bit for bit.

What those translation units return on the inputs below is stored in tests/golden/reference_tu.{json,npz}
(tests/golden/make_reference_golden.py; format and inputs in tests/golden/reference_golden.py).
"""
import os
import sys

import numpy as np
import pytest

import refpin

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
import reference_golden as G  # noqa: E402

D = G.digest


@pytest.fixture(scope="module")
def ref():
    return G.load()


def assert_data_costs(g, o):
    assert int(o["face_ptr"][-1]) == g["nnz"]
    assert D(o["face_ptr"]) == g["face_ptr"] and D(o["view"]) == g["view"]
    assert D(o["cost"]) == g["cost"]


@pytest.mark.parametrize("name", ["tiny", "small", "occ", "messy"])
@pytest.mark.parametrize("data_term", [1, 0])
def test_data_costs_match_reference_tu(ref, orc, get_scene, name, data_term):
    """tex::calculate_data_costs (calculate_data_costs.cpp:131-323) vs orc_data_costs: same (face, view) set,
    bit-identical costs."""
    s = get_scene(name)
    g = ref[0][f"data_costs/{name}/{data_term}"]
    assert g["nnz"] > s.num_faces
    assert_data_costs(g, orc.data_costs(s, data_term=data_term))


@pytest.mark.parametrize("name", ["tiny", "occ"])
def test_data_costs_without_visibility_test(ref, orc, get_scene, name):
    s = get_scene(name)
    g = ref[0][f"data_costs_no_visibility/{name}"]
    assert_data_costs(g, orc.data_costs(s, visibility=False))
    with_test = ref[0][f"data_costs/{name}/1"]
    assert g["nnz"] >= with_test["nnz"]
    if name == "occ":                                                    # floating plates occlude
        assert g["nnz"] > with_test["nnz"]
        assert_data_costs(with_test, orc.data_costs(s))


@pytest.mark.parametrize("mode", [1, 2])
def test_outlier_removal_matches_reference_tu(ref, orc, get_scene, mode, monkeypatch):
    """photometric_outlier_detection (calculate_data_costs.cpp:35-129).  The reference's per-face info order
    before detection depends on the OpenMP merge (:241-249; one thread -> descending view id), the oracle uses
    ascending view id, so sums may differ in the last bits: same survivors, costs within 1e-5."""
    s = get_scene("tiny")
    g = ref[0][f"outlier_removal/{mode}"]
    o = orc.data_costs(s, outlier_removal=mode)
    assert int(o["face_ptr"][-1]) == g["nnz"] and D(o["face_ptr"]) == g["face_ptr"] and D(o["view"]) == g["view"]
    assert np.allclose(ref[1][f"outlier_removal_{mode}_cost"], o["cost"], rtol=0, atol=1e-5)
    base = orc.data_costs(s)
    assert int(o["face_ptr"][-1]) <= int(base["face_ptr"][-1])


def test_validity_mask_and_erosion_quirk(ref, orc):
    """texture_view.cpp:42-94 (corner flood fill over black pixels) and :109-132 (erosion that leaves the image
    border untouched because the border write lands in the array that is swapped away)."""
    img, img2 = G.validity_images()
    m_ref, m_orc = ref[1]["validity_mask"], orc.validity_mask(img)
    assert np.array_equal(m_ref, m_orc) and m_ref[16, 21] == 1 and m_ref[2, 10] == 0
    e_ref, e_orc = ref[1]["validity_mask_eroded"], orc.erode(m_orc)
    assert np.array_equal(e_ref, e_orc)
    assert e_ref[6, 10] == 0 and e_ref[7, 10] == 1            # one ring eaten next to the black frame
    e2_ref = ref[1]["validity_mask_eroded_no_black"]
    assert e2_ref.all()                                       # the quirk: border pixels stay valid
    assert np.array_equal(e2_ref, orc.erode(orc.validity_mask(img2)))


def test_face_info_matches_reference_tu(ref, orc, get_scene):
    """TextureView::get_face_info (texture_view.cpp:134-251) on random triangles of every size class: sub-pixel
    (vertex sampling), slivers (slow path / skipped scan lines) and large footprints (fast scan line path)."""
    import ctypes as C
    s = get_scene("small")
    k = G.FACE_INFO_VIEW
    v, keep = refpin._one_view(s, k)
    grad = orc.gradient_magnitude(s.images[k])
    tris = G.face_info_triangles(s, orc.data_costs(s), k)
    for data_term in (1, 0):
        q_ref = ref[1][f"face_quality_{data_term}"]
        assert len(q_ref) == len(tris)
        q_orc = np.empty(len(tris), np.float32)
        L = orc.lib()
        for i, t in enumerate(tris):
            q_orc[i] = L.orc_face_quality(C.byref(v), orc._p(grad), orc._p(t[0].copy()), orc._p(t[1].copy()), orc._p(t[2].copy()), data_term)
        ok = ~np.isnan(q_ref)                                  # NaN = projects outside the valid area
        assert ok.sum() > len(tris) // 2
        assert np.array_equal(q_ref[ok].view(np.uint32), q_orc[ok].view(np.uint32))
        if data_term == 1:
            assert (q_ref[ok] > 0).sum() > ok.sum() // 2


def test_tri_and_histogram_match_reference_tu(ref, orc):
    import ctypes as C
    L = orc.lib()
    area, inside = ref[1]["tri_area"], ref[1]["tri_inside"]
    draws, hist = G.triangle_and_histogram_draws()
    for i, (p, x, y) in enumerate(draws):
        assert area[i] == L.orc_tri_area(orc._p(p[0].copy()), orc._p(p[1].copy()), orc._p(p[2].copy()))
        assert inside[i] == L.orc_tri_inside(orc._p(p[0].copy()), orc._p(p[1].copy()), orc._p(p[2].copy()), C.c_float(x), C.c_float(y))
    for i, v in enumerate(hist):
        n = len(v)
        vmax = float(v.max())
        r = ref[1]["histogram_percentile"][i]
        o = float(L.orc_histogram_percentile(orc._p(v), C.c_uint64(n), C.c_float(vmax), 10000, C.c_float(0.995)))
        assert r == o


def test_pixel_coords_match_reference_tu(ref, orc, get_scene):
    import ctypes as C
    s = get_scene("tiny")
    L = orc.lib()
    for j, k in enumerate(G.PIXEL_COORD_VIEWS):
        v, keep = refpin._one_view(s, k)
        for n, i in enumerate(G.pixel_coord_vertices(s)):
            x = s.verts[i].copy()
            out = np.empty(2, np.float32)
            L.orc_pixel_coords(C.byref(v), orc._p(x), orc._p(out))
            assert np.array_equal(ref[1]["pixel_coords"][j, n].view(np.uint32), out.view(np.uint32))


# ---- adjacency graph and MRF model (build_adjacency_graph.cpp, view_selection.cpp) ------------------------------
@pytest.mark.parametrize("name", ["tiny", "small", "occ", "C2s", "messy"])
def test_adjacency_matches_reference_tu(ref, scene_mod, get_scene, name):
    """tex::build_adjacency_graph (:16-53) on the reference's UniGraph vs scene.face_adjacency (what the oracle and the
    C ABI are fed): same neighbours in the same adjacency-list order, borders (C2s) and separate components (occ) included."""
    s = get_scene(name)
    g = ref[0][f"adjacency/{name}"]
    a_ptr, a_idx = scene_mod.face_adjacency(s.faces)
    assert D(a_ptr) == g["ptr"] and D(a_idx) == g["idx"]


@pytest.mark.parametrize("name", ["tiny", "occ"])
def test_mrf_model_and_label_decoding_match_reference_tu(ref, orc, scene_mod, get_scene, name):
    """view_selection.cpp:26-82 builds the model, :120-131 decodes the solution.  With the recording mapMAP shim: edges
    only between seen faces (i < j, weight 1), label set = view id + 1 in DataCosts column order, unary = data cost, unseen
    faces get the single label 0 with cost 1, Potts weight 1, StopWhenReturnsDiminish(5, 0.01), deterministic seed
    548923723.  The oracle's energy function must be the energy of exactly this model."""
    s = get_scene(name)
    dc = orc.data_costs(s)
    if name == "tiny":                                           # make a few faces unseen
        dc = G.without_views(dc)
    adj = scene_mod.face_adjacency(s.faces)
    g = ref[0][f"mrf_model/{name}"]
    F = s.num_faces
    ptr = dc["face_ptr"].astype(np.int64)
    seen = ptr[1:] > ptr[:-1]
    assert (~seen).sum() >= (4 if name == "tiny" else 0)
    # edges
    exp = [(i, int(j)) for i in range(F) if seen[i] for j in adj[1][adj[0][i]:adj[0][i + 1]] if i < j and seen[j]]
    edges = np.array(exp, np.uint32).reshape(-1, 2)
    assert D(edges) == g["edges"]
    # label sets and unaries
    ls_label = [dc["view"][ptr[f]:ptr[f + 1]].astype(np.int32) + 1 if seen[f] else np.zeros(1, np.int32) for f in range(F)]
    ls_cost = [dc["cost"][ptr[f]:ptr[f + 1]] if seen[f] else np.ones(1, np.float32) for f in range(F)]
    lp = np.r_[0, np.cumsum([len(ll) for ll in ls_label])].astype(np.uint64)
    ls_label, ls_cost = np.concatenate(ls_label), np.concatenate(ls_cost).astype(np.float32)
    assert D(lp) == g["ls_ptr"] and D(ls_label) == g["ls_label"] and D(ls_cost) == g["ls_cost"]
    p = g["params"]
    assert p["potts"] == 1.0 and p["window"] == 5 and abs(p["ratio"] - 0.01) < 1e-12
    assert p["seed"] == 548923723 and p["deterministic"] == 1 and p["model_complete"] == 1 and p["components_updated"] == 1
    assert p["use_multilevel"] == 1 and p["use_spanning_tree"] == 1 and p["use_acyclic"] == 1 and p["force_acyclic"] == 1
    # decoding of the shim's solution (cheapest label per node, first minimum)
    exp_labels = np.zeros(F, np.uint32)
    for f in range(F):
        if seen[f]:
            c = dc["cost"][ptr[f]:ptr[f + 1]]
            exp_labels[f] = int(dc["view"][ptr[f] + int(np.argmin(c))]) + 1
    assert D(exp_labels) == g["labels"]
    # the oracle's objective = energy of the recorded model, for the greedy and for the optimised labeling
    o = orc.view_selection(adj[0], adj[1], dc["face_ptr"], dc["view"], dc["cost"], threads=1)
    lp = lp.astype(np.int64)
    def model_energy(labels):
        e = 0.0
        for f in range(F):
            ll = ls_label[lp[f]:lp[f + 1]]
            k = int(np.flatnonzero(ll == labels[f])[0])
            e += float(ls_cost[lp[f] + k])
        e += sum(1.0 for a, b in edges if labels[a] != labels[b])
        return e
    for lab in (exp_labels, o["labels"]):
        e_model = model_energy(lab)
        e_orc = orc.mrf_energy(adj[0], adj[1], dc["face_ptr"], dc["view"], dc["cost"], lab)
        assert abs(e_model - e_orc) < 1e-6 * max(1.0, e_model)
    assert model_energy(o["labels"]) < model_energy(exp_labels)


# ---- texture patches, global and local seam leveling ---------------------------------------------------------------
@pytest.fixture(scope="module")
def seam_inputs(orc, scene_mod, get_scene):
    cache = {}
    def _get(name):
        if name not in cache:
            s = get_scene(name)
            cache[name] = (s, *G.seam_inputs(orc, scene_mod, s))
        return cache[name]
    return _get


@pytest.mark.parametrize("name", ["tiny", "occ", "messy"])
def test_texture_patches_match_reference_tu(ref, orc, seam_inputs, name):
    """generate_texture_patches.cpp:453-538 (+ generate_candidate :78-138, merge_vertex_projection_infos :40-65) and the
    zero-adjust pass texrecon.cpp:174-183 (TexturePatch::adjust_colors, texture_patch.cpp:41-116) vs oracle/patches.py:
    same patches, faces, bit-identical texcoords, vertex projections, images, validity and blending masks."""
    import patches as P
    s, adj, rings, labels = seam_inputs(name)
    g = ref[0][f"texture_patches/{name}"]                      # label 0 (hole-filling patches, not restated) left out
    pp, pvpi = P.generate_texture_patches(orc, s, adj, labels)
    assert len(g["labels"]) == len(pp) >= s.num_views // 2
    for i, b in enumerate(pp):
        img, validity, blending = P.adjust_colors(b, np.zeros((3 * len(b.faces), 3), np.float32))
        mine = G.patch_digests([dict(faces=b.faces, texcoords=b.texcoords, image=img, validity=validity, blending=blending)],
                               ("faces", "texcoords", "validity", "blending", "image"))
        assert g["labels"][i] == b.label
        for field, d in mine.items():
            assert g[field][i] == d[0], field
    mine = [sorted((pid, np.asarray(proj, np.float32)) for pid, (proj, _f) in pvpi[v].items()) for v in range(s.verts.shape[0])]
    assert D(np.array([len(m) for m in mine], np.uint32)) == g["projection_count"]
    assert D(np.array([pid for m in mine for pid, _ in m], np.uint32)) == g["projection_patch"]
    assert D(np.array([xy for m in mine for _, xy in m], np.float32).reshape(-1, 2)) == g["projection_xy"]


@pytest.mark.parametrize("name", ["tiny", "occ", "messy"])
def test_global_seam_leveling_matches_reference_tu(ref, orc, seam_inputs, name):
    """tex::global_seam_leveling (global_seam_leveling.cpp:140-324: unknown numbering, Gamma, A, b from patch-relative
    edge samples, Lhs, CG per channel, mean subtraction, adjust_colors per patch) vs orc_global_seam_leveling +
    oracle/patches.apply_adjust_values.  The CG of both sides is the same restatement of Eigen's (shim / seam.c); the
    right-hand sides are sampled in patch vs view coordinates, so the adjusted images agree to rounding (2e-5)."""
    import patches as P
    s, adj, rings, labels = seam_inputs(name)
    g = ref[0][f"global_seam_leveling/{name}"]
    seam = orc.global_seam_leveling(s, rings, labels)
    pp, _ = P.generate_texture_patches(orc, s, adj, labels)
    pa = P.apply_adjust_values(s, pp, seam["row_ptr"], seam["row_label"], seam["x"])
    assert len(g["validity"]) == len(pa)
    moved = 0.0
    for i, (b, raw) in enumerate(zip(pa, pp)):
        assert g["validity"][i] == D(b.validity) and g["blending"][i] == D(b.blending)
        moved = max(moved, float(np.abs(b.image - raw.image)[b.validity != 0].max()))
    assert G.image_error(ref, f"global_seam_leveling/{name}", [b.image for b in pa]) < 2e-5
    assert moved > 0.02                                        # the leveling really changed the colours


def test_local_seam_leveling_matches_reference_tu(ref, orc, seam_inputs):
    """tex::local_seam_leveling (local_seam_leveling.cpp:105-204, draw_line :39-92, prepare_blending_mask
    texture_patch.cpp:197-297, poisson_blend poisson_blending.cpp:49-138) vs oracle/patches.local_seam_leveling.
    Both solve the same fp32 systems with a direct solver in double (shim elimination / scipy splu): 2e-5."""
    import patches as P
    s, adj, rings, labels = seam_inputs("tiny")
    g = ref[0]["local_seam_leveling/tiny"]
    seam = orc.global_seam_leveling(s, rings, labels)
    pp, pvpi = P.generate_texture_patches(orc, s, adj, labels)
    pa = P.apply_adjust_values(s, pp, seam["row_ptr"], seam["row_label"], seam["x"])
    before = [p.image.copy() for p in pa]
    P.local_seam_leveling(s, adj, labels, pa, pvpi)
    assert len(g["validity"]) == len(pa)
    changed = 0.0
    for i, (b, b0) in enumerate(zip(pa, before)):
        assert g["validity"][i] == D(b.validity)
        changed = max(changed, float(np.abs(b.image - b0).max()))
    assert G.image_error(ref, "local_seam_leveling/tiny", [b.image for b in pa]) < 2e-5
    assert changed > 0.01


def test_adjacency_of_non_manifold_mesh_matches_reference_tu(ref, scene_mod, get_scene):
    """An edge shared by three faces (a fin glued onto `tiny`): tex::build_adjacency_graph links all of them; the order of
    the adjacency lists is what scene.face_adjacency has to reproduce (face graphs with degree > 3 take the generic paths of
    the MRF kernels)."""
    verts, faces = G.mesh_with_fins(get_scene("tiny"))
    g = ref[0]["adjacency/tiny_with_fins"]
    a_ptr, a_idx = scene_mod.face_adjacency(faces)
    assert g["max_degree"] > 3
    assert D(a_ptr) == g["ptr"] and D(a_idx) == g["idx"]
