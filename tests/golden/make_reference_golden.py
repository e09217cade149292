"""Generates tests/golden/reference_tu.json and tests/golden/reference_tu.npz: what the reference's own translation units
return on the inputs of tests/test_ref_pinning.py and of the reference comparisons in tests/test_cuda_emulation.py, so
that those tests run where the reference is absent.  Storage format and inputs: tests/golden/reference_golden.py.

Needs oracle/_ref/libtexref.so (`make -C oracle ref REF=<checkout of the reference>`, see oracle/refshim/README.md).

    python tests/golden/make_reference_golden.py
"""
import importlib
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle"), os.path.dirname(os.path.abspath(__file__))]
import oracle as O  # noqa: E402
import patches as P  # noqa: E402
import reference_golden as G  # noqa: E402
import refpin as R  # noqa: E402

scene = importlib.import_module("mvs-texturing_b200.scene")
D = G.digest
PATCH_FIELDS = ("faces", "texcoords", "image", "validity", "blending")
js, arrays = {}, {}


def dc_digests(r):
    return dict(nnz=int(r["face_ptr"][-1]), face_ptr=D(r["face_ptr"]), view=D(r["view"]), cost=D(r["cost"]))


def store_images(key, ref_patches, orc_patches, **extra):
    """validity (+ extra) digests per patch and the image sample of the reference's patches."""
    pixels, values = G.image_sample([p.image for p in ref_patches], [p.image for p in orc_patches])
    k = key.replace("/", "_")
    arrays[k + "_pixels"], arrays[k + "_values"] = pixels, values
    js[key] = dict(validity=[D(p.validity) for p in ref_patches], pixels=sum(p.image.shape[0] * p.image.shape[1] for p in ref_patches),
                   **extra)


def zero_adjusted(patches):
    out = []
    for q in patches:
        img, val, bl = P.adjust_colors(q, np.zeros((3 * len(q.faces), 3), np.float32))
        z = P.Patch(q.label, q.faces, q.texcoords, img, q.bbox)
        z.validity, z.blending = val, bl
        out.append(z)
    return out


# ---- data costs ----------------------------------------------------------------------------------------------------
for name in ["tiny", "small", "occ", "messy"]:
    s = scene.config(name)
    for data_term in (1, 0):
        js[f"data_costs/{name}/{data_term}"] = dc_digests(R.data_costs(s, data_term=data_term))
for name in ["tiny", "occ"]:
    js[f"data_costs_no_visibility/{name}"] = dc_digests(R.data_costs(scene.config(name), visibility=False))
for mode in (1, 2):
    r = R.data_costs(scene.config("tiny"), outlier_removal=mode)
    js[f"outlier_removal/{mode}"] = dc_digests(r)
    arrays[f"outlier_removal_{mode}_cost"] = r["cost"]

# ---- validity mask, face infos, triangles, histogram, projection ---------------------------------------------------
img, img2 = G.validity_images()
arrays["validity_mask"] = R.validity_mask(img)
arrays["validity_mask_eroded"] = R.validity_mask(img, erode=True)
arrays["validity_mask_eroded_no_black"] = R.validity_mask(img2, erode=True)

s = scene.config("small")
tris = G.face_info_triangles(s, O.data_costs(s))
for data_term in (1, 0):
    arrays[f"face_quality_{data_term}"] = R.face_infos(s, G.FACE_INFO_VIEW, tris, data_term=data_term)[0]

draws, hist = G.triangle_and_histogram_draws()
arrays["tri_area"] = np.array([R.tri_area(*p) for p, x, y in draws], np.float32)
arrays["tri_inside"] = np.array([R.tri_inside(p[0], p[1], p[2], x, y) for p, x, y in draws], np.int32)
arrays["histogram_percentile"] = np.array([R.histogram_percentile(v, float(v.max())) for v in hist], np.float32)

s = scene.config("tiny")
arrays["pixel_coords"] = np.array([[R.pixel_coords(s, k, s.verts[i].copy()) for i in G.pixel_coord_vertices(s)]
                                   for k in G.PIXEL_COORD_VIEWS], np.float32)

# ---- adjacency graph and MRF model ---------------------------------------------------------------------------------
for name in ["tiny", "small", "occ", "C2s", "messy"]:
    s = scene.config(name)
    r_ptr, r_idx = R.build_adjacency(s.faces, s.verts.shape[0], scene.vertex_rings(s.faces, s.verts.shape[0]))
    js[f"adjacency/{name}"] = dict(ptr=D(r_ptr), idx=D(r_idx))
verts, faces = G.mesh_with_fins(scene.config("tiny"))
r_ptr, r_idx = R.build_adjacency(faces, verts.shape[0], scene.vertex_rings(faces, verts.shape[0]))
js["adjacency/tiny_with_fins"] = dict(ptr=D(r_ptr), idx=D(r_idx), max_degree=int(np.diff(r_ptr).max()))

for name in ["tiny", "occ"]:
    s = scene.config(name)
    dc = O.data_costs(s)
    if name == "tiny":
        dc = G.without_views(dc)
    m = R.view_selection_model(scene.face_adjacency(s.faces), dc["face_ptr"], dc["view"], dc["cost"], s.num_views)
    js[f"mrf_model/{name}"] = dict(edges=D(m["edges"]), ls_ptr=D(m["ls_ptr"]), ls_label=D(m["ls_label"]),
                                   ls_cost=D(m["ls_cost"]), labels=D(m["labels"]), params=m["params"])

# ---- texture patches, global and local seam leveling (label 0 = hole-filling patches, not restated: left out) -------
for name in ["tiny", "occ", "messy"]:
    s = scene.config(name)
    adj, rings, labels = G.seam_inputs(O, scene, s)
    rp, rvpi = R.seam_leveling(s, rings, adj, labels, do_global=False)
    rp = [p for p in rp if p.label != 0]
    n = len(rp)
    vp = [sorted((pid, xy) for pid, xy in rvpi[v].items() if pid < n) for v in range(s.verts.shape[0])]
    js[f"texture_patches/{name}"] = dict(
        labels=[int(p.label) for p in rp], **G.patch_digests(rp, PATCH_FIELDS),
        projection_count=D(np.array([len(x) for x in vp], np.uint32)),
        projection_patch=D(np.array([pid for x in vp for pid, _ in x], np.uint32)),
        projection_xy=D(np.array([xy for x in vp for _, xy in x], np.float32).reshape(-1, 2)))

    seam = O.global_seam_leveling(s, rings, labels)
    pp, pvpi = P.generate_texture_patches(O, s, adj, labels)
    pa = P.apply_adjust_values(s, pp, seam["row_ptr"], seam["row_label"], seam["x"])
    rp, _ = R.seam_leveling(s, rings, adj, labels, do_global=True)
    store_images(f"global_seam_leveling/{name}", [p for p in rp if p.label != 0], pa,
                 blending=[D(p.blending) for p in rp if p.label != 0])

    rp, _ = R.seam_leveling(s, rings, adj, labels, do_global=True, do_local=True)
    P.local_seam_leveling(s, adj, labels, pa, pvpi)
    store_images(f"local_seam_leveling/{name}", [p for p in rp if p.label != 0], pa)

    if name == "tiny":                                         # texrecon --skip_global_seam_leveling
        rp, _ = R.seam_leveling(s, rings, adj, labels, do_global=False, do_local=True)
        pz = zero_adjusted(pp)
        P.local_seam_leveling(s, adj, labels, pz, pvpi)
        store_images("local_seam_leveling_without_global/tiny", [p for p in rp if p.label != 0], pz)

# candidate merging: label islands inside the bounding box of another component of the same label
s = scene.config("small")
adj, rings, labels = G.seam_inputs(O, scene, s)
labels, islands = G.island_labels(O, s, adj, labels)
rp, _ = R.seam_leveling(s, rings, adj, labels, do_global=False)
js["texture_patches_with_islands/small"] = dict(islands=islands, labels=[int(p.label) for p in rp], **G.patch_digests(rp, PATCH_FIELDS))

json.dump(js, open(G.PATH + ".json", "w"), indent=1, sort_keys=True)
np.savez_compressed(G.PATH + ".npz", **arrays)
print(f"{G.PATH}.json: {os.path.getsize(G.PATH + '.json')} bytes, {G.PATH}.npz: {os.path.getsize(G.PATH + '.npz')} bytes")
