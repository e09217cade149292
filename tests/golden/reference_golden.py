"""What the reference's own translation units returned, as stored in tests/golden/reference_tu.{json,npz}, and the inputs
they were run on.  Shared by tests/golden/make_reference_golden.py, which writes the data, and the tests that compare with
it, so that both build the very same inputs.

Results compared bit for bit are stored as digests (shape + bytes), results compared within a tolerance as values.  A
leveled image set is stored as a sample of its pixels: per patch a seeded share and the pixels farthest from the oracle,
plus the farthest pixels over all patches.
"""
import hashlib
import json
import os

import numpy as np

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "reference_tu")
IMAGE_SAMPLE, IMAGE_WORST, IMAGE_WORST_PER_PATCH = 1024, 256, 8


def digest(a) -> str:
    a = np.ascontiguousarray(a)
    return hashlib.sha256(str(a.shape).encode() + a.tobytes()).hexdigest()[:16]


def load():
    """(json dict, dict of arrays)"""
    with np.load(PATH + ".npz") as z:
        arrays = dict(z)
    with open(PATH + ".json") as f:
        return json.load(f), arrays


def patch_digests(patches, fields):
    """{field: [digest per patch]} of patch dicts or objects (faces as u32, texcoords as f32)."""
    get = lambda p, k: p[k] if isinstance(p, dict) else getattr(p, k)
    conv = dict(faces=lambda v: np.asarray(v, np.uint32), texcoords=lambda v: np.asarray(v, np.float32))
    return {k: [digest(conv.get(k, np.asarray)(get(p, k))) for p in patches] for k in fields}


def _flat(images):
    return np.concatenate([np.asarray(im, np.float32).reshape(-1, 3) for im in images])


def image_sample(images, closest):
    """Positions (in the concatenated pixels of all patches) and values of the stored pixels of `images`; `closest` is
    the oracle's image set, which decides which pixels are the farthest."""
    ref, diff = _flat(images), np.abs(_flat(images) - _flat(closest)).max(1)
    rng = np.random.RandomState(0)
    pick, start = [np.argsort(-diff, kind="stable")[:IMAGE_WORST]], 0
    for im in images:
        n = im.shape[0] * im.shape[1]
        pick.append(start + rng.choice(n, min(n, -(-IMAGE_SAMPLE * n // len(ref))), replace=False))
        pick.append(start + np.argsort(-diff[start:start + n], kind="stable")[:IMAGE_WORST_PER_PATCH])
        start += n
    pick = np.unique(np.concatenate(pick))
    return pick.astype(np.uint32), ref[pick]


def image_error(golden, key, images):
    """Largest difference of `images` from the stored pixels of the reference's image set `key`."""
    img = _flat(images)
    assert len(img) == golden[0][key]["pixels"], "number of patch pixels differs from the reference's"
    k = key.replace("/", "_")
    return float(np.abs(golden[1][k + "_values"] - img[golden[1][k + "_pixels"]]).max())


# ---- inputs --------------------------------------------------------------------------------------------------------
def validity_images():
    """An image with black frame pieces connected to the corners and an interior black blob, and one without black."""
    rng = np.random.RandomState(5)
    img = rng.randint(1, 255, size=(40, 56, 3)).astype(np.uint8)
    img[:6, :] = 0; img[:, :4] = 0; img[30:, 50:] = 0          # black frame pieces connected to corners
    img[15:18, 20:23] = 0                                     # an interior black blob: stays valid
    img2 = rng.randint(1, 255, size=(20, 20, 3)).astype(np.uint8)
    return img, img2


FACE_INFO_VIEW = 3


def face_info_triangles(scene, dc, k=FACE_INFO_VIEW):
    """Triangles around faces seen by view k (data costs `dc`), at every size class: as is, shrunk to sub-pixel size,
    stretched, and slivers."""
    rng = np.random.RandomState(11)
    faces = [f for f in range(scene.num_faces) if k in dc["view"][int(dc["face_ptr"][f]):int(dc["face_ptr"][f + 1])]]
    tris = []
    for f in faces[:300]:
        t = scene.verts[scene.faces[f]].astype(np.float32)
        c = t.mean(axis=0)
        for scale in (1.0, 0.05, 3.0):
            tris.append((c + (t - c) * np.float32(scale)).astype(np.float32))
        sl = t.copy(); sl[2] = (sl[0] + (sl[1] - sl[0]) * np.float32(0.5) + rng.normal(0, 1e-4, 3)).astype(np.float32)
        tris.append(sl)
    return np.array(tris, np.float32)


HISTOGRAM_SIZES = (1, 7, 1000, 200000)


def triangle_and_histogram_draws():
    """300 (triangle, x, y) draws and one value set per HISTOGRAM_SIZES entry."""
    rng = np.random.RandomState(3)
    tris = []
    for _ in range(300):
        p = rng.uniform(0, 50, size=(3, 2)).astype(np.float32)
        x, y = rng.uniform(0, 50, size=2).astype(np.float32)
        tris.append((p, x, y))
    return tris, [(rng.gamma(2.0, 3.0, size=n)).astype(np.float32) for n in HISTOGRAM_SIZES]


PIXEL_COORD_VIEWS = (0, 5)


def pixel_coord_vertices(scene):
    return range(0, scene.verts.shape[0], 37)


def mesh_with_fins(scene):
    """`scene` with three fins glued onto existing edges (an edge shared by three faces): (verts, faces)."""
    s = scene
    verts = np.concatenate([s.verts, (s.verts[s.faces[5]].mean(0) * 1.3)[None].astype(np.float32),
                            (s.verts[s.faces[40]].mean(0) * 1.3)[None].astype(np.float32)], 0)
    nv = verts.shape[0]
    fins = np.array([[s.faces[5][0], s.faces[5][1], nv - 2], [s.faces[5][1], s.faces[5][2], nv - 2],
                     [s.faces[40][2], s.faces[40][0], nv - 1]], np.uint32)
    return verts, np.ascontiguousarray(np.concatenate([s.faces, fins], 0))


def without_views(dc, faces=(3, 17, 18, 200)):
    """Data costs with every entry of `faces` removed (those faces become unseen)."""
    keep = np.ones(len(dc["view"]), bool)
    ptr = dc["face_ptr"].astype(np.int64)
    for f in faces:
        keep[ptr[f]:ptr[f + 1]] = False
    cnt = np.add.reduceat(keep.astype(np.int64), ptr[:-1]) * (ptr[1:] > ptr[:-1])
    return dict(face_ptr=np.r_[0, np.cumsum(cnt)].astype(np.uint64), view=dc["view"][keep], cost=dc["cost"][keep])


def seam_inputs(orc, scene_mod, scene):
    """(adjacency, vertex rings, the oracle's labels) of a scene."""
    adj = scene_mod.face_adjacency(scene.faces)
    rings = scene_mod.vertex_rings(scene.faces, scene.verts.shape[0])
    dc = orc.data_costs(scene)
    labels = orc.view_selection(adj[0], adj[1], dc["face_ptr"], dc["view"], dc["cost"], threads=1)["labels"]
    return adj, rings, labels


def island_labels(orc, scene, adj, labels):
    """`labels` with up to six one-face islands: the three neighbours of a face inside a one-label region (two rings deep)
    move to another view that sees all three, which cuts the face off from its component.  Returns (labels, islands)."""
    s = scene
    dc = orc.data_costs(s)
    labels = labels.copy()
    ptr = dc["face_ptr"].astype(np.int64)
    vis = [set((dc["view"][ptr[f]:ptr[f + 1]] + 1).tolist()) for f in range(s.num_faces)]
    nb = lambda f: [int(a) for a in adj[1][adj[0][f]:adj[0][f + 1]]]
    islands, used = 0, set()
    for f in range(s.num_faces):
        L = labels[f]
        ring1 = nb(f)
        if len(ring1) != 3 or any(labels[a] != L for a in ring1):
            continue
        ring2 = set(b for a in ring1 for b in nb(a)) - {f} - set(ring1)
        if any(labels[b] != L for b in ring2) or used & ({f} | set(ring1) | ring2):
            continue
        common = set.intersection(*[vis[a] for a in ring1]) - {int(L)}
        if not common:
            continue
        for a in ring1:
            labels[a] = min(common)          # cut face f off from its component
        used |= {f} | set(ring1) | ring2
        islands += 1
        if islands >= 6:
            break
    return labels, islands
