"""Shared parity checker: GPU results vs the oracle, with exact-t tie classification (SURVEY.md F3)."""
import hashlib
import json
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


REF_DIFF = ("differs from the unmodified reference's recorded result; with oracle/_ref built, "
            "tests/golden/make_reference_golden.py reruns the reference on the same inputs for a per-ray comparison")


def digest(*arrays):
    """SHA-256 over the dtype, shape and raw bytes of the arrays: a bit-for-bit fingerprint of a result of the
    unmodified reference that is too large to store (tests/golden/reference_digests.json)."""
    h = hashlib.sha256()
    for a in arrays:
        a = np.ascontiguousarray(a)
        h.update(f"{a.dtype.str}{a.shape}".encode())
        h.update(a.tobytes())
    return h.hexdigest()


def tree_digest(nodes, indices):
    """Node array + indices_.  A leaf's `axis` is never written by the reference (nanort.h:1795-1813): zeroed."""
    nodes = np.array(nodes, copy=True)
    nodes["axis"][nodes["flag"] != 0] = 0
    return digest(nodes, np.asarray(indices, np.uint32))


def hits_digest(hits, mask):
    """Hit flags of every ray + every field (padding aside) of the records of the rays that hit."""
    mask = np.asarray(mask, np.uint8)
    hit = mask == 1
    return digest(mask, *(hits[k][hit] for k in hits.dtype.names if k != "pad"))


def list_digest(lists):
    """Node-hit lists, one (t_min, t_max, node_id) triple of arrays per ray."""
    return digest(*(x for tmin, tmax, ids in lists for x in (np.array([len(ids)], np.int64), tmin, tmax, ids)))


def reference_golden():
    with open(os.path.join(GOLDEN, "reference_digests.json")) as f:
        return json.load(f)


def compare_hits(port, verts, faces, rays, got_hits, got_mask, want_hits, want_mask, topts=None, cpp11=True,
                 exact=True, rel_tol=1e-5):
    """Returns a dict of mismatch counts.  `exact`: t/u/v must match bit-for-bit; otherwise within rel_tol
    (the north star's 1e-5 relative).  A prim_id difference is a tie when the oracle, re-testing the GPU's
    primitive alone with the reference arithmetic, reports exactly the same t."""
    got_mask = got_mask.astype(bool)
    want_mask = want_mask.astype(bool)
    out = {"n": len(rays), "hits": int(want_mask.sum()), "mask_diff": int((got_mask != want_mask).sum()),
           "prim_diff": 0, "ties": 0, "near_ties": 0, "tuv_diff": 0}
    both = got_mask & want_mask
    g, w = got_hits[both], want_hits[both]
    pd = g["prim_id"] != w["prim_id"]
    idx_both = np.nonzero(both)[0]
    for j in np.nonzero(pd)[0]:
        ok, h = port.test_prim(verts, faces, rays[idx_both[j]], int(g["prim_id"][j]), topts=topts, cpp11=cpp11)
        # the GPU's record must be exactly what the reference arithmetic gives for that primitive
        valid = ok and all(h[k] == g[k][j] for k in ("t", "u", "v"))
        if valid and g["t"][j] == w["t"][j]:
            out["ties"] += 1
        elif valid and abs(float(g["t"][j]) - float(w["t"][j])) <= rel_tol * abs(float(w["t"][j])):
            # two different primitives (coplanar, overlapping) whose hits differ by an ulp or so: which one the
            # REFERENCE reports depends on its own visiting order, because its box test culls with the current
            # best t at that precision (SURVEY.md F3); t is within the north star's 1e-5
            out["near_ties"] += 1
        else:
            out["prim_diff"] += 1
    same = ~pd
    if exact:
        bad = np.zeros(same.sum(), bool)
        for k in ("t", "u", "v"):
            bad |= g[k][same].view(np.uint32) != w[k][same].view(np.uint32)
    else:
        bad = np.zeros(same.sum(), bool)
        for k in ("t", "u", "v"):
            a, b = g[k][same].astype(np.float64), w[k][same].astype(np.float64)
            bad |= np.abs(a - b) > rel_tol * np.maximum(np.abs(b), 1e-30) + 1e-12
    out["tuv_diff"] = int(bad.sum())
    return out


def assert_parity(res, allow_ties=True, max_near_ties=None):
    assert res["mask_diff"] == 0, res
    assert res["prim_diff"] == 0, res
    assert res["tuv_diff"] == 0, res
    if not allow_ties:
        assert res["ties"] == 0 and res["near_ties"] == 0, res
    if max_near_ties is not None:
        assert res["near_ties"] <= max_near_ties, res


def check_tree_structure(nodes, indices, verts, faces, min_leaf=4, max_depth=256, preorder=True):
    """Structural invariants every nanort-layout tree must satisfy (SURVEY.md section 4.3, 8b)."""
    n_prims = len(faces)
    n = len(nodes)
    assert n >= 1
    assert np.array_equal(np.sort(indices), np.arange(n_prims, dtype=np.uint32)), "each primitive exactly once"
    flag = nodes["flag"]
    assert np.all((flag == 0) | (flag == 1))
    leaf = flag == 1
    n_leaf, n_branch = int(leaf.sum()), int((~leaf).sum())
    assert n_leaf == n_branch + 1
    # exact triangle boxes
    tri = verts[faces]  # [nf,3,3]
    tmin, tmax = tri.min(axis=1), tri.max(axis=1)
    depth = np.zeros(n, np.int64)
    bmin = np.zeros((n, 3), np.float32)
    bmax = np.zeros((n, 3), np.float32)
    covered = np.zeros(n_prims, np.int64)
    # children always follow their parent in the array -> reverse sweep propagates boxes bottom-up
    d0, d1 = nodes["data"][:, 0].astype(np.int64), nodes["data"][:, 1].astype(np.int64)
    br = np.nonzero(~leaf)[0]
    assert np.all(d0[br] > br) and np.all(d1[br] > br) and np.all(d0[br] < n) and np.all(d1[br] < n)
    assert np.all((nodes["axis"][br] >= 0) & (nodes["axis"][br] <= 2))
    if preorder:
        assert np.all(d0[br] == br + 1), "left child directly follows its parent (DFS pre-order)"
    for i in range(n):
        if not leaf[i]:
            depth[d0[i]] = depth[i] + 1
            depth[d1[i]] = depth[i] + 1
    first = np.zeros(n, np.int64)
    count = np.zeros(n, np.int64)
    for i in range(n - 1, -1, -1):
        if leaf[i]:
            c, f0 = int(d0[i]), int(d1[i])
            assert c >= 1 and f0 + c <= n_prims
            p = indices[f0:f0 + c]
            covered[f0:f0 + c] += 1
            bmin[i], bmax[i] = tmin[p].min(axis=0), tmax[p].max(axis=0)
            first[i], count[i] = f0, c
            assert c <= min_leaf or depth[i] >= max_depth, (i, c, depth[i])
        else:
            a, b = d0[i], d1[i]
            bmin[i] = np.minimum(bmin[a], bmin[b])
            bmax[i] = np.maximum(bmax[a], bmax[b])
            assert first[a] + count[a] == first[b], "children cover adjacent index ranges"
            first[i], count[i] = first[a], count[a] + count[b]
    assert np.all(covered == 1), "leaves partition indices_"
    assert first[0] == 0 and count[0] == n_prims
    assert np.all(depth <= max_depth)
    # boxes are the exact float min/max of the member triangles (numerically: -0.0 == 0.0)
    assert np.array_equal(nodes["bmin"], bmin) and np.array_equal(nodes["bmax"], bmax), "exact node boxes"
    return {"max_tree_depth": int(depth.max()), "num_leaf_nodes": n_leaf, "num_branch_nodes": n_branch}
