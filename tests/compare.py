"""Set-based comparison of SIFT outputs (SURVEY.md section 8c parity protocol) -- test helper."""
from __future__ import annotations

import hashlib

import numpy as np


def match_keypoints(kp_a: np.ndarray, kp_b: np.ndarray, tol_xy=0.5, tol_sig=0.05, tol_th=0.1):
    """One-to-one greedy matching of rows (x, y, sigma, theta) in input-image coordinates.

    Returns (pairs[(i, j)], precision, recall, f1); a is the candidate, b the reference."""
    na, nb = len(kp_a), len(kp_b)
    if na == 0 or nb == 0:
        return [], 0.0 if na else 1.0, 0.0 if nb else 1.0, 1.0 if na == nb else 0.0
    order = np.argsort(kp_b[:, 0], kind="stable")
    bx = kp_b[order, 0]
    cands = []
    for i in range(na):
        lo = np.searchsorted(bx, kp_a[i, 0] - tol_xy, "left")
        hi = np.searchsorted(bx, kp_a[i, 0] + tol_xy, "right")
        for jj in range(lo, hi):
            j = order[jj]
            if abs(kp_a[i, 1] - kp_b[j, 1]) >= tol_xy:
                continue
            if abs(kp_a[i, 2] - kp_b[j, 2]) >= tol_sig * kp_b[j, 2]:
                continue
            dth = abs(kp_a[i, 3] - kp_b[j, 3]) % (2 * np.pi)
            dth = min(dth, 2 * np.pi - dth)
            if dth >= tol_th:
                continue
            d = np.hypot(kp_a[i, 0] - kp_b[j, 0], kp_a[i, 1] - kp_b[j, 1]) + dth
            cands.append((d, i, j))
    cands.sort()
    used_a, used_b, pairs = set(), set(), []
    for d, i, j in cands:
        if i in used_a or j in used_b:
            continue
        used_a.add(i); used_b.add(j); pairs.append((i, j))
    prec = len(pairs) / na
    rec = len(pairs) / nb
    f1 = 2 * prec * rec / (prec + rec) if prec + rec > 0 else 0.0
    return pairs, prec, rec, f1


def descriptor_l2(desc_a, desc_b, pairs):
    if not pairs:
        return np.zeros(0)
    ia = np.array([p[0] for p in pairs]); ib = np.array([p[1] for p in pairs])
    return np.linalg.norm(desc_a[ia].astype(np.float64) - desc_b[ib].astype(np.float64), axis=1)


def report(kp_a, desc_a, kp_b, desc_b, **tol):
    pairs, p, r, f1 = match_keypoints(kp_a, kp_b, **tol)
    l2 = descriptor_l2(desc_a, desc_b, pairs)
    return {"n_a": len(kp_a), "n_b": len(kp_b), "matched": len(pairs), "precision": p, "recall": r,
            "f1": f1, "desc_l2_max": float(l2.max()) if len(l2) else 0.0,
            "desc_l2_median": float(np.median(l2)) if len(l2) else 0.0,
            "desc_l2_p99": float(np.percentile(l2, 99)) if len(l2) else 0.0}


def _feature_table(feat):
    """one uint32 row per feature: octave, x, y, sigma, num_ori, ori[4] (bits of the floats, -0.0 as 0.0, unused
    orientation slots 0), and the row order that sorts the table.  Takes this library's and the reference's records."""
    n = len(feat)
    t = np.zeros((n, 9), np.uint32)
    t[:, 0] = feat["octave"].astype(np.int32).view(np.uint32)
    for j, name in enumerate(("x", "y", "sigma"), 1):
        t[:, j] = (feat[name].astype(np.float32) + np.float32(0)).view(np.uint32)
    t[:, 4] = feat["num_ori"].astype(np.int32).view(np.uint32)
    used = np.arange(4)[None, :] < feat["num_ori"][:, None]
    t[:, 5:] = (np.where(used, feat["ori"], 0).astype(np.float32) + np.float32(0)).view(np.uint32)
    return t, np.lexsort(t.T[::-1])


def keypoint_digest(feat) -> str:
    """sha256 of a feature set (keypoints and their orientations, bit for bit, independent of the order)"""
    t, order = _feature_table(feat)
    return hashlib.sha256(np.ascontiguousarray(t[order]).tobytes()).hexdigest()


def descriptor_sample(feat, desc, desc_idx, k, seed=0):
    """k descriptors drawn with a fixed seed from the (feature, orientation) rows in sorted-table order:
    keys [k, 5] (octave, x, y, sigma, theta) and descriptors [k, 128]"""
    _, order = _feature_table(feat)
    rows = [(i, j) for i in order for j in range(int(feat["num_ori"][i]))]
    pick = [rows[p] for p in np.sort(np.random.default_rng(seed).choice(len(rows), min(k, len(rows)), replace=False))]
    keys = np.array([(feat["octave"][i], feat["x"][i], feat["y"][i], feat["sigma"][i], feat["ori"][i][j]) for i, j in pick],
                    np.float32).reshape(-1, 5)
    return keys, np.asarray(desc)[[int(desc_idx[i][j]) for i, j in pick]].astype(np.float32).reshape(-1, 128)


def sampled_descriptor_l2(feat, desc, desc_idx, keys, ref_desc):
    """L2 distance of each sampled reference descriptor to the descriptor of the same (keypoint, orientation) in
    `feat`/`desc`; a key that `feat` does not have is an AssertionError"""
    out = []
    for key, d in zip(keys, ref_desc):
        m = (feat["octave"] == int(key[0])) & (feat["x"] == key[1]) & (feat["y"] == key[2]) & (feat["sigma"] == key[3])
        hits = [(i, j) for i in np.nonzero(m)[0] for j in range(int(feat["num_ori"][i])) if feat["ori"][i][j] == key[4]]
        assert hits, ("sampled reference keypoint not found", key.tolist())
        i, j = hits[0]
        out.append(float(np.linalg.norm(desc[int(desc_idx[i][j])].astype(np.float64) - d.astype(np.float64))))
    return np.array(out)


def affine_scores(kp1, d1, kpk, dk, A):
    """repeatability: share of image-1 keypoints whose projection into image k lands within 2.5 px of a keypoint
    of comparable scale; matching score: share whose nearest descriptor in image k is that keypoint (the 800x640
    affine set of popsift_b200.synth.affine_set, 8 px border)"""
    p = kp1[:, :2] @ A[:, :2].T + A[:, 2]
    s = kp1[:, 2] * np.sqrt(abs(np.linalg.det(A[:, :2])))
    inside = (p[:, 0] > 8) & (p[:, 0] < 791) & (p[:, 1] > 8) & (p[:, 1] < 631)
    d2 = ((p[:, None, :] - kpk[None, :, :2]) ** 2).sum(-1)
    ok = (d2 < 2.5 ** 2) & (np.abs(np.log(s[:, None] / kpk[None, :, 2])) < np.log(1.4))
    rep = ok.any(1)[inside].mean()
    nn = np.argmin(((d1[:, None, :] - dk[None, :, :]) ** 2).sum(-1), axis=1)
    ms = ok[np.arange(len(kp1)), nn][inside].mean()
    return float(rep), float(ms)
