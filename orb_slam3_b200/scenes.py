"""Synthetic matching scenes on top of extracted keypoints (SURVEY.md 8d,
configs 2 and 3).  Pure numpy; shared by the tests and bench.py."""
import numpy as np

from .views import make_featvec_view, make_frame_view, make_lastframe_view, make_mappoint_view

FX = FY = 700.0


def scale_factors(nlevels=8, sf=1.2):
    s = [np.float32(1.0)]
    for _ in range(1, nlevels):
        s.append(np.float32(np.float64(s[-1]) * np.float64(np.float32(sf))))
    return np.array(s, np.float32)


def flip_bits(desc, nflip, rng):
    d = desc.copy()
    n = len(d)
    for _ in range(nflip):
        byte = rng.integers(0, 32, n)
        bit = rng.integers(0, 8, n)
        d[np.arange(n), byte] ^= (1 << bit).astype(np.uint8)
    return d


def stereo_u_right(kps, rng, frac=0.8, bf=386.0):
    """mvuRight: `frac` of the keypoints get a right coordinate from a random depth."""
    n = len(kps)
    depth = rng.uniform(4, 40, n).astype(np.float32)
    ur = (kps["x"] - np.float32(bf) / depth).astype(np.float32)
    ur[rng.random(n) > frac] = -1.0
    return ur


def last_frame_scene(last_kps, last_desc, cur_kps, cur_desc, width, height, shift, seed, stereo=False,
                     depth=8.0, obs0_frac=0.1, nomp_frac=0.15, taken_frac=0.05):
    """Frame t (last) -> frame t+1 (current) for SearchByProjection(Cur, Last): every
    last keypoint carries a MapPoint at `depth` in front of the last camera; the
    current pose is the pure translation that moves projections by `shift` px."""
    rng = np.random.default_rng(seed)
    sf = scale_factors()
    cx, cy = width / 2.0, height / 2.0
    n = len(last_kps)
    z = np.full(n, depth, np.float32) * rng.uniform(0.7, 1.4, n).astype(np.float32)
    X = np.stack([(last_kps["x"] - cx) / FX * z, (last_kps["y"] - cy) / FY * z, z], 1).astype(np.float32)
    t = np.array([shift[0] * depth / FX, shift[1] * depth / FY, 0.0], np.float32)
    Tcw = np.concatenate([[0, 0, 0, 1], t]).astype(np.float32)
    if seed % 2:  # a small rotation about z so the quaternion path is exercised
        a = 0.01
        Tcw[:4] = [0, 0, np.sin(a / 2), np.cos(a / 2)]
    has_mp = (rng.random(n) > nomp_frac)
    has_obs = (rng.random(n) > obs0_frac)
    mp_desc = flip_bits(last_desc, 3, rng)
    bf = 386.0 if stereo else 0.0
    ur = stereo_u_right(cur_kps, rng) if stereo else None
    taken = (rng.random(len(cur_kps)) < taken_frac).astype(np.uint8)
    cur = make_frame_view(cur_kps, cur_desc, width, height, sf, u_right=ur, kp_taken=taken, fx=FX, fy=FY,
                          cx=cx, cy=cy, bf=bf, b=bf / FX)
    last = make_lastframe_view(X, mp_desc, last_kps["octave"], last_kps["angle"], has_mp, has_obs)
    return cur, last, Tcw


def local_map_scene(kps, desc, width, height, n_extra, seed, stereo=False, th_noise=1.0, taken_frac=0.3):
    """SearchByProjection(F, vpMapPoints): one MapPoint per keypoint (projection =
    keypoint + N(0, th_noise) px, predicted level = octave) plus n_extra random ones."""
    rng = np.random.default_rng(seed)
    sf = scale_factors()
    n = len(kps)
    sel = rng.permutation(n)
    px = np.concatenate([kps["x"][sel] + rng.normal(0, th_noise, n), rng.uniform(20, width - 20, n_extra)])
    py = np.concatenate([kps["y"][sel] + rng.normal(0, th_noise, n), rng.uniform(20, height - 20, n_extra)])
    lvl = np.concatenate([kps["octave"][sel], rng.integers(0, 8, n_extra)])
    lvl = np.clip(lvl + (rng.random(n + n_extra) < 0.2) * rng.integers(-1, 2, n + n_extra), 0, 7)
    d = np.concatenate([flip_bits(desc[sel], 6, rng), rng.integers(0, 256, (n_extra, 32), dtype=np.uint8)])
    m = n + n_extra
    order = rng.permutation(m)
    vcos = np.where(rng.random(m) < 0.5, 0.9995, 0.9).astype(np.float32)
    depth = rng.uniform(2, 80, m).astype(np.float32)
    ur = stereo_u_right(kps, rng) if stereo else None
    pxr = (px - 386.0 / depth).astype(np.float32) if stereo else None
    mps = make_mappoint_view(px[order], py[order], lvl[order], d[order], view_cos=vcos[order],
                             proj_xr=None if pxr is None else pxr[order], depth=depth[order],
                             track_in_view=(rng.random(m) > 0.1), is_bad=(rng.random(m) < 0.02),
                             has_obs=(rng.random(m) > 0.1))
    taken = (rng.random(n) < taken_frac).astype(np.uint8)
    F = make_frame_view(kps, desc, width, height, sf, u_right=ur, kp_taken=taken, fx=FX, fy=FY, bf=386.0 if stereo else 0.0)
    return F, mps


def triangulation_scene(kps1, desc1, kps2, desc2, width, height, seed, n_nodes=1000, stereo=True,
                        shift=(5.0, -3.0)):
    """SearchForTriangulation: FeatureVectors bucket features by a descriptor hash
    (DBoW2 itself is out of scope), KF2 = KF1 translated along x (rectified pair
    geometry: F12 = [t]x for identical intrinsics up to scale)."""
    rng = np.random.default_rng(seed)
    sf = scale_factors()

    def nodes(desc):
        w = desc[:, :2].astype(np.int64)
        return ((w[:, 0] >> 3) * 32 + (w[:, 1] >> 3)) % n_nodes

    n1, n2 = len(kps1), len(kps2)
    node1, node2 = nodes(desc1), nodes(desc2)
    node1[rng.random(n1) < 0.02] = -1
    ur1 = stereo_u_right(kps1, rng, 0.6) if stereo else None
    ur2 = stereo_u_right(kps2, rng, 0.6) if stereo else None
    k1 = make_frame_view(kps1, desc1, width, height, sf, u_right=ur1, kp_taken=(rng.random(n1) < 0.4), fx=FX, fy=FY)
    k2 = make_frame_view(kps2, desc2, width, height, sf, u_right=ur2, kp_taken=(rng.random(n2) < 0.4), fx=FX, fy=FY)
    cx, cy = width / 2.0, height / 2.0
    K = np.array([[FX, 0, cx], [0, FY, cy], [0, 0, 1]], np.float64)
    R = np.eye(3)
    # translation (almost) parallel to the image plane along the image shift between the two
    # frames, so true correspondences satisfy the epipolar test
    t = np.array([shift[0] * 0.02, shift[1] * 0.02, 0.003])
    tx = np.array([[0, -t[2], t[1]], [t[2], 0, -t[0]], [-t[1], t[0], 0]])
    F12 = (np.linalg.inv(K).T @ tx @ R @ np.linalg.inv(K)).astype(np.float32)
    ep = np.array([FX * t[0] / t[2] + cx, FY * t[1] / t[2] + cy], np.float32)
    return k1, k2, make_featvec_view(node1), make_featvec_view(node2), F12.reshape(9), ep


def hash_nodes(desc, n_nodes=1000):
    """A FeatureVector stand-in without a vocabulary: node of a feature = a hash of its first two descriptor bytes."""
    w = np.asarray(desc)[:, :2].astype(np.int64)
    return ((w[:, 0] >> 3) * 32 + (w[:, 1] >> 3)) % n_nodes


def nodes_from_featvec(n, fv_node_ids, fv_ptr, fv_idx):
    """Per-feature node id (-1 = not in the vector) of a FeatureVector CSR, e.g. the output of bow_transform."""
    node = -np.ones(n, np.int64)
    for k, nid in enumerate(fv_node_ids):
        node[fv_idx[fv_ptr[k]:fv_ptr[k + 1]]] = int(nid)
    return node


def bow_match_scene(n, seed, node_of, width=1280, height=720, bad_frac=0.3, dup_frac=0.1, outlier_frac=0.15,
                    max_flip=60):
    """SearchByBoW: two views of one set of n keypoints.  View 2 holds a permuted (1 - dup_frac - outlier_frac) share
    of view 1's keypoints with each descriptor perturbed by 0..max_flip flipped bits, dup_frac second copies of some
    of them (near ties for the ratio test), and outlier_frac gross outliers (random descriptors).  Its angles are view
    1's minus an offset drawn around 0, 30, 75, 200 and 355 degrees, so the matches fill several rotation bins.
    bad_frac of the map points of either side are missing or bad.  node_of(desc) -> node id per feature (-1 = not in
    the FeatureVector), e.g. the vocabulary descent of DBoW2::transform at some levelsup, or hash_nodes.
    Returns dict(kf1, ok1, fv1, kf2, ok2, fv2): view 1 is the keyframe (query side), view 2 the frame or second
    keyframe."""
    from ._lib import KP_DTYPE
    rng = np.random.default_rng(seed)
    sf = scale_factors()

    def keypoints(x, y, angle, octave):
        k = np.zeros(len(x), KP_DTYPE)
        k["x"], k["y"], k["angle"], k["octave"] = x, y, angle, octave
        k["size"] = 31.0 * sf[octave]
        k["response"] = rng.uniform(10, 100, len(x))
        k["class_id"] = -1
        return k

    ang1 = rng.uniform(0, 360, n).astype(np.float32)
    oct1 = rng.integers(0, 8, n)
    k1 = keypoints(rng.uniform(20, width - 20, n), rng.uniform(20, height - 20, n), ang1, oct1)
    d1 = rng.integers(0, 256, (n, 32), dtype=np.uint8)
    n_dup, n_out = int(dup_frac * n), int(outlier_frac * n)
    base = rng.permutation(n)[:n - n_dup - n_out]
    rows = np.concatenate([base, rng.choice(base, n_dup)]) if len(base) else base
    d2 = d1[rows].copy()
    for i, k in enumerate(rng.integers(0, max_flip + 1, len(rows))):
        bits = np.unpackbits(d2[i])
        bits[rng.choice(256, k, replace=False)] ^= 1
        d2[i] = np.packbits(bits)
    d2 = np.concatenate([d2, rng.integers(0, 256, (n_out, 32), dtype=np.uint8)])
    offset = rng.choice([0.0, 30.0, 75.0, 200.0, 355.0], len(rows), p=[0.4, 0.2, 0.15, 0.1, 0.15])
    ang2 = np.mod(ang1[rows] - offset - rng.uniform(-8, 8, len(rows)), 360.0)
    ang2 = np.concatenate([ang2, rng.uniform(0, 360, n_out)]).astype(np.float32)
    ang2[ang2 >= 360.0] = 0.0
    x2 = np.concatenate([k1["x"][rows] + rng.normal(0, 2, len(rows)), rng.uniform(20, width - 20, n_out)])
    y2 = np.concatenate([k1["y"][rows] + rng.normal(0, 2, len(rows)), rng.uniform(20, height - 20, n_out)])
    oct2 = np.concatenate([oct1[rows], rng.integers(0, 8, n_out)])
    order = rng.permutation(len(d2))
    k2 = keypoints(x2[order], y2[order], ang2[order], oct2[order])
    d2 = np.ascontiguousarray(d2[order])
    kf1 = make_frame_view(k1, d1, width, height, sf, fx=FX, fy=FY)
    kf2 = make_frame_view(k2, d2, width, height, sf, fx=FX, fy=FY)
    return dict(kf1=kf1, ok1=(rng.random(n) >= bad_frac).astype(np.uint8), fv1=make_featvec_view(node_of(d1)),
                kf2=kf2, ok2=(rng.random(len(d2)) >= bad_frac).astype(np.uint8), fv2=make_featvec_view(node_of(d2)))


# ---------------------------------------------------------------- local BA graphs
def _quat_from_yaw_pitch(yaw, pitch):
    cy, sy, cp, sp = np.cos(yaw / 2), np.sin(yaw / 2), np.cos(pitch / 2), np.sin(pitch / 2)
    # R = Ry(yaw) * Rx(pitch)
    return np.array([cy * sp, sy * cp, -sy * sp, cy * cp])


def _quat_mul(a, b):
    ax, ay, az, aw = a
    bx, by, bz, bw = b
    return np.array([aw * bx + ax * bw + ay * bz - az * by, aw * by + ay * bw + az * bx - ax * bz,
                     aw * bz + az * bw + ax * by - ay * bx, aw * bw - ax * bx - ay * by - az * bz])


def _quat_rot(q, v):
    u = np.cross(q[:3], v)
    u = u + u
    return v + q[3] * u + np.cross(q[:3], u)


def _qrot_many(q, v):
    """Rotate v[...,3] by quaternions q[...,4] (x,y,z,w), broadcasting."""
    qv = q[..., :3]
    u = np.cross(qv, v)
    u = u + u
    return v + q[..., 3:4] * u + np.cross(qv, u)


def lba_graph(n_kf_opt, n_mp, seed=0, fixed_frac=0.1, stereo_frac=0.8, outlier_frac=0.02,
              width=1280, height=720, fx=700.0, bf=386.0):
    """Synthetic LocalBundleAdjustment graph (SURVEY.md 8d, configs 4/5): K optimisable
    KFs on a smooth trajectory (1 m spacing, yaw drift) + ceil(K/10) fixed ones,
    landmarks seen by 3..10 KFs of a sliding window, 80% stereo edges, octave noise
    model, 2% gross outliers, perturbed initial estimates.  Returns (graph dict, truth)."""
    rng = np.random.default_rng(seed)
    n_fixed = int(np.ceil(n_kf_opt * fixed_frac))
    K = n_kf_opt + n_fixed
    cx, cy = width / 2.0, height / 2.0
    k_idx = np.arange(K)
    Twc_q = np.stack([_quat_from_yaw_pitch(0.01 * k + 0.05 * np.sin(0.3 * k), 0.01 * np.cos(0.2 * k)) for k in k_idx])
    Twc_t = np.stack([0.3 * np.sin(0.1 * k_idx), (0.02 * k_idx) % 0.3, 1.0 * k_idx], 1)
    Tcw = np.zeros((K, 7))
    Tcw[:, :4] = Twc_q * np.array([-1, -1, -1, 1])
    Tcw[:, 4:] = -_qrot_many(Tcw[:, :4], Twc_t)
    fixed = np.zeros(K, np.uint8)
    fixed[:n_fixed] = 1  # the oldest KFs see local points but are not local KFs
    inv_sigma2 = (1.0 / (scale_factors() ** 2)).astype(np.float32)

    pts_l, ekf_l, emp_l = [], [], []
    have = 0
    while have < n_mp:
        m_try = int((n_mp - have) * 1.3) + 64
        k0 = rng.integers(0, K, m_try)
        depth = rng.uniform(4, 40, m_try)
        u = rng.uniform(40, width - 40, m_try)
        v = rng.uniform(40, height - 40, m_try)
        Xc = np.stack([(u - cx) / fx * depth, (v - cy) / fx * depth, depth], 1)
        Xw = _qrot_many(Twc_q[k0], Xc) + Twc_t[k0]
        offs = np.arange(-7, 8)
        kk = k0[:, None] + offs[None, :]                      # candidate observers (window)
        inb = (kk >= 0) & (kk < K)
        kc = np.clip(kk, 0, K - 1)
        Xk = _qrot_many(Tcw[kc, :4], Xw[:, None, :]) + Tcw[kc, 4:]
        zz = Xk[..., 2]
        with np.errstate(divide="ignore", invalid="ignore"):
            uu = fx * Xk[..., 0] / zz + cx
            vv = fx * Xk[..., 1] / zz + cy
        vis = inb & (zz >= 1.0) & (uu >= 0) & (uu < width) & (vv >= 0) & (vv < height)
        want = rng.integers(3, 11, m_try)
        pri = np.where(vis, rng.random(vis.shape), 2.0)        # keep `want` random visible observers
        rank = np.argsort(np.argsort(pri, axis=1), axis=1)
        keep = vis & (rank < want[:, None])
        nobs = keep.sum(1)
        free_seen = (keep & (fixed[kc] == 0)).any(1)
        ok = np.nonzero((nobs >= 3) & free_seen)[0][: n_mp - have]
        for j, l_src in enumerate(ok):
            ks = kc[l_src][keep[l_src]]
            ekf_l.append(ks)
            emp_l.append(np.full(len(ks), have + j))
        pts_l.append(Xw[ok])
        have += len(ok)
    pts = np.concatenate(pts_l)
    e_kf = np.concatenate(ekf_l).astype(np.int32)
    e_mp = np.concatenate(emp_l).astype(np.int32)
    E = len(e_kf)
    Xk = _qrot_many(Tcw[e_kf, :4], pts[e_mp]) + Tcw[e_kf, 4:]
    uu = fx * Xk[:, 0] / Xk[:, 2] + cx
    vv = fx * Xk[:, 1] / Xk[:, 2] + cy
    octv = rng.integers(0, 8, E)
    sig = 1.2 ** octv
    noise = rng.normal(0, 1, (E, 3)) * sig[:, None]
    out = rng.random(E) < outlier_frac
    noise[out, 0] += rng.choice([-50.0, 50.0], out.sum())
    e_st = (rng.random(E) < stereo_frac).astype(np.uint8)
    ur = np.where(e_st == 1, (uu - bf / Xk[:, 2] + noise[:, 2]).astype(np.float32), np.float32(-1.0))
    e_obs = np.stack([(uu + noise[:, 0]).astype(np.float32), (vv + noise[:, 1]).astype(np.float32), ur], 1).astype(np.float64)
    e_is2 = inv_sigma2[octv]
    truth = dict(kf_pose=Tcw.copy(), mp_pos=pts.copy())
    # initial perturbation: poses 2 cm / 0.5 deg (free KFs only), points 5 cm
    pose0 = Tcw.copy()
    for k in range(K):
        if fixed[k]:
            continue
        w = rng.normal(0, np.deg2rad(0.5) / np.sqrt(3), 3)
        th = np.linalg.norm(w)
        dq = np.concatenate([np.sin(th / 2) * w / max(th, 1e-12), [np.cos(th / 2)]])
        pose0[k, :4] = _quat_mul(dq, Tcw[k, :4])
        pose0[k, 4:] = _quat_rot(dq, Tcw[k, 4:]) + rng.normal(0, 0.02 / np.sqrt(3), 3)
    # Sophus stores float poses; LocalBundleAdjustment casts them to double (:1216-1217)
    pose0 = pose0.astype(np.float32).astype(np.float64)
    pts0 = (pts + rng.normal(0, 0.05 / np.sqrt(3), pts.shape)).astype(np.float32).astype(np.float64)
    cam = np.tile(np.array([fx, fx, cx, cy, bf], np.float32), (K, 1))
    g = dict(kf_pose=pose0, kf_fixed=fixed, kf_cam=cam, mp_pos=pts0, e_kf=e_kf, e_mp=e_mp, e_stereo=e_st,
             e_obs=e_obs, e_inv_sigma2=e_is2.astype(np.float32))
    return g, truth


def kb8_project(p8, X):
    """KannalaBrandt8::project (KannalaBrandt8.cpp:46-65) of points X[...,3], p8 = fx, fy, cx, cy, k0..k3; fp64 throughout
    (scene generation only: the solvers restate the float atan2f / sqrtf of the reference themselves)."""
    r = np.hypot(X[..., 0], X[..., 1])
    th = np.arctan2(r, X[..., 2])
    psi = np.arctan2(X[..., 1], X[..., 0])
    t2 = th * th
    rd = th * (1 + t2 * (p8[4] + t2 * (p8[5] + t2 * (p8[6] + t2 * p8[7]))))
    return np.stack([p8[0] * rd * np.cos(psi) + p8[2], p8[1] * rd * np.sin(psi) + p8[3]], -1)


def lba_rig_graph(n_kf_opt, n_mp, seed=0, model1=1, model2=1, right_frac=0.6, left_drop=0.15, mono_only=False):
    """LocalBundleAdjustment graph of a two-camera rig (SURVEY.md 8a row a17; Optimizer.cc:1305-1331 + :1366-1400):
    the geometry of `lba_graph`, observed by a left camera (mono edges, EdgeSE3ProjectXYZ with pCamera = mpCamera)
    and a right camera at Trl (body edges, EdgeSE3ProjectXYZToBody with pCamera = mpCamera2); model 1 =
    KannalaBrandt8 (TUM-VI-like intrinsics), 0 = Pinhole.  A landmark seen by a keyframe has a left observation, a
    right one, or both (the two edges then share the pose and the landmark).  `mono_only`: a monocular fisheye rig
    (no second camera, no body edges).  Returns (graph dict incl. the rig fields of lba_graph_view, truth)."""
    g, truth = lba_graph(n_kf_opt, n_mp, seed=seed, stereo_frac=0.0)
    rng = np.random.default_rng(seed + 7919)
    K, E = len(g["kf_fixed"]), len(g["e_kf"])
    kb_l = np.array([190.97, 190.97, 254.93, 256.89, 0.0034823894, 0.0007150348, -0.0020532361, 0.00020293673], np.float32)
    kb_r = np.array([190.44, 190.44, 252.59, 254.94, 0.0034003171, 0.0017662782, -0.0026631420, 0.00032997288], np.float32)
    ph_l = np.array([700.0, 700.0, 640.0, 360.0, 0, 0, 0, 0], np.float32)
    ph_r = np.array([705.0, 698.0, 633.0, 366.0, 0, 0, 0, 0], np.float32)
    c1 = kb_l if model1 == 1 else ph_l
    c2 = kb_r if model2 == 1 else ph_r
    # Trl: 10 cm baseline and a small relative rotation (a real calibration is never the identity)
    w = np.array([0.004, -0.011, 0.007])
    th = np.linalg.norm(w)
    q_rl = np.concatenate([np.sin(th / 2) * w / th, [np.cos(th / 2)]])
    t_rl = np.array([-0.1009, 0.0019, 0.0012])
    trl = np.concatenate([q_rl, t_rl]).astype(np.float32).astype(np.float64)  # Sophus::SE3f cast to double (:1384-1385)
    trl[:4] /= np.linalg.norm(trl[:4])

    def proj(model, c, X):
        if model == 1:
            return kb8_project(c.astype(np.float64), X)
        return np.stack([c[0] * X[:, 0] / X[:, 2] + c[2], c[1] * X[:, 1] / X[:, 2] + c[3]], -1)

    Tcw, pts = truth["kf_pose"], truth["mp_pos"]
    Xl = _qrot_many(Tcw[g["e_kf"], :4], pts[g["e_mp"]]) + Tcw[g["e_kf"], 4:]
    Xr = _qrot_many(trl[None, :4], Xl) + trl[None, 4:]
    octv = rng.integers(0, 8, (E, 2))
    sig = 1.2 ** octv
    uv_l = proj(model1, c1, Xl) + rng.normal(0, 1, (E, 2)) * sig[:, :1]
    uv_r = proj(model2, c2, Xr) + rng.normal(0, 1, (E, 2)) * sig[:, 1:]
    out = rng.random((E, 2)) < 0.02
    uv_l[out[:, 0], 0] += rng.choice([-50.0, 50.0], out[:, 0].sum())
    uv_r[out[:, 1], 1] += rng.choice([-50.0, 50.0], out[:, 1].sum())
    has_r = (rng.random(E) < right_frac) & (not mono_only)
    has_l = ~(has_r & (rng.random(E) < left_drop))
    inv_sigma2 = (1.0 / (scale_factors() ** 2)).astype(np.float32)
    il, ir = np.nonzero(has_l)[0], np.nonzero(has_r)[0]
    # per landmark: the observing keyframes in order, a keyframe's left edge before its right one (:1296-1400)
    order = np.argsort(np.concatenate([2 * il, 2 * ir + 1]), kind="stable")
    src = np.concatenate([il, ir])[order]
    typ = np.concatenate([np.zeros(len(il), np.uint8), np.full(len(ir), 2, np.uint8)])[order]
    obs = np.where((typ == 0)[:, None], uv_l[src], uv_r[src]).astype(np.float32).astype(np.float64)
    h = dict(g)
    h["e_kf"], h["e_mp"], h["e_stereo"] = g["e_kf"][src], g["e_mp"][src], typ
    h["e_obs"] = np.concatenate([obs, np.full((len(src), 1), -1.0)], 1)
    h["e_inv_sigma2"] = np.where(typ == 0, inv_sigma2[octv[src, 0]], inv_sigma2[octv[src, 1]]).astype(np.float32)
    h["kf_cam"] = np.tile(np.concatenate([c1[:4], [0.0]]).astype(np.float32), (K, 1))  # mbf unused: no stereo edges
    h["kf_cam_model"] = np.full(K, model1, np.uint8)
    h["kf_cam_dist"] = np.tile(c1[4:], (K, 1))
    if not mono_only:
        h["kf_cam2_model"] = np.full(K, model2, np.uint8)
        h["kf_cam2"] = np.tile(c2, (K, 1))
        h["kf_trl"] = np.tile(trl, (K, 1))
    return h, truth


def lba_rough_graph(seed=4):
    """Small graph with a wild start and almost no damping: forces rejected LM trials."""
    g, truth = lba_graph(5, 60, seed=seed)
    rng = np.random.default_rng(seed)
    g["mp_pos"] = g["mp_pos"] + rng.normal(0, 5.0, g["mp_pos"].shape)
    g["kf_pose"][:, 4:] += rng.normal(0, 0.3, (len(g["kf_pose"]), 3)) * (g["kf_fixed"][:, None] == 0)
    return g, truth


def permute_keyframes(g, perm):
    """The same graph with its keyframes listed in another order (new index i = old keyframe perm[i]):
    LocalBundleAdjustment collects the local keyframes from covisibility lists, not along the trajectory."""
    perm = np.asarray(perm)
    inv = np.empty_like(perm)
    inv[perm] = np.arange(len(perm))
    h = dict(g)
    for k in ("kf_pose", "kf_fixed", "kf_cam", "kf_cam_model", "kf_cam_dist", "kf_cam2_model", "kf_cam2", "kf_trl"):
        if k in g:
            h[k] = np.ascontiguousarray(g[k][perm])
    h["e_kf"] = inv[g["e_kf"]].astype(np.int32)
    return h


def lba_view(g):
    from .views import make_lba_graph_view
    return make_lba_graph_view(**g)


def shard_graph(g, rank, world):
    """Landmark shard of a graph for rank `rank` of `world` (SURVEY.md 8e): landmarks
    l with l % world == rank, with all their edges; keyframes replicated.  Returns
    (sub-graph dict, landmark ids, edge ids)."""
    n_mp = len(g["mp_pos"])
    lm = np.arange(rank, n_mp, world)
    new_id = -np.ones(n_mp, np.int64)
    new_id[lm] = np.arange(len(lm))
    ed = np.nonzero(new_id[g["e_mp"]] >= 0)[0]
    sub = dict(g)
    sub["mp_pos"] = g["mp_pos"][lm]
    sub["e_kf"] = g["e_kf"][ed]
    sub["e_mp"] = new_id[g["e_mp"][ed]].astype(np.int32)
    sub["e_stereo"] = g["e_stereo"][ed]
    sub["e_obs"] = g["e_obs"][ed]
    sub["e_inv_sigma2"] = g["e_inv_sigma2"][ed]
    return sub, lm, ed


def pose_scene(n, seed=0, stereo_frac=0.8, outlier_frac=0.1, rot_deg=1.0, trans=0.05, width=1280, height=720,
               fx=700.0, bf=386.0, wild=False):
    """One frame for Optimizer::PoseOptimization (SURVEY.md 8(f-2)): n matched MapPoints in the frustum
    (depth 2..30 m), observations with the octave noise model, `outlier_frac` gross mismatches (random
    positions), and an initial pose off the truth by `rot_deg` / `trans` (a constant-velocity prediction).
    `wild=True` starts far enough away to force rejected LM trials.  Returns (pose_opt_view, truth dict)."""
    from .views import make_pose_opt_view
    rng = np.random.default_rng(seed)
    cx, cy = width / 2.0, height / 2.0
    q_true = _quat_from_yaw_pitch(0.3 + 0.01 * seed, -0.05)
    t_true = np.array([0.4, -0.1, 2.0]) + 0.1 * rng.normal(size=3)
    depth = rng.uniform(2, 30, n)
    u = rng.uniform(30, width - 30, n)
    v = rng.uniform(30, height - 30, n)
    Xc = np.stack([(u - cx) / fx * depth, (v - cy) / fx * depth, depth], 1)
    qi = q_true * np.array([-1, -1, -1, 1])
    Xw = _qrot_many(np.tile(qi, (n, 1)), Xc - t_true)               # Tcw^-1 * Xc
    octv = rng.integers(0, 8, n)
    sig = 1.2 ** octv
    noise = rng.normal(0, 1, (n, 3)) * sig[:, None]
    ur = u - bf / depth + noise[:, 2]
    st = rng.random(n) < stereo_frac
    obs = np.stack([u + noise[:, 0], v + noise[:, 1], np.where(st, ur, -1.0)], 1)
    out = rng.random(n) < outlier_frac
    obs[out, 0] = rng.uniform(0, width, out.sum())
    obs[out, 1] = rng.uniform(0, height, out.sum())
    obs[out & st, 2] = obs[out & st, 0] - rng.uniform(2, 60, (out & st).sum())
    inv_sigma2 = (1.0 / (scale_factors() ** 2)).astype(np.float32)[octv]
    scale = 20.0 if wild else 1.0
    w = rng.normal(0, np.deg2rad(rot_deg * scale) / np.sqrt(3), 3)
    th = np.linalg.norm(w)
    dq = np.concatenate([np.sin(th / 2) * w / max(th, 1e-12), [np.cos(th / 2)]])
    q0 = _quat_mul(dq, q_true)
    t0 = _quat_rot(dq, t_true) + rng.normal(0, trans * scale / np.sqrt(3), 3)
    pose0 = np.concatenate([q0, t0]).astype(np.float32).astype(np.float64)  # Sophus::SE3f cast to double (:830-831)
    view = make_pose_opt_view(Xw.astype(np.float32), obs.astype(np.float32), inv_sigma2, (fx, fx, cx, cy, bf), pose0)
    return view, dict(pose=np.concatenate([q_true, t_true]), outlier=out, stereo=st)


def frustum_scene(n, seed=0, width=1280, height=720, fx=700.0, bf=386.0):
    """Local map points around one frame for Frame::isInFrustum (SURVEY.md 8(f-3)): a mix that takes every
    exit of the function -- behind the camera, outside the image bounds, outside the scale-invariance
    distance band, seen from too steep an angle, and in view.  Returns (orb_frustum_view, truth dict)."""
    from .views import make_frustum_view
    rng = np.random.default_rng(seed)
    cx, cy = width / 2.0, height / 2.0
    q = _quat_from_yaw_pitch(0.4 + 0.1 * seed, 0.1)                      # Rwc
    twc = np.array([1.0, -0.5, 2.0]) + rng.normal(0, 0.3, 3)
    qi = q * np.array([-1, -1, -1, 1])
    R = np.stack([_quat_rot(qi, e) for e in np.eye(3)], 1)               # Rcw
    tcw = -R @ twc
    depth = rng.uniform(-5, 40, n)                                       # ~11 % behind the camera
    u = rng.uniform(-200, width + 200, n)                                # some outside the image
    v = rng.uniform(-120, height + 120, n)
    Xc = np.stack([(u - cx) / fx * depth, (v - cy) / fx * depth, depth], 1)
    Xw = (Xc - tcw) @ R                                                  # Rcw^T (Xc - tcw)
    # reference keyframe of each point: somewhere else, sets the normal and the distance band
    ref = twc + rng.normal(0, 6.0, (n, 3))
    d_ref = np.linalg.norm(Xw - ref, axis=1)
    normal = (Xw - ref) / d_ref[:, None]
    level = rng.integers(0, 8, n)
    max_dist = d_ref * (1.2 ** level)
    min_dist = max_dist / (1.2 ** 7)
    view = make_frustum_view(Xw, normal, min_dist, max_dist, R, tcw, (fx, fx, cx, cy, bf), (0.0, width, 0.0, height))
    return view, dict(depth=depth, u=u, v=v)


def frustum_match_scene(kps, desc, width, height, seed, n_extra=500, th_noise=1.0):
    """3-D local map behind SearchByProjection(F, vpMapPoints): one MapPoint per keypoint, placed so that it
    projects within ~th_noise px of the keypoint and PredictScale gives the keypoint's octave, plus n_extra
    random points (some outside the frustum).  Returns (orb_frame_view, orb_frustum_view, desc[n,32],
    is_bad, has_obs): Frame::isInFrustum on the frustum view yields the orb_mappoint_view fields."""
    from .views import make_frame_view, make_frustum_view
    rng = np.random.default_rng(seed)
    sf = scale_factors()
    cx, cy = width / 2.0, height / 2.0
    q = _quat_from_yaw_pitch(0.2, -0.05)
    twc = np.array([0.5, 0.2, -1.0])
    qi = q * np.array([-1, -1, -1, 1])
    R = np.stack([_quat_rot(qi, e) for e in np.eye(3)], 1)               # Rcw
    tcw = -R @ twc
    n = len(kps)
    u = np.concatenate([kps["x"] + rng.normal(0, th_noise, n), rng.uniform(-100, width + 100, n_extra)])
    v = np.concatenate([kps["y"] + rng.normal(0, th_noise, n), rng.uniform(-60, height + 60, n_extra)])
    m = n + n_extra
    z = rng.uniform(3, 30, m)
    Xc = np.stack([(u - cx) / FX * z, (v - cy) / FY * z, z], 1)
    Xw = (Xc - tcw) @ R
    octv = np.concatenate([kps["octave"], rng.integers(0, 8, n_extra)])
    dist = np.linalg.norm(Xw - twc, axis=1)
    max_dist = dist * 1.2 ** (octv - 0.5)                                # ceil(log(max/dist)/log 1.2) = octave
    min_dist = max_dist / 1.2 ** 7
    view_dir = (Xw - twc) / dist[:, None]
    tilt = rng.normal(0, 0.02, (m, 3)) + (rng.random(m) < 0.3)[:, None] * rng.normal(0, 0.2, (m, 3))
    normal = view_dir + tilt
    normal /= np.linalg.norm(normal, axis=1)[:, None]
    d = np.concatenate([flip_bits(desc, 6, rng), rng.integers(0, 256, (n_extra, 32), dtype=np.uint8)])
    order = rng.permutation(m)
    fv = make_frustum_view(Xw[order], normal[order], min_dist[order], max_dist[order], R, tcw,
                           (FX, FY, cx, cy, 386.0), (0.0, width, 0.0, height))
    taken = (rng.random(n) < 0.2).astype(np.uint8)
    F = make_frame_view(kps, desc, width, height, sf, kp_taken=taken, fx=FX, fy=FY, bf=0.0)
    is_bad = (rng.random(m) < 0.02).astype(np.uint8)
    has_obs = (rng.random(m) > 0.1).astype(np.uint8)
    return F, fv, np.ascontiguousarray(d[order]), is_bad, has_obs


def synth_vocabulary(k=10, L=4, seed=0, irregular=True, stop_frac=0.02):
    """A DBoW2-shaped ORB vocabulary (SURVEY.md 8(f-4)): a k-ary tree of depth L built top-down, node
    descriptors = parent's with ~40 bits flipped (so a descriptor's descent is decided by real Hamming
    distances, with ties), idf-like word weights, `stop_frac` of the words stopped (weight 0), and --
    `irregular` -- a few nodes with fewer children and a few leaves above the last level, like k-means
    trees that run out of points.  Returns an orb_vocab_view."""
    from .views import make_vocab_view
    rng = np.random.default_rng(seed)
    desc = [rng.integers(0, 256, 32, dtype=np.uint8)]      # node 0: root (its descriptor is never read)
    children = [[]]
    level = [0]
    frontier = [0]
    for lv in range(1, L + 1):
        nxt = []
        for p in frontier:
            if irregular and lv > 1 and rng.random() < 0.03:
                continue                                   # an early leaf
            kk = k if not irregular or rng.random() > 0.1 else int(rng.integers(2, k + 1))
            for _ in range(kk):
                bits = np.unpackbits(desc[p])
                flip = rng.choice(256, 40, replace=False)
                bits[flip] ^= 1
                desc.append(np.packbits(bits))
                children.append([])
                level.append(lv)
                children[p].append(len(desc) - 1)
                nxt.append(len(desc) - 1)
        frontier = nxt
    n = len(desc)
    child_ptr = np.zeros(n + 1, np.int32)
    child_ids = []
    for i in range(n):
        child_ids.extend(children[i])
        child_ptr[i + 1] = len(child_ids)
    is_leaf = np.array([len(c) == 0 for c in children])
    word_id = -np.ones(n, np.int32)
    word_id[is_leaf] = np.arange(is_leaf.sum())            # m_words order = node order (create_words, :905-925)
    weight = np.zeros(n)
    weight[is_leaf] = np.log(rng.uniform(1.5, 400.0, is_leaf.sum()))
    stopped = is_leaf & (rng.random(n) < stop_frac)
    weight[stopped] = 0.0
    return make_vocab_view(L, child_ptr, np.array(child_ids, np.int32), np.stack(desc), weight, word_id)


# ------------------------------------------------------------------ visual-inertial local window (SURVEY.md 8(f-4b))
def _so3_exp(w):
    th = np.linalg.norm(w)
    W = np.array([[0, -w[2], w[1]], [w[2], 0, -w[0]], [-w[1], w[0], 0]])
    if th < 1e-8:
        return np.eye(3) + W
    return np.eye(3) + W * np.sin(th) / th + W @ W * (1 - np.cos(th)) / th ** 2


def _so3_right_jac(w):
    th = np.linalg.norm(w)
    W = np.array([[0, -w[2], w[1]], [w[2], 0, -w[0]], [-w[1], w[0], 0]])
    if th < 1e-8:
        return np.eye(3)
    return np.eye(3) - W * (1 - np.cos(th)) / th ** 2 + W @ W * (th - np.sin(th)) / th ** 3


def imu_preintegrate(acc, gyr, dt, ba, bg, Nga, NgaWalk):
    """IMU::Preintegrated::IntegrateNewMeasurement over a run of samples (reference src/ImuTypes.cc:176-237):
    returns dict(dR, dV, dP, JRg, JVg, JVa, JPg, JPa, C[15,15], dT).  float64 here; the caller casts."""
    dR, dV, dP = np.eye(3), np.zeros(3), np.zeros(3)
    JRg, JVg, JVa, JPg, JPa = (np.zeros((3, 3)) for _ in range(5))
    C = np.zeros((15, 15))
    dT = 0.0
    for a_m, w_m in zip(acc, gyr):
        a, w = a_m - ba, w_m - bg
        Wacc = np.array([[0, -a[2], a[1]], [a[2], 0, -a[0]], [-a[1], a[0], 0]])
        A, B = np.eye(9), np.zeros((9, 6))
        dP = dP + dV * dt + 0.5 * dR @ a * dt * dt
        dV = dV + dR @ a * dt
        A[3:6, 0:3] = -dR * dt @ Wacc
        A[6:9, 0:3] = -0.5 * dR * dt * dt @ Wacc
        A[6:9, 3:6] = np.eye(3) * dt
        B[3:6, 3:6] = dR * dt
        B[6:9, 3:6] = 0.5 * dR * dt * dt
        JPa = JPa + JVa * dt - 0.5 * dR * dt * dt
        JPg = JPg + JVg * dt - 0.5 * dR * dt * dt @ Wacc @ JRg
        JVa = JVa - dR * dt
        JVg = JVg - dR * dt @ Wacc @ JRg
        dRi, rJ = _so3_exp(w * dt), _so3_right_jac(w * dt)
        U, _, Vt = np.linalg.svd(dR @ dRi)
        dR = U @ Vt
        A[0:3, 0:3] = dRi.T
        B[0:3, 0:3] = rJ * dt
        C[0:9, 0:9] = A @ C[0:9, 0:9] @ A.T + B @ Nga @ B.T
        C[9:15, 9:15] += NgaWalk
        JRg = dRi.T @ JRg - rJ * dt
        dT += dt
    return dict(dR=dR, dV=dV, dP=dP, JRg=JRg, JVg=JVg, JVa=JVa, JPg=JPg, JPa=JPa, C=C, dT=dT)


def lia_scene(n_opt=6, n_mp=300, seed=0, n_fixed_visual=2, imu_rate=200, kf_dt=0.5, width=1280, height=720,
              fx=700.0, bf=386.0, perturb=1.0, outlier_frac=0.02):
    """A visual-inertial local window for Optimizer::LocalInertialBA: n_opt optimisable keyframes (newest
    first) with velocity and biases, the fixed keyframe before the window, n_fixed_visual extra fixed
    keyframes without IMU vertices, map points seen from several of them, and the IMU preintegrated between
    consecutive keyframes with the reference's own scheme.  The true trajectory is the discrete integral of
    the simulated IMU samples, so the preintegration constraints hold exactly at the truth.
    Returns (dict for oracle.make_lia_view, truth dict)."""
    rng = np.random.default_rng(seed)
    g = np.array([0.0, 0.0, -9.81])
    dt = 1.0 / imu_rate
    m = int(round(kf_dt * imu_rate))
    nk = n_opt + 1                                   # chronological keyframes 0 (fixed) .. n_opt
    R = np.array([[0.0, 0.0, 1.0], [-1.0, 0.0, 0.0], [0.0, -1.0, 0.0]])  # body = camera axes: z forward (world +x), y down
    p, v = np.zeros(3), np.array([1.2, 0.0, 0.0])
    ba_true, bg_true = rng.normal(0, 0.02, 3), rng.normal(0, 0.002, 3)
    sf = np.sqrt(imu_rate)
    ng, na, ngw, naw = 1.7e-4 * sf, 2.0e-3 * sf, 1.9e-5 / sf, 3.0e-3 / sf
    Nga = np.diag([ng ** 2] * 3 + [na ** 2] * 3)
    NgaWalk = np.diag([ngw ** 2] * 3 + [naw ** 2] * 3)
    states, acc_all, gyr_all = [(R.copy(), p.copy(), v.copy())], [], []
    for s in range((nk - 1) * m):
        t = s * dt
        a_w = np.array([0.3 * np.sin(0.9 * t), 0.5 * np.cos(0.7 * t), 0.2 * np.sin(1.3 * t)])
        w_b = np.array([0.05 * np.sin(1.1 * t), 0.08 * np.cos(0.8 * t), 0.04 * np.sin(0.5 * t)])
        a_b = R.T @ (a_w - g)
        acc_all.append(a_b + ba_true)
        gyr_all.append(w_b + bg_true)
        p = p + v * dt + 0.5 * (R @ a_b + g) * dt * dt
        v = v + (R @ a_b + g) * dt
        U, _, Vt = np.linalg.svd(R @ _so3_exp(w_b * dt))
        R = U @ Vt
        if (s + 1) % m == 0:
            states.append((R.copy(), p.copy(), v.copy()))
    acc_all, gyr_all = np.array(acc_all), np.array(gyr_all)
    # camera rig
    Rcb = _so3_exp(np.array([0.01, -0.02, 0.015]))
    tcb = np.array([0.05, 0.02, -0.01])
    tbc = -Rcb.T @ tcb
    cx, cy = width / 2.0, height / 2.0

    def cam_of(Rwb, twb):
        Rcw = Rcb @ Rwb.T
        return Rcw, Rcb @ (-Rwb.T @ twb) + tcb

    # extra fixed visual keyframes: older poses next to the start
    extra = []
    for j in range(n_fixed_visual):
        Re = states[0][0] @ _so3_exp(rng.normal(0, 0.03, 3))
        extra.append((Re, states[0][1] + np.array([-0.6 * (j + 1), 0.2 * (-1) ** j, 0.05]), np.zeros(3)))
    # view order: newest optimisable first ... oldest optimisable, the fixed one before the window, extras
    order = list(range(nk - 1, 0, -1)) + [0]
    all_states = [states[c] for c in order] + extra
    K = len(all_states)
    fixed = np.array([0] * n_opt + [1] * (1 + n_fixed_visual), np.uint8)
    has_imu = np.array([1] * (n_opt + 1) + [0] * n_fixed_visual, np.uint8)
    Rwb_t = np.stack([s[0] for s in all_states]); twb_t = np.stack([s[1] for s in all_states])
    vel_t = np.stack([s[2] for s in all_states])
    # map points ahead of the trajectory, observed where they project inside the image
    pts = np.stack([rng.uniform(3, 30, n_mp), rng.uniform(-7, 7, n_mp), rng.uniform(-3, 3, n_mp)], 1) + states[0][1]
    e_kf, e_mp, e_obs, e_st, e_is2 = [], [], [], [], []
    inv_sigma2 = (1.0 / (scale_factors() ** 2)).astype(np.float32)
    for l in range(n_mp):
        for k in range(K):
            Rcw, tcw = cam_of(Rwb_t[k], twb_t[k])
            Xc = Rcw @ pts[l] + tcw
            if Xc[2] < 0.5:
                continue
            u, w_ = fx * Xc[0] / Xc[2] + cx, fx * Xc[1] / Xc[2] + cy
            if not (20 < u < width - 20 and 20 < w_ < height - 20) or rng.random() < 0.25:
                continue
            o = int(rng.integers(0, 8))
            sig = 1.2 ** o
            st = rng.random() < 0.7
            n3 = rng.normal(0, 1, 3) * sig
            if rng.random() < outlier_frac:
                n3[0] += 40.0
            e_kf.append(k); e_mp.append(l); e_st.append(st); e_is2.append(inv_sigma2[o])
            e_obs.append([np.float32(u + n3[0]), np.float32(w_ + n3[1]), np.float32(u - bf / Xc[2] + n3[2]) if st else -1.0])
    # preintegration between consecutive keyframes (edge i: kf2 = view i, kf1 = view i + 1)
    lin_off = 1e-3
    pre = []
    for i in range(n_opt):
        c2 = order[i]
        seg = slice((c2 - 1) * m, c2 * m)
        pre.append(imu_preintegrate(acc_all[seg], gyr_all[seg], dt, ba_true + lin_off, bg_true - lin_off, Nga, NgaWalk))
    # initial estimates: truth + perturbation on the free vertices
    Rwb0, twb0, vel0 = Rwb_t.copy(), twb_t.copy(), vel_t.copy()
    bg0 = np.tile(bg_true, (K, 1)); ba0 = np.tile(ba_true, (K, 1))
    for k in range(n_opt):
        Rwb0[k] = Rwb_t[k] @ _so3_exp(rng.normal(0, np.deg2rad(0.3) * perturb, 3))
        twb0[k] = twb_t[k] + rng.normal(0, 0.01 * perturb, 3)
        vel0[k] = vel_t[k] + rng.normal(0, 0.02 * perturb, 3)
        bg0[k] = bg_true + rng.normal(0, 2e-4 * perturb, 3)
        ba0[k] = ba_true + rng.normal(0, 5e-3 * perturb, 3)
    # Sophus::SE3f / Vector3f storage of the reference: float, cast to double by the optimiser
    f32 = lambda a: np.asarray(a, np.float32).astype(np.float64)
    Rwb0, twb0, vel0, bg0, ba0 = f32(Rwb0), f32(twb0), f32(vel0), f32(bg0), f32(ba0)
    Rcw0 = np.stack([cam_of(Rwb0[k], twb0[k])[0] for k in range(K)])
    tcw0 = np.stack([cam_of(Rwb0[k], twb0[k])[1] for k in range(K)])
    pts0 = f32(pts + rng.normal(0, 0.03 * perturb, pts.shape))
    d = dict(kf_Rwb=Rwb0.reshape(K, 9), kf_twb=twb0, kf_Rcw=f32(Rcw0).reshape(K, 9), kf_tcw=f32(tcw0), kf_fixed=fixed,
             kf_has_imu=has_imu, kf_vel=vel0, kf_bg=bg0, kf_ba=ba0, Rcb=Rcb, tcb=tcb, tbc=tbc,
             cam=(fx, fx, cx, cy, bf), mp_pos=pts0, e_kf=e_kf, e_mp=e_mp, e_stereo=e_st,
             e_obs=np.array(e_obs, np.float64).reshape(-1, 3), e_inv_sigma2=e_is2,
             i_kf1=np.arange(1, n_opt + 1), i_kf2=np.arange(0, n_opt),
             i_dR=np.stack([q["dR"] for q in pre]).reshape(n_opt, 9), i_dV=np.stack([q["dV"] for q in pre]),
             i_dP=np.stack([q["dP"] for q in pre]),
             i_JRg=np.stack([q["JRg"] for q in pre]).reshape(n_opt, 9), i_JVg=np.stack([q["JVg"] for q in pre]).reshape(n_opt, 9),
             i_JVa=np.stack([q["JVa"] for q in pre]).reshape(n_opt, 9), i_JPg=np.stack([q["JPg"] for q in pre]).reshape(n_opt, 9),
             i_JPa=np.stack([q["JPa"] for q in pre]).reshape(n_opt, 9),
             i_bias=np.tile(np.concatenate([ba_true + lin_off, bg_true - lin_off]), (n_opt, 1)),
             i_dT=np.array([q["dT"] for q in pre]), i_C=np.stack([q["C"] for q in pre]).reshape(n_opt, 225),
             i_last=np.array([0] * (n_opt - 1) + [1], np.uint8), lambda_init=1.0, iterations=10)
    truth = dict(Rwb=Rwb_t, twb=twb_t, vel=vel_t, bg=bg_true, ba=ba_true, mp_pos=pts, cam_of=cam_of)
    return d, truth
