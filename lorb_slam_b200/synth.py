"""Seeded synthetic inputs of the shapes BASELINE.json names (SURVEY §8(d)).

Pure numpy; no oracle, no CUDA.  Used by bench.py and the tests to feed the
C-ABI with Frame/MapPoint-shaped SoA arrays (the layout lorb_cuda.h documents).
"""
import numpy as np

GRID_COLS, GRID_ROWS = 64, 48


def scale_factors(n_levels=8, scale=1.2):
    """mvScaleFactor as reference src/ORBextractor.cpp:428-436 builds it: the
    factor is a float parameter held in a double member, the vector is float."""
    sf = np.zeros(n_levels, np.float32)
    sf[0] = 1.0
    f = float(np.float32(scale))
    for i in range(1, n_levels):
        sf[i] = np.float32(float(sf[i - 1]) * f)
    return sf


# ----------------------------------------------------------------- descriptors

def descriptors_uniform(n, rng):
    return rng.integers(0, 256, size=(n, 32), dtype=np.uint8)


def descriptors_tie_stress(n, rng, nbytes=2, nvals=4):
    """Low-entropy descriptors: only the first `nbytes` bytes non-zero, values in
    [0, nvals) -> many equal distances, exercises the lowest-index tie-breaks."""
    d = np.zeros((n, 32), np.uint8)
    d[:, :nbytes] = rng.integers(0, nvals, size=(n, nbytes), dtype=np.uint8)
    return d


def descriptors_noisy_copy(src, rng, p_flip=0.08):
    """Each bit of `src` flipped with probability p_flip (a re-observed feature)."""
    bits = np.unpackbits(src, axis=1)
    flip = rng.random(bits.shape) < p_flip
    return np.packbits(bits ^ flip.astype(np.uint8), axis=1)


def kf_bank(n_kf, n_desc, seed=0, shared_frac=0.5, p_flip=0.08):
    """Keyframe descriptor bank for the pair sweep: consecutive keyframes share
    `shared_frac` of their features (noisy copies), the rest is uniform."""
    rng = np.random.default_rng(seed)
    bank = rng.integers(0, 256, size=(n_kf, n_desc, 32), dtype=np.uint8)
    ns = int(n_desc * shared_frac)
    if ns > 0 and n_kf <= 512:  # only worth the time for small banks
        for k in range(1, n_kf):
            idx = rng.permutation(n_desc)[:ns]
            bank[k, idx] = descriptors_noisy_copy(bank[k - 1, idx], rng, p_flip)
    return bank


def all_pairs(n_kf):
    a, b = np.triu_indices(n_kf, k=1)
    return a.astype(np.int32), b.astype(np.int32)


# ------------------------------------------------------------ frames / points

def make_frame(n_kp=2000, seed=0, width=640, height=480, stereo=False, n_levels=8,
               claimed_frac=0.0, claimed_protected_frac=0.5):
    """Current-frame SoA (lorb_frame_view).  Octaves drawn proportional to
    1.2^-l as mnFeaturesPerLevel does (reference src/ORBextractor.cpp:448-461)."""
    rng = np.random.default_rng(seed)
    w = (1.0 / 1.2) ** np.arange(n_levels)
    octave = rng.choice(n_levels, size=n_kp, p=w / w.sum()).astype(np.int32)
    fr = dict(
        n_kp=n_kp,
        kp_x=(rng.random(n_kp) * width).astype(np.float32),
        kp_y=(rng.random(n_kp) * height).astype(np.float32),
        kp_octave=octave,
        kp_angle=(rng.random(n_kp) * 360.0).astype(np.float32),
        kp_uright=np.full(n_kp, -1.0, np.float32),
        desc=descriptors_uniform(n_kp, rng),
        kp_claim_obs=np.full(n_kp, -1, np.int32),
        min_x=0.0, max_x=float(width), min_y=0.0, max_y=float(height),
        n_levels=n_levels, scale_factors=scale_factors(n_levels),
    )
    if stereo:
        has = rng.random(n_kp) < 0.7
        disp = (rng.random(n_kp) * 40.0 + 1.0).astype(np.float32)
        fr["kp_uright"] = np.where(has, fr["kp_x"] - disp, -1.0).astype(np.float32)
    if claimed_frac > 0:
        cl = rng.random(n_kp) < claimed_frac
        prot = rng.random(n_kp) < claimed_protected_frac
        fr["kp_claim_obs"] = np.where(cl, np.where(prot, 3, 0), -1).astype(np.int32)
    return fr


def make_proj_points(fr, n_pts=5000, seed=0, true_frac=0.6, nobs=1, sigma_px=2.0, p_flip=0.08,
                     inactive_frac=0.0):
    """Map points already projected into `fr` (what Frame::IsInFrustum leaves in
    MapPoint::mTrack*, reference src/frame.cpp:484-491)."""
    rng = np.random.default_rng(seed + 7919)
    n_kp = fr["n_kp"]
    n_true = int(n_pts * true_frac)
    src = rng.integers(0, n_kp, size=n_true)
    px = np.empty(n_pts, np.float32)
    py = np.empty(n_pts, np.float32)
    lvl = np.empty(n_pts, np.int32)
    desc = descriptors_uniform(n_pts, rng)
    px[:n_true] = fr["kp_x"][src] + rng.normal(0, sigma_px, n_true).astype(np.float32)
    py[:n_true] = fr["kp_y"][src] + rng.normal(0, sigma_px, n_true).astype(np.float32)
    lvl[:n_true] = np.minimum(fr["kp_octave"][src] + rng.integers(0, 2, n_true), fr["n_levels"] - 1)
    desc[:n_true] = descriptors_noisy_copy(fr["desc"][src], rng, p_flip)
    px[n_true:] = (rng.random(n_pts - n_true) * fr["max_x"]).astype(np.float32)
    py[n_true:] = (rng.random(n_pts - n_true) * fr["max_y"]).astype(np.float32)
    lvl[n_true:] = rng.integers(0, fr["n_levels"], n_pts - n_true)
    perm = rng.permutation(n_pts)  # processing order = array index
    px, py, lvl, desc = px[perm], py[perm], lvl[perm], desc[perm]
    disp = (rng.random(n_pts) * 40.0 + 1.0).astype(np.float32)
    if np.isscalar(nobs):
        mp_nobs = np.full(n_pts, nobs, np.int32)
    else:
        mp_nobs = rng.choice(np.asarray(nobs, np.int32), size=n_pts).astype(np.int32)
    active = (rng.random(n_pts) >= inactive_frac).astype(np.uint8)
    return dict(
        n_pts=n_pts, proj_x=np.ascontiguousarray(px), proj_y=np.ascontiguousarray(py),
        proj_xr=np.ascontiguousarray(px - disp), level=np.ascontiguousarray(lvl),
        view_cos=(0.5 + 0.5 * rng.random(n_pts)).astype(np.float32), active=active,
        mp_desc=np.ascontiguousarray(desc), mp_nobs=mp_nobs,
    )


def rodrigues(rvec):
    """Angle-axis -> rotation matrices, vectorised ([...,3] -> [...,3,3])."""
    rvec = np.asarray(rvec, np.float64)
    th = np.linalg.norm(rvec, axis=-1)[..., None, None]
    k = rvec / np.maximum(th[..., 0], 1e-300)
    K = np.zeros(rvec.shape[:-1] + (3, 3))
    K[..., 0, 1], K[..., 0, 2] = -k[..., 2], k[..., 1]
    K[..., 1, 0], K[..., 1, 2] = k[..., 2], -k[..., 0]
    K[..., 2, 0], K[..., 2, 1] = -k[..., 1], k[..., 0]
    I = np.broadcast_to(np.eye(3), K.shape)
    return I + np.sin(th) * K + (1 - np.cos(th)) * (K @ K)


def make_frame_pair(n_kp=2000, seed=0, width=640, height=480, motion="forward", stereo=True,
                    nobs=(0, 1, 2), valid_frac=0.9, sigma_px=1.5, p_flip=0.06):
    """Inputs of Matcher::SearchByProjection(Cur, Last, th) (reference
    src/matcher.cpp:64-218): Last's map points re-observed in Cur after a small
    camera motion, plus clutter keypoints in Cur."""
    rng = np.random.default_rng(seed + 104729)
    fx = fy = np.float32(458.0)
    cx, cy = np.float32(width / 2), np.float32(height / 2)
    mbf = np.float32(47.9)
    mb = np.float32(mbf / fx)
    n_levels = 8
    sf = scale_factors(n_levels)
    # Last frame at identity; points in front of it
    u = rng.random(n_kp) * width
    v = rng.random(n_kp) * height
    z = 2.0 + rng.random(n_kp) * 18.0
    xw = np.stack([(u - cx) / fx * z, (v - cy) / fy * z, z], 1).astype(np.float32)
    w = (1.0 / 1.2) ** np.arange(n_levels)
    last_oct = rng.choice(n_levels, size=n_kp, p=w / w.sum()).astype(np.int32)
    last_angle = (rng.random(n_kp) * 360.0).astype(np.float32)
    last_desc = descriptors_uniform(n_kp, rng)
    tz = {"forward": 0.4, "backward": -0.4, "still": 0.02}[motion]
    rv = rng.normal(0, 0.01, 3)
    Rcl = rodrigues(rv)
    tcl = np.array([0.03, -0.02, -tz])  # x_cur = Rcl x_last + tcl (camera moved +tz)
    tcw_last = np.eye(4, dtype=np.float32)
    tcw_cur = np.eye(4, dtype=np.float32)
    tcw_cur[:3, :3] = Rcl.astype(np.float32)
    tcw_cur[:3, 3] = tcl.astype(np.float32)
    xc = (Rcl @ xw.astype(np.float64).T).T + tcl
    uc = fx * xc[:, 0] / xc[:, 2] + cx
    vc = fy * xc[:, 1] / xc[:, 2] + cy
    cur = make_frame(n_kp, seed + 1, width, height, stereo=False, n_levels=n_levels)
    n_re = int(0.7 * n_kp)  # re-observed features occupy the first slots of Cur (shuffled below)
    src = rng.permutation(n_kp)[:n_re]
    ok = (uc[src] > 0) & (uc[src] < width) & (vc[src] > 0) & (vc[src] < height) & (xc[src, 2] > 0.1)
    src = src[ok]
    slot = rng.permutation(n_kp)[:len(src)]
    cur["kp_x"][slot] = (uc[src] + rng.normal(0, sigma_px, len(src))).astype(np.float32)
    cur["kp_y"][slot] = (vc[src] + rng.normal(0, sigma_px, len(src))).astype(np.float32)
    cur["kp_x"] = np.clip(cur["kp_x"], 0, width - 1e-3).astype(np.float32)
    cur["kp_y"] = np.clip(cur["kp_y"], 0, height - 1e-3).astype(np.float32)
    d_oct = {"forward": rng.integers(0, 2, len(src)), "backward": -rng.integers(0, 2, len(src)),
             "still": rng.integers(-1, 2, len(src))}[motion]
    cur["kp_octave"][slot] = np.clip(last_oct[src] + d_oct, 0, n_levels - 1)
    # most re-observations keep their orientation (+ a common rotation), some do not
    rot = np.where(rng.random(len(src)) < 0.85, 12.0 + rng.normal(0, 2.0, len(src)),
                   rng.random(len(src)) * 360.0)
    cur["kp_angle"][slot] = np.mod(last_angle[src] - rot, 360.0).astype(np.float32)
    cur["desc"][slot] = descriptors_noisy_copy(last_desc[src], rng, p_flip)
    if stereo:
        has = rng.random(n_kp) < 0.7
        ur = cur["kp_x"] - mbf / np.maximum(2.0 + rng.random(n_kp) * 18.0, 1e-3)
        ur[slot] = (cur["kp_x"][slot] - mbf / xc[src, 2] + rng.normal(0, 1.0, len(src)))
        cur["kp_uright"] = np.where(has, ur, -1.0).astype(np.float32)
    last = dict(
        n_last=n_kp, valid=(rng.random(n_kp) < valid_frac).astype(np.uint8),
        xw=np.ascontiguousarray(xw), octave=last_oct, angle=last_angle,
        mp_desc=np.ascontiguousarray(last_desc),
        mp_nobs=rng.choice(np.asarray(nobs, np.int32), size=n_kp).astype(np.int32),
        tcw_cur=np.ascontiguousarray(tcw_cur.reshape(16)),
        tcw_last=np.ascontiguousarray(tcw_last.reshape(16)),
        K=dict(fx=float(fx), fy=float(fy), cx=float(cx), cy=float(cy), mbf=float(mbf),
               mb=float(mb)),
    )
    return cur, last


def make_frustum_points(n=5000, seed=0, width=640, height=480):
    """Inputs of Frame::IsInFrustum for n local map points (reference
    src/frame.cpp:425-494): a camera pose, 3-D points in and around its frustum,
    mean viewing directions and scale-invariance distance ranges."""
    rng = np.random.default_rng(seed + 611953)
    fx = fy = np.float32(458.0)
    cx, cy = np.float32(width / 2), np.float32(height / 2)
    mbf = np.float32(47.9)
    rv = rng.normal(0, 0.2, 3)
    R = rodrigues(rv)
    t = rng.normal(0, 1.0, 3)
    tcw = np.eye(4, dtype=np.float32)
    tcw[:3, :3] = R.astype(np.float32)
    tcw[:3, 3] = t.astype(np.float32)
    ow = (-R.T @ t).astype(np.float32)
    # points: 75 % inside a widened frustum, the rest anywhere (behind, outside, far)
    u = rng.uniform(-0.3 * width, 1.3 * width, n)
    v = rng.uniform(-0.3 * height, 1.3 * height, n)
    z = np.where(rng.random(n) < 0.9, rng.uniform(0.5, 30.0, n), rng.uniform(-5.0, 0.5, n))
    xc = np.stack([(u - cx) / fx * z, (v - cy) / fy * z, z], 1)
    xw = ((xc - t) @ R).astype(np.float32)
    d = np.linalg.norm(xw - ow, axis=1)
    ref_d = d * rng.uniform(0.4, 2.5, n)               # distance at which the point was created
    lvl = rng.integers(0, 8, n)
    sf = scale_factors(8)
    max_dist = (ref_d * sf[lvl]).astype(np.float32)     # UpdateNormalAndDepth, map_point.cpp:263-264
    min_dist = (max_dist / sf[7]).astype(np.float32)
    to_pt = (xw - ow) / np.maximum(d, 1e-6)[:, None]
    nrm = to_pt + rng.normal(0, 0.5, (n, 3))
    nrm = (nrm / np.linalg.norm(nrm, axis=1)[:, None]).astype(np.float32)
    return dict(n=n, tcw=np.ascontiguousarray(tcw.reshape(16)), ow=ow,
                K=dict(fx=float(fx), fy=float(fy), cx=float(cx), cy=float(cy), mbf=float(mbf)),
                min_x=0.0, max_x=float(width), min_y=0.0, max_y=float(height),
                xw=np.ascontiguousarray(xw), normal=np.ascontiguousarray(nrm), min_dist=min_dist,
                max_dist=max_dist, cos_limit=0.5, n_levels=8,
                # = logf(1.2f) of reference src/frame.cpp:35 (numpy's float32 log is 1 ulp off here)
                log_sf=float(np.float32(np.log(np.float64(np.float32(1.2))))))


# --------------------------------------------------------------------- BA

K_DEFAULT = np.array([458.0, 458.0, 320.0, 240.0], np.float32)


def _project(rv, tv, X, K):
    R = rodrigues(rv)
    q = np.einsum("...ij,...j->...i", R, X) + tv
    u = q[..., 0] / q[..., 2] * K[0] + K[2]
    v = q[..., 1] / q[..., 2] * K[1] + K[3]
    return u, v, q[..., 2]


def make_ba_problem(seed=0, C=10, P=5000, obs_per_point=(6,), traj_len=5.0, fixed_frac=0.0,
                    width=640, height=480, pose_noise=(0.01, 0.05), point_noise=0.05,
                    pixel_noise=1.0):
    """Local-BA window (SURVEY §8(d) cfg 3 / cfg 5).  Cameras on a gentle arc of
    length `traj_len` looking down +z at a cloud 4-20 m ahead; every point is
    observed by k in `obs_per_point` cameras drawn among those that see it.
    Initial parameters = truth + noise, rounded through fp32 (the reference
    stores poses and points as float, src/bundle_adjust.cpp:250-264).
    Observations sorted by point.  `fixed_frac` of each point's observers are
    turned into out-of-window MPCost observations with a fixed float pose."""
    rng = np.random.default_rng(seed)
    K = K_DEFAULT
    s = np.linspace(0.0, 1.0, C) if C > 1 else np.zeros(1)
    cam_c = np.stack([s * traj_len, 0.15 * np.sin(2 * np.pi * s), 0.1 * s], 1)  # centres
    cam_rv = np.stack([0.02 * np.sin(3 * s), 0.08 * (s - 0.5), 0.01 * s], 1)     # small rotations
    R = rodrigues(cam_rv)
    cam_t = -np.einsum("cij,cj->ci", R, cam_c)  # x_c = R x_w + t
    half = max(5.0, traj_len / 2 + 5.0)
    pts = np.empty((P, 3))
    obs_cam, obs_pt = [], []
    ks = np.minimum(rng.choice(np.asarray(obs_per_point), size=P), C)
    todo = np.arange(P)
    chunk = 20000
    while len(todo):
        n = len(todo)
        cand = np.stack([rng.uniform(traj_len / 2 - half, traj_len / 2 + half, n),
                         rng.uniform(-3.0, 3.0, n), rng.uniform(4.0, 20.0, n)], 1)
        done = np.zeros(n, bool)
        kmax = min(int(np.max(obs_per_point)), C)
        for a in range(0, n, chunk):
            X = cand[a:a + chunk]
            u, v, z = _project(cam_rv[None], cam_t[None], X[:, None, :], K)
            vis = (z > 0.5) & (u > 1) & (u < width - 1) & (v > 1) & (v < height - 1)
            kk = ks[todo[a:a + chunk]]
            good = vis.sum(1) >= kk
            # k random visible cameras per point: smallest random scores among the visible
            score = np.where(vis, rng.random(vis.shape), 2.0)
            pick = np.argsort(score, axis=1)[:, :kmax]
            use = (np.arange(kmax)[None, :] < kk[:, None]) & good[:, None]
            rows = np.nonzero(good)[0]
            pts[todo[a + rows]] = X[rows]
            sel_cam = np.sort(np.where(use, pick, C + 1), axis=1)
            m = sel_cam <= C
            obs_cam.append(sel_cam[m])
            obs_pt.append(np.broadcast_to(todo[a:a + chunk][:, None], sel_cam.shape)[m])
            done[a + rows] = True
        todo = todo[~done]
    obs_cam = np.concatenate(obs_cam).astype(np.int32)
    obs_pt = np.concatenate(obs_pt).astype(np.int32)
    order = np.argsort(obs_pt, kind="stable")
    obs_cam, obs_pt = obs_cam[order], obs_pt[order]
    u, v, _ = _project(cam_rv[obs_cam], cam_t[obs_cam], pts[obs_pt], K)
    uv = np.stack([u, v], 1) + rng.normal(0, pixel_noise, (len(u), 2))
    uv = uv.astype(np.float32)
    cams0 = np.concatenate([cam_rv + rng.normal(0, pose_noise[0], (C, 3)),
                            cam_t + rng.normal(0, pose_noise[1], (C, 3))], 1)
    cams0 = cams0.astype(np.float32).astype(np.float64)
    pts0 = (pts + rng.normal(0, point_noise, (P, 3))).astype(np.float32).astype(np.float64)
    pb = dict(C=C, P=P, K=K.copy(), cams=cams0, pts=pts0,
              cams_true=np.concatenate([cam_rv, cam_t], 1), pts_true=pts.copy())
    if fixed_frac > 0:
        fx = rng.random(len(obs_cam)) < fixed_frac
        truth = np.concatenate([cam_rv, cam_t], 1).astype(np.float32)
        pb["fix_pt"] = obs_pt[fx].copy()
        pb["fix_uv"] = uv[fx].copy()
        pb["fix_rt"] = np.ascontiguousarray(truth[obs_cam[fx]])
        obs_cam, obs_pt, uv = obs_cam[~fx], obs_pt[~fx], uv[~fx]
    else:
        pb["fix_pt"] = np.zeros(0, np.int32)
        pb["fix_uv"] = np.zeros((0, 2), np.float32)
        pb["fix_rt"] = np.zeros((0, 6), np.float32)
    pb["obs_cam"] = np.ascontiguousarray(obs_cam)
    pb["obs_pt"] = np.ascontiguousarray(obs_pt)
    pb["obs_uv"] = np.ascontiguousarray(uv)
    pb["O"] = len(obs_cam)
    pb["F"] = len(pb["fix_pt"])
    return pb


def make_pose_only(seed=0, n=500, pixel_noise=1.0, pose_noise=(0.02, 0.1)):
    """Inputs of BA::ProjectPoseOptimization (reference src/bundle_adjust.cpp:158-202).
    fx = fy so the reference's fx-for-v quirk (:51) is consistent with the data."""
    rng = np.random.default_rng(seed + 15485863)
    K = K_DEFAULT
    rv = rng.normal(0, 0.1, 3)
    tv = rng.normal(0, 0.3, 3)
    Xc = np.stack([rng.uniform(-4, 4, n), rng.uniform(-3, 3, n), rng.uniform(3, 20, n)], 1)
    R = rodrigues(rv)
    xw = ((Xc - tv) @ R).astype(np.float32)  # R^T (Xc - t)
    u, v, _ = _project(rv, tv, xw.astype(np.float64), np.array([K[0], K[0], K[2], K[3]]))
    uv = (np.stack([u, v], 1) + rng.normal(0, pixel_noise, (n, 2))).astype(np.float32)
    rt0 = np.concatenate([rv + rng.normal(0, pose_noise[0], 3), tv + rng.normal(0, pose_noise[1], 3)])
    rt0 = rt0.astype(np.float32).astype(np.float64)
    return dict(n=n, xw=xw, uv=uv, K=K.copy(), rt=rt0, rt_true=np.concatenate([rv, tv]))


def make_pnp_problems(seed=0, n=300, n_problems=1, outlier_frac=0.3, pixel_noise=1.0, K=None, n_levels=8,
                      scale=1.2, collinear=False, noise="gauss"):
    """Inputs of lorb_pnp_ransac_batched: n_problems independent 2D-3D match sets of n correspondences each
    (n an int or a sequence of n_problems ints), each with its own planted pose (rt_true [B, 6], angle-axis +
    translation, x_c = R X + t).  Points lie 3-20 m in front of the camera; keypoints get Gaussian noise of
    pixel_noise * scale^octave (octaves drawn as an ORB pyramid fills them), so info = 1 / sigma^2 of the octave
    are the true inverse variances (noise="uniform": uniform in +-pixel_noise * scale^octave per axis instead);
    `outlier_frac` of the keypoints are replaced by uniform pixels (mismatches).  collinear=True puts every world
    point of a problem on one line."""
    rng = np.random.default_rng(seed + 7919)
    K = K_DEFAULT if K is None else np.asarray(K, np.float32)
    sizes = [int(n)] * n_problems if np.isscalar(n) else [int(v) for v in n]
    wl = (1.0 / scale) ** np.arange(n_levels)
    xw, uv, info, outl, rts = [], [], [], [], []
    for m in sizes:
        rv = rng.normal(0, 0.5, 3)
        tv = rng.normal(0, 1.0, 3)
        if collinear:
            a, d = rng.normal(0, 1, 3) + [0, 0, 10], rng.normal(0, 1, 3)
            Xc = a + np.outer(rng.uniform(-3, 3, m), d / np.linalg.norm(d))
        else:
            Xc = np.stack([rng.uniform(-4, 4, m), rng.uniform(-3, 3, m), rng.uniform(3, 20, m)], 1)
        R = rodrigues(rv)
        X = (Xc - tv) @ R  # R^T (Xc - t)
        oc = rng.choice(n_levels, size=m, p=wl / wl.sum())
        sig = pixel_noise * scale ** oc
        nz = rng.normal(0, 1, (m, 2)) if noise == "gauss" else rng.uniform(-1, 1, (m, 2))
        u = K[0] * Xc[:, 0] / Xc[:, 2] + K[2] + nz[:, 0] * sig
        v = K[1] * Xc[:, 1] / Xc[:, 2] + K[3] + nz[:, 1] * sig
        bad = rng.random(m) < outlier_frac
        u[bad] = rng.uniform(0, 2 * K[2], bad.sum())
        v[bad] = rng.uniform(0, 2 * K[3], bad.sum())
        xw.append(X)
        uv.append(np.stack([u, v], 1))
        info.append(1.0 / (scale ** oc) ** 2)
        outl.append(bad)
        rts.append(np.concatenate([rv, tv]))
    cat = lambda a, d: np.ascontiguousarray(np.concatenate(a).reshape(-1, d)) if a else np.zeros((0, d))
    return dict(corr_off=np.concatenate([[0], np.cumsum(sizes)]).astype(np.int32), K=K.copy(),
                xw=cat(xw, 3).astype(np.float32), uv=cat(uv, 2).astype(np.float32),
                info=cat(info, 1).reshape(-1).astype(np.float32), outlier=cat(outl, 1).reshape(-1).astype(bool),
                rt_true=np.array(rts).reshape(-1, 6))


def batch_windows(pbs):
    """Concatenate independent windows into the offset-array form of
    lorb_ba_local_batched (observation indices stay window-local)."""
    cam_off = np.cumsum([0] + [p["C"] for p in pbs]).astype(np.int32)
    pt_off = np.cumsum([0] + [p["P"] for p in pbs]).astype(np.int32)
    obs_off = np.cumsum([0] + [p["O"] for p in pbs]).astype(np.int32)
    bt = dict(
        n_windows=len(pbs), cam_off=cam_off, pt_off=pt_off, obs_off=obs_off,
        cams=np.concatenate([p["cams"] for p in pbs]), pts=np.concatenate([p["pts"] for p in pbs]),
        obs_cam=np.concatenate([p["obs_cam"] for p in pbs]),
        obs_pt=np.concatenate([p["obs_pt"] for p in pbs]),
        obs_uv=np.concatenate([p["obs_uv"] for p in pbs]), K=pbs[0]["K"].copy())
    if any(p.get("F", 0) for p in pbs):  # fixed observations (window-local point indices), same offset form
        bt["fix_off"] = np.cumsum([0] + [p.get("F", 0) for p in pbs]).astype(np.int32)
        bt["fix_pt"] = np.concatenate([p["fix_pt"] for p in pbs]).astype(np.int32)
        bt["fix_uv"] = np.concatenate([p["fix_uv"] for p in pbs]).astype(np.float32).reshape(-1, 2)
        bt["fix_rt"] = np.concatenate([p["fix_rt"] for p in pbs]).astype(np.float32).reshape(-1, 6)
    return bt


# ------------------------------------------------------------- stereo matches

def _blur(img, k):
    ker = np.ones(k) / k
    img = np.apply_along_axis(lambda r: np.convolve(r, ker, mode="same"), 1, img)
    return np.apply_along_axis(lambda c: np.convolve(c, ker, mode="same"), 0, img)


def _resample(img, w, h):
    """Bilinear resize (the pyramid is an INPUT of the path; any resampler will do)."""
    H, W = img.shape
    xs = (np.arange(w) + 0.5) * W / w - 0.5
    ys = (np.arange(h) + 0.5) * H / h - 0.5
    x0 = np.clip(np.floor(xs).astype(int), 0, W - 2)
    y0 = np.clip(np.floor(ys).astype(int), 0, H - 2)
    fx = np.clip(xs - x0, 0, 1)[None, :]
    fy = np.clip(ys - y0, 0, 1)[:, None]
    a = img[y0][:, x0]
    b = img[y0][:, x0 + 1]
    c = img[y0 + 1][:, x0]
    d = img[y0 + 1][:, x0 + 1]
    return (a * (1 - fx) + b * fx) * (1 - fy) + (c * (1 - fx) + d * fx) * fy


def make_stereo_pair(n_kp=1000, seed=0, width=640, height=480, n_levels=8, matched_frac=0.75,
                     p_flip=0.05, border=19):
    """Inputs of Frame::ComputeStereoMatches (reference src/frame.cpp:125-333): rectified left /
    right image pyramids (the right image is the left one shifted by a per-band disparity), left and
    right keypoints at least `border` px from the border of their pyramid level (what
    ORBextractor's EDGE_THRESHOLD guarantees, reference src/ORBextractor.cpp:808-811) and their
    descriptors."""
    rng = np.random.default_rng(seed + 424243)
    sf = scale_factors(n_levels)
    inv_sf = (np.float32(1.0) / sf).astype(np.float32)  # mvInvScaleFactor, src/ORBextractor.cpp:434
    tex = rng.random((height, width)) * 255.0
    img = 0.5 * _blur(tex, 3) + 0.5 * _blur(tex, 9)
    for _ in range(300):
        x, y = int(rng.integers(0, width - 10)), int(rng.integers(0, height - 10))
        w, h = int(rng.integers(4, 50)), int(rng.integers(4, 50))
        img[y:y + h, x:x + w] = 0.6 * img[y:y + h, x:x + w] + 0.4 * rng.integers(0, 256)
    left0 = np.clip(img, 0, 255)
    n_bands = 8
    band_d = rng.uniform(3.0, 60.0, n_bands)
    row_d = band_d[np.minimum(np.arange(height) * n_bands // height, n_bands - 1)]
    xs = np.arange(width)[None, :] + row_d[:, None]  # right(x, y) = left(x + d(y), y)
    x0 = np.clip(np.floor(xs).astype(int), 0, width - 2)
    fx = np.clip(xs - x0, 0, 1)
    rows = np.arange(height)[:, None]
    right0 = left0[rows, x0] * (1 - fx) + left0[rows, x0 + 1] * fx
    right0 = np.clip(right0 + rng.normal(0, 1.0, right0.shape), 0, 255)
    dims = [(int(np.rint(np.float32(width) * inv_sf[l])), int(np.rint(np.float32(height) * inv_sf[l])))
            for l in range(n_levels)]
    pyr_l = [np.ascontiguousarray(np.rint(_resample(left0, w, h)).astype(np.uint8)) for (w, h) in dims]
    pyr_r = [np.ascontiguousarray(np.rint(_resample(right0, w, h)).astype(np.uint8)) for (w, h) in dims]
    wgt = (1.0 / 1.2) ** np.arange(n_levels)
    loct = rng.choice(n_levels, size=n_kp, p=wgt / wgt.sum()).astype(np.int32)
    lw = np.array([dims[o][0] for o in loct])
    lh = np.array([dims[o][1] for o in loct])
    lx = ((border + rng.random(n_kp) * (lw - 2 * border)) * sf[loct]).astype(np.float32)
    ly = ((border + rng.random(n_kp) * (lh - 2 * border)) * sf[loct]).astype(np.float32)
    ldesc = descriptors_uniform(n_kp, rng)
    # right keypoints: re-detections of a part of the left ones + clutter
    d_at = row_d[np.clip(ly.astype(int), 0, height - 1)]
    is_m = rng.random(n_kp) < matched_frac
    rx = lx - d_at + rng.normal(0, 0.3, n_kp)
    ry = ly + rng.normal(0, 0.5, n_kp)
    roct = np.clip(loct + np.where(rng.random(n_kp) < 0.1, rng.integers(-1, 2, n_kp), 0), 0, n_levels - 1)
    flip = np.where(rng.random(n_kp) < 0.85, p_flip, 0.3)  # some re-detections look different
    rdesc = ldesc.copy()
    for p in np.unique(flip):
        m = flip == p
        rdesc[m] = descriptors_noisy_copy(ldesc[m], rng, float(p))
    clutter = ~is_m
    rw_ = np.array([dims[o][0] for o in roct])
    rh_ = np.array([dims[o][1] for o in roct])
    rx = np.where(clutter, (border + rng.random(n_kp) * (rw_ - 2 * border)) * sf[roct], rx)
    ry = np.where(clutter, (border + rng.random(n_kp) * (rh_ - 2 * border)) * sf[roct], ry)
    rdesc[clutter] = descriptors_uniform(int(clutter.sum()), rng)
    ok = ((rx * inv_sf[roct] >= border) & (rx * inv_sf[roct] <= rw_ - border) &
          (ry * inv_sf[roct] >= border) & (ry * inv_sf[roct] <= rh_ - border))
    perm = rng.permutation(np.nonzero(ok)[0])
    fxc = np.float32(458.0)
    mbf = np.float32(47.9)
    return dict(
        n_levels=n_levels, scale_factors=sf, inv_scale_factors=inv_sf, pyr_left=pyr_l, pyr_right=pyr_r,
        fx=float(fxc), mbf=float(mbf), mb=float(np.float32(mbf / fxc)),
        n_left=n_kp, lx=lx, ly=ly, loct=loct, ldesc=np.ascontiguousarray(ldesc),
        n_right=len(perm), rx=np.ascontiguousarray(rx[perm].astype(np.float32)),
        ry=np.ascontiguousarray(ry[perm].astype(np.float32)),
        roct=np.ascontiguousarray(roct[perm].astype(np.int32)), rdesc=np.ascontiguousarray(rdesc[perm]))


# ------------------------------------------------------- ORB descriptor stage

def make_orb_inputs(n_kp=1000, seed=0, width=640, height=480, n_levels=8, border=19):
    """Inputs of the orientation + steered-BRIEF stage of ORBextractor (reference
    src/ORBextractor.cpp:79-149): a raw and a blurred image pyramid (the blur is an input of the
    stage: the extractor applies cv::GaussianBlur 7x7 / sigma 2 per level, :1131-1132) and keypoints
    in the coordinates of their level, at least `border` px inside it (EDGE_THRESHOLD, :76)."""
    rng = np.random.default_rng(seed + 90001)
    st = make_stereo_pair(8, seed, width, height, n_levels)  # reuse its textured left pyramid
    raw = st["pyr_left"]
    ker = np.array([1, 6, 15, 20, 15, 6, 1], np.float64) / 64.0  # binomial 7-tap stand-in for the blur

    def blur(img):
        f = np.pad(img.astype(np.float64), 3, mode="reflect")
        f = sum(ker[k] * f[:, k:k + img.shape[1]] for k in range(7))
        f = sum(ker[k] * f[k:k + img.shape[0], :] for k in range(7))
        return np.ascontiguousarray(np.rint(f).astype(np.uint8))

    blurred = [blur(a) for a in raw]
    wgt = (1.0 / 1.2) ** np.arange(n_levels)
    lvl = rng.choice(n_levels, size=n_kp, p=wgt / wgt.sum()).astype(np.int32)
    lw = np.array([raw[o].shape[1] for o in lvl])
    lh = np.array([raw[o].shape[0] for o in lvl])
    kx = (border + rng.random(n_kp) * (lw - 2 * border - 1)).astype(np.float32)
    ky = (border + rng.random(n_kp) * (lh - 2 * border - 1)).astype(np.float32)
    half = rng.random(n_kp) < 0.3  # FAST keypoints are integer pixels; refined ones are not: keep both
    kx = np.where(half, kx, np.rint(kx)).astype(np.float32)
    ky = np.where(half, ky, np.rint(ky)).astype(np.float32)
    return dict(n_levels=n_levels, pyr_raw=raw, pyr_blur=blurred, n_kp=n_kp, kx=kx, ky=ky, klevel=lvl)


# ------------------------------------------------------- ORB extractor images (BASELINE config 0)

def make_orb_image(seed=0, width=640, height=480):
    """A synthetic 8-bit frame for ORBextractor::operator() (reference src/ORBextractor.cpp:1087):
    blurred noise with random filled rectangles (corners at every contrast), a low-contrast band
    where only minThFAST finds anything, and a flat patch where nothing does."""
    rng = np.random.default_rng(seed + 515151)
    tex = rng.random((height, width)) * 255.0
    img = 0.5 * _blur(tex, 3) + 0.5 * _blur(tex, 9)
    for _ in range(400):
        x, y = int(rng.integers(0, width - 10)), int(rng.integers(0, height - 10))
        w, h = int(rng.integers(4, 60)), int(rng.integers(4, 60))
        img[y:y + h, x:x + w] = 0.5 * img[y:y + h, x:x + w] + 0.5 * rng.integers(0, 256)
    y0 = height // 3
    band = img[y0:y0 + height // 6]
    img[y0:y0 + height // 6] = 128 + (band - band.mean()) * 0.12  # weak corners only
    img[height - height // 5:height - height // 10, width // 8:width // 2] = 90.0  # flat
    return np.ascontiguousarray(np.clip(np.rint(img), 0, 255).astype(np.uint8))


def warp_orb_image(img, angle_deg=3.0, scale=1.02, shift=(4.0, -3.0)):
    """The second frame of the config-0 pair: `img` under a small similarity (bilinear sampling,
    border replicated)."""
    h, w = img.shape
    a = np.deg2rad(angle_deg)
    ca, sa = np.cos(a) / scale, np.sin(a) / scale
    ys, xs = np.mgrid[0:h, 0:w].astype(np.float64)
    xc, yc = xs - w / 2 - shift[0], ys - h / 2 - shift[1]
    sx = np.clip(ca * xc + sa * yc + w / 2, 0, w - 1.001)
    sy = np.clip(-sa * xc + ca * yc + h / 2, 0, h - 1.001)
    x0, y0 = np.floor(sx).astype(int), np.floor(sy).astype(int)
    fx, fy = sx - x0, sy - y0
    f = img.astype(np.float64)
    out = (f[y0, x0] * (1 - fx) + f[y0, x0 + 1] * fx) * (1 - fy) + (f[y0 + 1, x0] * (1 - fx) + f[y0 + 1, x0 + 1] * fx) * fy
    return np.ascontiguousarray(np.clip(np.rint(out), 0, 255).astype(np.uint8))
