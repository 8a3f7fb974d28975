"""Shared helpers for the parity tests."""
import os

import numpy as np

from theiasfm_b200 import _abi

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reprojection_golden.npz")


def golden_problem(ext=False):
    """All golden cases as ONE problem: case i = camera i, group i, point i, observation i.  ext=True: the FISHEYE / FOV /
    DIVISION_UNDISTORTION vectors (reprojection_golden_ext.npz)."""
    g = np.load(GOLDEN.replace("reprojection_golden.npz", "reprojection_golden_ext.npz") if ext else GOLDEN)
    n = len(g["model"])
    prob = _abi.Problem(g["ext"], np.zeros(n, np.uint8), np.arange(n, dtype=np.int32), g["model"], g["intr"],
                        np.zeros(n, np.uint32), g["pt"], np.zeros(n, np.uint8), np.arange(n, dtype=np.int32),
                        np.arange(n, dtype=np.int32), g["xy"])
    return prob, g


def rel_err(a, b):
    a = np.asarray(a, float); b = np.asarray(b, float)
    return float(np.max(np.abs(a - b)) / max(1e-300, np.max(np.abs(b))))


def free_masks(p):
    """(free_cam [n_cam,6], free_intr [n_group,10], free_pt [n_pt,4]) booleans."""
    fc = np.ones((p.n_cam, 6), bool)
    fc[:, :3] = (p.ext_const & _abi.EXT_POSITION_CONST)[:, None] == 0
    fc[:, 3:] = (p.ext_const & _abi.EXT_ORIENTATION_CONST)[:, None] == 0
    fi = np.zeros((p.n_group, 10), bool)
    for g in range(p.n_group):
        K = _abi.MODEL_NUM_PARAMS[int(p.group_model[g])]
        for j in range(K):
            fi[g, j] = not ((int(p.group_const_mask[g]) >> j) & 1)
    fp = np.repeat((p.pt_const == 0)[:, None], 4, axis=1)
    return fc, fi, fp


def dense_jacobian(p, J_obs):
    """Assemble the dense (masked, unscaled) Jacobian [2*n_obs, 6*n_cam + 10*n_group + 4*n_pt]."""
    fc, fi, fp = free_masks(p)
    nc, ng, npt, no = p.n_cam, p.n_group, p.n_pt, p.n_obs
    J = np.zeros((2 * no, 6 * nc + 10 * ng + 4 * npt))
    for k in range(no):
        c, q = int(p.obs_cam[k]), int(p.obs_pt[k]); g = int(p.cam_group[c])
        J[2 * k:2 * k + 2, 6 * c:6 * c + 6] = J_obs[k][:, 0:6] * fc[c]
        J[2 * k:2 * k + 2, 6 * nc + 10 * g:6 * nc + 10 * g + 10] = J_obs[k][:, 6:16] * fi[g]
        J[2 * k:2 * k + 2, 6 * nc + 10 * ng + 4 * q:6 * nc + 10 * ng + 4 * q + 4] = J_obs[k][:, 16:20] * fp[q]
    return J


FOUNTAIN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "fountain11_ir.npz")


def fountain_problem(intrinsics_to_optimize=_abi.INTR_NONE):
    """The reference's fountain-11 reconstruction as a Problem (shared PINHOLE intrinsics; constant by default, as in
    the run that produced it: the stored intrinsics equal the ground-truth calibration exactly)."""
    g = dict(np.load(FOUNTAIN))
    # undo the lossless compaction of tests/golden/make_fountain_fixture.py
    for k, dtype, cols in (("pt", np.float64, 4), ("obs_xy", np.float32, 2)):
        g[k] = np.ascontiguousarray(g[k].T).view(dtype).reshape(cols, -1).T.astype(np.float64)
    g["obs_cam"] = g["obs_cam"].astype(np.int32)
    g["obs_pt"] = np.cumsum(g["obs_pt"], dtype=np.int32)
    n = len(g["names"])
    mask = _abi.constant_intrinsics_mask(_abi.MODEL_PINHOLE, intrinsics_to_optimize)
    p = _abi.Problem(g["ext"], np.zeros(n, np.uint8), np.zeros(n, np.int32), [_abi.MODEL_PINHOLE], g["intr"], [mask], g["pt"],
                     np.zeros(len(g["pt"]), np.uint8), g["obs_cam"], g["obs_pt"], g["obs_xy"])
    return p, g


def umeyama_align(src, dst):
    """Similarity transform (scale, rotation, translation) minimising |s R src + t - dst| (Umeyama 1991); what
    AlignReconstructions (transformation/align_reconstructions.cc:97-130) applies to camera positions."""
    src = np.asarray(src, float); dst = np.asarray(dst, float)
    mu_s, mu_d = src.mean(0), dst.mean(0)
    xs, xd = src - mu_s, dst - mu_d
    U, S, Vt = np.linalg.svd(xd.T @ xs / len(src))
    D = np.eye(3)
    if np.linalg.det(U) * np.linalg.det(Vt) < 0:
        D[2, 2] = -1
    R = U @ D @ Vt
    scale = np.trace(np.diag(S) @ D) / (xs ** 2).sum() * len(src)
    t = mu_d - scale * R @ mu_s
    return (scale * (R @ src.T)).T + t, scale
