"""Geometry utilities behind the reference's `utils.py` API
(reference evenvizion/processing/utils.py:23-363); arithmetic runs in libevz.so."""
import json

import numpy as np
import torch

from .. import _lib
from .constants import INFINITY_COORDINATE, THRESHOLD_FOR_FIND_HOMOGRAPHY, LENGTH_ACCOUNTED_POINTS, \
    RANSAC_HYPOTHESES, RANSAC_SEED


class HomographyException(Exception):
    """reference utils.py:23-38."""

    def __init__(self, message="can't calculate homography matrix"):
        self.message = message
        super().__init__(message)


def _engine():
    from .. import default_engine
    return default_engine()


def _pack_points(eng, pts_a, pts_b):
    a = np.asarray(pts_a, np.float32).reshape(-1, 2)
    b = np.asarray(pts_b, np.float32).reshape(-1, 2)
    if len(a) != len(b):
        raise ValueError("pts_a and pts_b differ in length")
    n = len(a)
    pts = torch.zeros((max(n, 4), 4), dtype=torch.float32)
    pts[:n, :2] = torch.from_numpy(a)
    pts[:n, 2:] = torch.from_numpy(b)
    dev = eng.device
    return (pts.to(dev), torch.zeros(1, dtype=torch.int32, device=dev),
            torch.full((1,), n, dtype=torch.int32, device=dev), n)


def remove_double_matching(pts_a, pts_b):
    """reference utils.py:41-68: unique (x, y) keys of pts_a, first position / last value.  Host-side
    helper for API compatibility; the device pipeline fuses this step into the filter kernel."""
    matching = {}
    for i in range(len(pts_a)):
        matching[(pts_a[i][0], pts_a[i][1])] = pts_b[i]
    return [np.array(k) for k in matching], list(matching.values())


def homography_transformation(vector, matrix_H):
    """reference utils.py:71-92."""
    while len(vector) < 3:
        vector = np.append(vector, [1])
    new_vector = np.dot(matrix_H, vector)
    return new_vector[:-1] / new_vector[-1]


def inverse_homography_transformation(vector, matrix_H):
    """reference utils.py:95-115."""
    while len(vector) < 3:
        vector = np.append(vector, [1])
    new_vector = np.dot(np.linalg.inv(matrix_H), vector)
    return new_vector[:-1] / new_vector[-1]


def matrix_superposition(H, matrix_H_superposition, matrix_H_first=False):
    """reference utils.py:118-145 (one step of the left fold; the batched form is superposition_dict)."""
    if H is not None:
        if matrix_H_first:
            matrix_H_superposition = H
        else:
            matrix_H_superposition = np.dot(H, matrix_H_superposition)
            matrix_H_superposition = np.divide(matrix_H_superposition, matrix_H_superposition[2][2])
    return matrix_H_superposition


def read_homography_dict(path_to_homography_dict):
    """reference utils.py:148-181."""
    with open(path_to_homography_dict, "r") as curr_json:
        homography_dict = json.load(curr_json)
    if "resize_info" not in homography_dict:
        raise ValueError("Specify the height and width of the frame "
                         "for which the homography matrix was obtained")
    resize_info = homography_dict.pop("resize_info")
    homography_dict = {int(k): v for k, v in homography_dict.items()}
    return homography_dict, resize_info


def superposition_dict(homography_dict):
    """Cumulative superposition for every frame (reference utils.py:184-211) as a parallel prefix
    product on the GPU.  The reference folds on the LEFT (S_k = H_k . S_{k-1}); the scan kernel
    multiplies on the right, so it runs on the transposes.  `H is None` entries carry S forward."""
    out = {1: [[1, 0, 0], [0, 1, 0], [0, 0, 1]]}
    keys = list(homography_dict.keys())
    if not keys:
        return out
    n = len(keys)
    Ht = np.tile(np.eye(3), (n, 1, 1))
    status = np.ones(n, np.int32)
    for i, k in enumerate(keys):
        H = homography_dict[k]["H"]
        if H is not None:
            Ht[i] = np.asarray(H, np.float64).T
            status[i] = 0
    eng = _engine()
    S, _, _ = eng.chain_scan(torch.from_numpy(Ht.reshape(n, 9)).to(eng.device),
                             torch.from_numpy(status).to(eng.device), policy=False, want_fixed=False)
    S = S.cpu().numpy().reshape(n, 3, 3).transpose(0, 2, 1)
    seen_valid = False
    for i, k in enumerate(keys):
        if status[i] == 0 and not seen_valid:
            out[k] = homography_dict[k]["H"]           # the reference stores the first matrix itself
            seen_valid = True
        else:
            out[k] = np.ascontiguousarray(S[i]) if seen_valid else None
    return out


def are_infinity_coordinates(coordinates_value):
    """reference utils.py:214-230."""
    try:
        return any(i >= INFINITY_COORDINATE for i in coordinates_value)
    except TypeError:
        return coordinates_value >= INFINITY_COORDINATE


def read_json_with_coordinates(path_to_coordinate):
    """reference utils.py:233-255."""
    with open(path_to_coordinate, 'r') as f:
        coordinates = json.load(f)
    return {int(k): v for k, v in coordinates.items()}


def find_point_displacement(matrix_H, pts_a, pts_b):
    """Group points by round(||H a - b||) (reference utils.py:289-325).  The rounded displacements are
    computed by the static-filter kernel; only the grouping of the integers happens on the host."""
    if len(pts_a) != len(pts_b):
        raise ValueError("in find_static_part, len(pts_a) != len(pts_b)")
    eng = _engine()
    pts, off, cnt, n = _pack_points(eng, pts_a, pts_b)
    H = torch.from_numpy(np.asarray(matrix_H, np.float64).reshape(1, 9)).to(eng.device)
    status = torch.zeros(1, dtype=torch.int32, device=eng.device)
    if n > _lib.EVZ_MAX_KP:
        raise ValueError("at most %d point pairs are supported" % _lib.EVZ_MAX_KP)
    _, _, _, flags, r = eng.static_filter(pts, off, cnt, H, status, want_r=True, max_cnt=n)
    if int(flags[0]):
        raise OverflowError("a displacement is not finite or exceeds %d px" % _lib.EVZ_R_MAX)
    groups = {}
    for i, v in enumerate(r[:n].cpu().tolist()):
        groups.setdefault(v, []).append(i)
    return groups


def get_largest_group_points(r_moving_dict, pts_a, pts_b):
    """reference utils.py:258-286: the largest group, ties to the first inserted key."""
    k_max_len, max_len = None, 0
    for key, value in r_moving_dict.items():
        if len(value) > max_len:
            max_len, k_max_len = len(value), key
    idx = r_moving_dict[k_max_len]
    return np.array([pts_a[i] for i in idx]), np.array([pts_b[i] for i in idx])


def compute_homography(pts_a, pts_b, matrix_H_prev=None, n_hyp=None, seed=None, pair_id=0, confidence=None):
    """Second-level RANSAC homography with the 70 % inlier gate (reference utils.py:328-363).
    matrix_H_prev: superposition between the origin and frame_a; both point sets are mapped through
    it first, so that H lives in the fixed plane.  confidence: None scores n_hyp hypotheses; a float in (0, 1) stops
    where cv2's RANSAC would (n_hyp = maxIters).  Raises HomographyException."""
    eng = _engine()
    pts, off, cnt, n = _pack_points(eng, pts_a, pts_b)
    if n < 4:
        raise HomographyException("not enough points in homography calculation")
    status = torch.zeros(1, dtype=torch.int32, device=eng.device)
    pre = None
    if matrix_H_prev is not None:
        pre = torch.from_numpy(np.asarray(matrix_H_prev, np.float64).reshape(1, 9)).to(eng.device)
    out = eng.find_homography(pts, off, cnt, status, max(n, 4), RANSAC_HYPOTHESES if n_hyp is None else n_hyp,
                              RANSAC_SEED if seed is None else seed, pair_id, 2, THRESHOLD_FOR_FIND_HOMOGRAPHY,
                              LENGTH_ACCOUNTED_POINTS, _lib.ST_NO_MODEL_2, pre_H=pre, confidence=confidence)
    s = int(status[0])
    if s == _lib.ST_FEW_INLIERS:
        raise HomographyException("not enough points in homography calculation")
    if s != 0:
        raise HomographyException()
    return out["H"][0].cpu().numpy().reshape(3, 3)
