"""Synthetic SMPL-X model files (TEST INFRASTRUCTURE): seeded arrays in the key layout of the licensed
``SMPLX_{MALE,FEMALE,NEUTRAL}.npz`` that ``smplx.create`` reads, for any vertex count V.

* ``kintree_table`` (2,55): the published SMPL-X tree, root parent stored as 2**32 - 1 like the real files.
* vertices scattered around a seeded rest skeleton; every vertex has 1..4 non-zero skinning weights on its nearest
  joints (summing to 1); ``J_regressor`` rows are sparse (up to 6 nearby vertices) and sum to 1; ``f`` random faces.
* ``shapedirs`` (V,3,16) and ``posedirs`` (V,3,486) scaled so that shape offsets are ~1-2 cm per unit beta and pose
  offsets reach several centimetres at poses of ~0.4 rad per joint: the blend shapes matter in every comparison.
"""
import numpy as np

from temporal_inverse_kinematics_b200.smpl_util import SMPLX_FULL_PARENTS

PARENTS55 = list(SMPLX_FULL_PARENTS[:55])


def make_smplx_arrays(V, seed=0, num_betas=16, n_faces=None):
    rs = np.random.RandomState(seed)
    J = 55
    joints = np.zeros((J, 3))
    for i, p in enumerate(PARENTS55):
        joints[i] = rs.standard_normal(3) * 0.1 if p < 0 else joints[p] + rs.standard_normal(3) * 0.1
    owner = rs.randint(0, J, size=V)
    v_template = joints[owner] + rs.standard_normal((V, 3)) * 0.05
    d = np.linalg.norm(v_template[:, None, :] - joints[None], axis=2)          # (V, J)
    weights = np.zeros((V, J))
    for v in range(V):
        n = rs.randint(1, 5)
        near = np.argsort(d[v])[:n]
        weights[v, near] = rs.dirichlet(np.ones(n))
    J_regressor = np.zeros((J, V))
    for j in range(J):
        n = min(V, rs.randint(1, 7))
        near = np.argsort(d[:, j])[:n]
        J_regressor[j, near] = rs.dirichlet(np.ones(n))
    n_faces = n_faces if n_faces is not None else max(1, 2 * V)
    return {
        "v_template": v_template,
        "shapedirs": rs.standard_normal((V, 3, num_betas)) * 0.01,
        "posedirs": rs.standard_normal((V, 3, 486)) * 0.01,
        "J_regressor": J_regressor,
        "weights": weights,
        "kintree_table": np.stack([np.array([2 ** 32 - 1] + PARENTS55[1:], dtype=np.int64), np.arange(J, dtype=np.int64)]),
        "f": rs.randint(0, V, size=(n_faces, 3)).astype(np.uint32),
    }


def write_smplx_npz(path, V, seed=0, with_object_key=True, **kw):
    """Writes one model file; with_object_key adds a pickled object array (real files carry some, e.g. part2num) that a
    loader must never touch.  Returns the arrays written."""
    arrays = make_smplx_arrays(V, seed, **kw)
    extra = {"part2num": np.array({"global": 0}, dtype=object)} if with_object_key else {}
    np.savez(path, **arrays, **extra)
    return arrays


def write_smplx_dir(dirname, V, seed=0):
    """SMPLX_{MALE,FEMALE,NEUTRAL}.npz with the reference's file names -> {gender: arrays}."""
    import os
    return {g: write_smplx_npz(os.path.join(dirname, f"SMPLX_{g.upper()}.npz"), V, seed + i)
            for i, g in enumerate(("male", "female", "neutral"))}
