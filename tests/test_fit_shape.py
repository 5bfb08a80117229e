"""Shape fitting on the GPU (smpl_util.fit_keypoints_shape / tik_fit_keypoints_shape) against the fp64 reference of
tests/fit_shape_reference.py and scipy, on a smplx_synth mesh model with pose-blended landmarks and on the synthetic
full skeleton: one iteration against the dense solve, monotone and recomputed cost, n_iter = 0, a start at the solution,
shape recovery, agreement with scipy at convergence, batch independence, a 20,000-frame sequence against the Schur
reference, guard regions, F = 0, CUDA-graph replay, a non-finite start, errors before launch, and the network's poses
fitted with their shape."""
import ctypes as C

import numpy as np
import pytest
import torch

import fit_reference as FR
import fit_shape_reference as FS
from oracle import smplx_synth
from temporal_inverse_kinematics_b200 import _lib as L
from temporal_inverse_kinematics_b200 import smpl_util as SU

pytestmark = pytest.mark.gpu

_MODELS = {}


def _model(kind):
    if kind not in _MODELS:
        if kind == "mesh":
            a = smplx_synth.make_smplx_arrays(200, seed=5)
            _MODELS[kind] = SU.SmplxBodyModel(a, skeleton="full", landmark_vertex_ids=[10, 20, 30, 40, 199])
        else:
            _MODELS[kind] = SU.SyntheticBodyModel(skeleton="full")
    return _MODELS[kind]


def _cuda(a):
    return None if a is None else torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).cuda()


def _problem(kind, lengths, seed, noise=0.1, target_noise=0.01, pose_scale=0.4, beta_scale=1.0):
    """Per sequence a shape beta* ~ N(0, beta_scale); per frame theta*, tau*; targets = keypoints + noise; the start
    theta* + N(0, noise), tau* + N(0, 0.05)."""
    rs = np.random.RandomState(seed)
    F, S = sum(lengths), len(lengths)
    theta = (rs.standard_normal((F, 22, 3)) * pose_scale).astype(np.float32)
    tau = rs.standard_normal((F, 3)).astype(np.float32)
    betas = (rs.standard_normal((S, 10)) * beta_scale).astype(np.float32)
    per_frame = np.repeat(betas, lengths, axis=0)
    y = SU.keypoints(_cuda(theta), _model(kind), _cuda(per_frame), _cuda(tau)).cpu().numpy()
    y = (y + rs.standard_normal(y.shape) * target_noise).astype(np.float32)
    init = (theta + rs.standard_normal(theta.shape) * noise).astype(np.float32)
    tau0 = (tau + rs.standard_normal(tau.shape) * 0.05).astype(np.float32)
    w = rs.uniform(0.5, 2.0, 17).astype(np.float32)
    wf = rs.uniform(0.5, 2.0, (F, 17)).astype(np.float32)
    return dict(theta=theta, tau=tau, betas=betas, y=y, init=init, tau0=tau0, w=w, wf=wf, lengths=list(lengths))


def _fit(kind, pr, weights=None, fit_transl=True, n_iter=10, prior=1e-3, shape_prior=1e-3, betas=None):
    return SU.fit_keypoints_shape(_cuda(pr["y"]), _model(kind), _cuda(pr["init"]), pr["lengths"], betas,
                                  _cuda(pr["tau0"]), "coco", weights, prior, shape_prior, n_iter, fit_transl)


def _cost_torch(kind, pr, poses, transl, betas, w, prior, shape_prior):
    """E_s recomputed through keypoints() with each sequence's betas broadcast to its frames, in fp64."""
    per_frame = torch.repeat_interleave(betas, torch.tensor(pr["lengths"], device="cuda"), dim=0)
    kp = SU.keypoints(poses, _model(kind), per_frame, transl).double()
    r2 = ((kp - torch.from_numpy(pr["y"]).cuda().double()) ** 2).sum(-1)
    wt = torch.ones_like(r2) if w is None else torch.as_tensor(np.asarray(w), dtype=torch.float64, device="cuda").expand_as(r2)
    d = ((poses.double() - torch.from_numpy(pr["init"]).cuda().double()) ** 2).sum((1, 2))
    e = (wt * r2).sum(-1) + prior * d
    seq = torch.repeat_interleave(torch.arange(len(pr["lengths"]), device="cuda"), torch.tensor(pr["lengths"], device="cuda"))
    out = torch.zeros(len(pr["lengths"]), dtype=torch.float64, device="cuda").index_add_(0, seq, e)
    return out + shape_prior * (betas.double() ** 2).sum(1)


# ------------------------------------------------------------------ 1. one iteration against the dense fp64 reference

# prior_weight = shape_prior_weight = 0.05: every eigenvalue of the damped full system is >= 0.05.  The pose part is
# bounded as in test_fit_keypoints.py (1e-3 rad, 1e-4 m).  The beta system sums, per frame, H_bb,f - C_f^T Y_f with
# |C_f^T Y_f| <= |H_bb,f| (S_f is PSD).  S_f is formed as H_bb,f - Z^T Z with Z = L^-1 C_f from the fp32 factor, so its
# error follows the factor's backward error, ~ P 2^-24 ~ 4e-6 relative to |H_bb,f| (not cond(H_f) times that), plus
# ~1e-6 m of point error through |J_beta| < 0.1.  Over <= 40 frames of |H_bb,f| < 0.2 the error of the B x B matrix is
# < 40 * 0.2 * 4e-6 = 3.2e-5, which moves dbeta by < 3.2e-5 |dbeta| / 0.05 < 1.3e-3 for |dbeta| < 2 (beta* ~ N(0, 1)),
# plus 1e-6 * 0.1 * sqrt(51 * 40) / 0.05 < 1e-4 from the points: bound 2e-3 on beta.
# A beta error e moves each frame's step by |Y_f e| <= |H_f^-1 C_f| e, < 1e-3 rad for e = 2e-3.
TOL_THETA, TOL_TAU, TOL_BETA = 2e-3, 2e-4, 2e-3


@pytest.mark.parametrize("kind", ["mesh", "synthetic"])
@pytest.mark.parametrize("fit_transl,wmode", [(True, "point"), (False, "frame"), (True, "frame"), (False, None)])
def test_one_iteration_matches_dense_reference(kind, fit_transl, wmode):
    lam = 0.05
    pr = _problem(kind, (1, 7, 40), 11 + fit_transl + len(str(wmode)))
    w = {"point": pr["w"], "frame": pr["wf"], None: None}[wmode]
    got = _fit(kind, pr, _cuda(w) if wmode == "frame" else w, fit_transl, 1, lam, lam)
    p, t, b, e0, e = FS.fit_shape(_model(kind), pr["y"], pr["init"], pr["lengths"], None, pr["tau0"], "coco", w, lam, lam,
                                  1, fit_transl, "dense")
    assert (e < e0).all()                                             # the step was taken in the reference
    dth = np.abs(got["poses"].cpu().numpy() - p).max()
    dtau = np.abs(got["transl"].cpu().numpy() - t).max()
    db = np.abs(got["betas"].cpu().numpy() - b).max()
    print(f"one iteration {kind} {fit_transl} {wmode}: theta {dth:.2e} tau {dtau:.2e} beta {db:.2e} (|beta| {np.abs(b).max():.2e})")
    assert dth < TOL_THETA and dtau < TOL_TAU and db < TOL_BETA
    assert np.allclose(got["cost_init"].cpu().numpy(), e0, rtol=1e-5, atol=0)
    assert np.allclose(got["cost"].cpu().numpy(), e, rtol=1e-3, atol=0)
    if not fit_transl:
        assert torch.equal(got["transl"], _cuda(pr["tau0"]))


# ------------------------------------------------------------------ 2-4. cost, n_iter = 0, the solution


@pytest.mark.parametrize("kind", ["mesh", "synthetic"])
def test_monotone_cost_equals_recomputed_cost(kind):
    pr = _problem(kind, (300, 1, 57), 21, noise=0.2)
    got = _fit(kind, pr, pr["w"], True, 10)
    assert bool((got["cost"] <= got["cost_init"]).all())
    assert float((got["cost"] / got["cost_init"]).max()) < 0.5
    want0 = _cost_torch(kind, pr, _cuda(pr["init"]), _cuda(pr["tau0"]), torch.zeros(3, 10, device="cuda"), pr["w"], 1e-3, 1e-3)
    assert torch.allclose(got["cost_init"].double(), want0, rtol=1e-5, atol=0)
    fin = _cost_torch(kind, pr, got["poses"], got["transl"], got["betas"], pr["w"], 1e-3, 1e-3)
    assert torch.allclose(got["cost"].double(), fin, rtol=1e-4, atol=1e-9)


@pytest.mark.parametrize("kind", ["mesh", "synthetic"])
def test_zero_iterations_is_the_identity(kind):
    pr = _problem(kind, (20, 3), 3)
    b0 = _cuda(pr["betas"][:, :7])
    got = _fit(kind, pr, n_iter=0, betas=b0)
    assert torch.equal(got["poses"], _cuda(pr["init"])) and torch.equal(got["transl"], _cuda(pr["tau0"]))
    assert torch.equal(got["betas"][:, :7], b0) and not bool(got["betas"][:, 7:].any())
    assert torch.equal(got["cost"], got["cost_init"])


@pytest.mark.parametrize("kind", ["mesh", "synthetic"])
def test_a_start_at_the_solution_stays(kind):
    pr = _problem(kind, (200, 50), 4, noise=0.0, target_noise=0.0)
    pr["tau0"] = pr["tau"]
    got = _fit(kind, pr, n_iter=10, shape_prior=1e-9, betas=_cuda(pr["betas"]))
    assert (got["poses"] - _cuda(pr["theta"])).abs().max().item() < 1e-4
    assert (got["transl"] - _cuda(pr["tau"])).abs().max().item() < 1e-4
    assert (got["betas"] - _cuda(pr["betas"])).abs().max().item() < 1e-3
    # the start's cost is the shape prior's 1e-9 |beta*|^2 plus fp32 rounding of the points
    data0 = got["cost_init"].double() - 1e-9 * (_cuda(pr["betas"]).double() ** 2).sum(1)
    assert bool((got["cost"] <= got["cost_init"]).all()) and data0.abs().max().item() < 1e-10


# ------------------------------------------------------------------ 5. shape recovery


# The synthetic skeleton only, for the reason given at test_fit_keypoints.py's recovery test (DESIGN.md section 9).
def test_shape_recovery_synthetic():
    kind = "synthetic"
    pr = _problem(kind, (200, 200), 5, noise=0.1, target_noise=0.0, pose_scale=0.3)
    got = _fit(kind, pr, n_iter=30, prior=1e-6, shape_prior=1e-6)
    per_frame = torch.repeat_interleave(got["betas"], 200, dim=0)
    kp = SU.keypoints(got["poses"], _model(kind), per_frame, got["transl"])
    err = (kp - _cuda(pr["y"])).norm(dim=-1).max().item()
    base = SU.fit_keypoints(_cuda(pr["y"]), _model(kind), _cuda(pr["init"]), None, _cuda(pr["tau0"]), "coco", None, 1e-6, 30)
    kp0 = SU.keypoints(base["poses"], _model(kind), None, base["transl"])
    err0 = (kp0 - _cuda(pr["y"])).norm(dim=-1).max().item()
    dbeta = (got["betas"] - _cuda(pr["betas"])).abs().max().item()
    print(f"shape recovery: max point error {err:.2e} m with the shape fit, {err0:.2e} m by fit_keypoints at beta = 0; "
          f"max beta error {dbeta:.2e}")
    assert err <= 5e-4 < err0


# ------------------------------------------------------------------ 6. scipy at convergence


@pytest.mark.parametrize("kind", ["mesh", "synthetic"])
def test_agrees_with_scipy_at_convergence(kind):
    from scipy.optimize import least_squares
    lam = lb = 1e-2
    F = 6
    pr = _problem(kind, (F,), 6, noise=0.1, target_noise=0.02)
    got = _fit(kind, pr, pr["w"], True, 60, lam, lb)
    m = FR.model_arrays(_model(kind))
    sel = SU.keypoint_indices("coco")
    sw = np.repeat(np.sqrt(pr["w"].astype(np.float64)), 3)
    y, th0 = pr["y"].astype(np.float64), pr["init"].reshape(F, 66).astype(np.float64)

    def res_many(Z):                                                 # Z (k, 6*69 + 10) -> (k, residuals)
        k = Z.shape[0]
        X, b = Z[:, :F * 69].reshape(k * F, 69), np.repeat(Z[:, F * 69:], F, 0)
        st = FR.forward(m, X[:, :66], b, X[:, 66:])
        r = ((st["points"][:, sel] - np.tile(y, (k, 1, 1))).reshape(k * F, -1) * sw).reshape(k, -1)
        pp = (np.sqrt(lam) * (X[:, :66] - np.tile(th0, (k, 1)))).reshape(k, -1)
        return np.concatenate([r, pp, np.sqrt(lb) * Z[:, F * 69:]], 1)

    N = F * 69 + 10
    h = 1e-6

    def jac(z):                                                      # central differences, every column in one forward
        E = np.eye(N) * h
        R = res_many(np.concatenate([z + E, z - E]))
        return (R[:N] - R[N:]).T / (2 * h)
    z0 = np.concatenate([np.concatenate([pr["init"].reshape(F, 66), pr["tau0"]], 1).reshape(-1), np.zeros(10)])
    sol = least_squares(lambda z: res_many(z[None])[0], z0.astype(np.float64), jac=jac, method="lm", xtol=1e-15,
                        ftol=1e-15, gtol=1e-15, max_nfev=500)
    c_ref, c_gpu = 2 * sol.cost, float(got["cost"][0])
    dp = np.abs(got["poses"].cpu().numpy().reshape(F, 66) - sol.x[:F * 69].reshape(F, 69)[:, :66]).max()
    db = np.abs(got["betas"][0].cpu().numpy() - sol.x[F * 69:]).max()
    print(f"scipy {kind}: cost rel {abs(c_gpu - c_ref) / c_ref:.2e}, pose {dp:.2e} rad, beta {db:.2e}")
    assert abs(c_gpu - c_ref) / c_ref <= 1e-4 and dp <= 1e-3 and db <= 1e-2


# ------------------------------------------------------------------ 7. batch independence


def _raw(pack, y, w, wpf, pose0, tr, fit_transl, fs, S, b0, lb, prior, n_iter, F, ws, nbytes, pose, tro, bo, cost):
    sel = SU.keypoint_indices("coco")
    s = (C.c_int32 * len(sel))(*sel)
    return L.lib().tik_fit_keypoints_shape(C.byref(pack.c), L.ptr(y), L.ptr(w), wpf, L.ptr(pose0), L.ptr(tr), fit_transl,
                                           L.ptr(fs), S, L.ptr(b0), lb, s, len(sel), prior, n_iter, F, L.ptr(ws), nbytes,
                                           L.ptr(pose), L.ptr(tro), L.ptr(bo), L.ptr(cost), L.stream_ptr())


def _ws(pack, F, S, fit_transl=1):
    n = C.c_int64()
    L.check(L.lib().tik_fit_keypoints_shape_workspace_bytes(C.byref(pack.c), 17, fit_transl, F, S, C.byref(n)))
    return torch.empty(n.value, dtype=torch.uint8, device="cuda"), n.value


def _unaligned(a):
    """A CUDA copy of ``a`` that starts 4 bytes past a 16-byte boundary."""
    t = torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).reshape(-1)
    buf = torch.zeros(t.numel() + 4, device="cuda")
    out = buf[1:1 + t.numel()]
    out.copy_(t)
    return out.view(a.shape)


@pytest.mark.parametrize("kind", ["mesh", "synthetic"])
def test_sequences_do_not_depend_on_the_batch(kind):
    T = 64
    target = _problem(kind, (T,), 70)
    others = _problem(kind, (1, 63, 65, 4099), 71)
    alone = _fit(kind, target, _cuda(target["wf"]), n_iter=5)

    def cat(order):                                                  # "t" is the target sequence, ints index others
        ks, starts = [], np.concatenate([[0], np.cumsum(others["lengths"])])
        out = {k: [] for k in ("y", "init", "tau0", "wf")}
        for o in order:
            src, sl = (target, slice(0, T)) if o == "t" else (others, slice(starts[o], starts[o + 1]))
            for k in out:
                out[k].append(src[k][sl])
            ks.append(T if o == "t" else others["lengths"][o])
        return dict({k: np.concatenate(v) for k, v in out.items()}, lengths=ks)
    for order in (["t", 0, 1, 2, 3], [0, 1, "t", 2, 3], [3, 0, 1, 2, "t"]):
        b = cat(order)
        got = _fit(kind, b, _cuda(b["wf"]), n_iter=5)
        i = order.index("t")
        f0 = sum(b["lengths"][:i])
        for k in ("poses", "transl"):
            assert torch.equal(got[k][f0:f0 + T], alone[k]), (order, k)
        for k in ("betas", "cost_init", "cost"):
            assert torch.equal(got[k][i], alone[k][0]), (order, k)
    # the middle batch again from inputs and outputs at unaligned addresses
    b = cat([0, 1, "t", 2, 3])
    F, S = sum(b["lengths"]), 5
    pack = _model(kind).keypoint_pack(torch.device("cuda"))
    fs = torch.from_numpy(np.concatenate([[0], np.cumsum(b["lengths"])])).cuda()
    ws, nb = _ws(pack, F, S)
    pose, tr, bo, cost = (_unaligned(np.zeros(s)) for s in ((F, 22, 3), (F, 3), (S, 10), (S, 2)))
    L.check(_raw(pack, _unaligned(b["y"]), _unaligned(b["wf"]), 1, _unaligned(b["init"]), _unaligned(b["tau0"]), 1, fs, S,
                 None, 1e-3, 1e-3, 5, F, ws, nb, pose, tr, bo, cost))
    torch.cuda.synchronize()
    f0 = 1 + 63
    assert torch.equal(pose[f0:f0 + T], alone["poses"]) and torch.equal(tr[f0:f0 + T], alone["transl"])
    assert torch.equal(bo[2], alone["betas"][0]) and torch.equal(cost[2, 1], alone["cost"][0])


# ------------------------------------------------------------------ 8. a long sequence: the fp64 sums


@pytest.mark.parametrize("kind", ["mesh", "synthetic"])
def test_long_sequence_matches_the_schur_reference(kind):
    lam = 0.05
    pr = _problem(kind, (20000,), 8)
    got = _fit(kind, pr, None, True, 1, lam, lam)
    p, t, b, e0, e = FS.fit_shape(_model(kind), pr["y"], pr["init"], None, None, pr["tau0"], "coco", None, lam, lam, 1,
                                  True, "schur")
    assert (e < e0).all()
    dth = np.abs(got["poses"].cpu().numpy() - p).max()
    db = np.abs(got["betas"].cpu().numpy() - b).max()
    print(f"20,000 frames {kind}: theta {dth:.2e} beta {db:.2e} (|beta| {np.abs(b).max():.2e})")
    # The frame terms enter the B x B system through fp64 sums, so its error is that of one frame's fp32 terms relative
    # to their sum (the bound of the one-iteration test, which is independent of F), not F times it.
    assert dth < TOL_THETA and db < TOL_BETA


# ------------------------------------------------------------------ 9. hygiene


def test_writes_only_its_outputs_and_workspace():
    """Outputs and the workspace carved out of sentinel-filled buffers, ragged batches at 4-byte offsets."""
    GUARD, SENT = 4096, 12345.0
    kind = "mesh"
    pack = _model(kind).keypoint_pack(torch.device("cuda"))
    for lengths in ((1,), (2, 7), (1, 50, 49)):
        pr = _problem(kind, lengths, 30 + sum(lengths))
        F, S = sum(lengths), len(lengths)
        fs = torch.from_numpy(np.concatenate([[0], np.cumsum(lengths)])).cuda()
        nb = _ws(pack, F, S)[1]
        for shift in (0, 1):
            bufs, outs = [], []
            for n in (F * 66, F * 3, S * 10, S * 2):
                buf = torch.full((GUARD + n + GUARD + 1,), SENT, device="cuda")
                bufs.append(buf)
                outs.append(buf[GUARD + shift:GUARD + shift + n])
            wbuf = torch.full((GUARD + nb // 4 + GUARD,), SENT, device="cuda")
            ws = wbuf[GUARD:GUARD + nb // 4]
            L.check(_raw(pack, _cuda(pr["y"]), _cuda(pr["w"]), 0, _cuda(pr["init"]), _cuda(pr["tau0"]), 1, fs, S, None, 1e-3,
                         1e-3, 5, F, ws, nb, *outs))
            torch.cuda.synchronize()
            for buf, out in zip(bufs, outs):
                n = out.numel()
                assert bool((buf[:GUARD + shift] == SENT).all()) and bool((buf[GUARD + shift + n:] == SENT).all())
                assert bool(torch.isfinite(out).all()) and not bool((out == SENT).any())
            assert bool((wbuf[:GUARD] == SENT).all()) and bool((wbuf[GUARD + nb // 4:] == SENT).all())
            ref = _fit(kind, pr, pr["w"], True, 5)
            assert torch.equal(outs[0].view(F, 22, 3), ref["poses"]) and torch.equal(outs[2].view(S, 10), ref["betas"])


def test_zero_frames_cuda_graph_and_errors_before_launch():
    kind = "mesh"
    m = _model(kind)
    z = SU.fit_keypoints_shape(torch.zeros(0, 17, 3, device="cuda"), m, torch.zeros(0, 66, device="cuda"), betas=np.ones(10))
    assert z["poses"].shape == (0, 22, 3) and z["betas"].shape == (0, 10) and z["cost"].shape == (0,)
    pr = _problem(kind, (300, 1, 99), 9)
    F, S = 400, 3
    pack = m.keypoint_pack(torch.device("cuda"))
    fs = torch.from_numpy(np.array([0, 300, 301, 400])).cuda()
    ws, nb = _ws(pack, F, S)
    args = (_cuda(pr["y"]), _cuda(pr["w"]), 0, _cuda(pr["init"]), _cuda(pr["tau0"]), 1, fs, S, _cuda(pr["betas"] * 0.5),
            1e-3, 1e-3, 10, F, ws, nb)
    eager = [torch.empty(F, 22, 3, device="cuda"), torch.empty(F, 3, device="cuda"), torch.empty(S, 10, device="cuda"),
             torch.empty(S, 2, device="cuda")]
    graphed = [torch.zeros_like(t) for t in eager]
    L.check(_raw(pack, *args, *eager))
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        L.check(_raw(pack, *args, *graphed))
    g.replay()
    g.replay()
    torch.cuda.synchronize()
    assert all(torch.equal(a, b) for a, b in zip(graphed, eager))
    # every error is raised before a launch
    y, p = _cuda(pr["y"]), _cuda(pr["init"])
    for kw in (dict(target=y[:, :16]), dict(init_pose=p[:, :21]), dict(transl=torch.zeros(2, 3, device="cuda")),
               dict(betas=torch.zeros(2, 10, device="cuda")), dict(betas=np.zeros(11)), dict(prior_weight=0.0),
               dict(shape_prior_weight=0.0), dict(shape_prior_weight=float("inf")), dict(weights=-np.ones(17)),
               dict(weights=torch.ones(F, 16, device="cuda")), dict(n_iter=-1), dict(lengths=[300, 99]),
               dict(lengths=[300, 0, 100]), dict(lengths=[]), dict(betas=torch.zeros(3, 11, device="cuda"))):
        a = dict(target=y, model=m, init_pose=p, lengths=[300, 1, 99])
        a.update(kw)
        with pytest.raises(ValueError):
            SU.fit_keypoints_shape(**a)
    with pytest.raises(RuntimeError):
        SU.fit_keypoints_shape(y, m, p, transl=torch.zeros(F, 3))
    with pytest.raises(RuntimeError):
        SU.fit_keypoints_shape(y, m, p, betas=torch.zeros(1, 10))


def test_nonfinite_start_is_returned_unchanged():
    kind = "synthetic"
    pr = _problem(kind, (10, 5, 7), 12)
    pr["y"][12, 2, 0] = np.nan                                       # a frame of the second sequence
    got = _fit(kind, pr, n_iter=5)
    assert torch.equal(got["poses"][10:15], _cuda(pr["init"][10:15])) and torch.equal(got["transl"][10:15], _cuda(pr["tau0"][10:15]))
    assert not bool(got["betas"][1].any()) and bool(torch.isnan(got["cost"][1]))
    assert bool(torch.isfinite(got["cost"][[0, 2]]).all()) and bool((got["cost"][[0, 2]] < got["cost_init"][[0, 2]]).all())


# ------------------------------------------------------------------ 10. end to end


def test_network_poses_fitted_with_their_shape():
    from oracle import stgcn_port as sp, synth
    from temporal_inverse_kinematics_b200 import inference
    from temporal_inverse_kinematics_b200.pose_regressor import IKPoseTrainer
    tr = IKPoseTrainer().eval()
    tr.regressor.load_state_dict(synth.make_regressor_state(sp.build_adjacency("coco", "uniform", 2, 1), seed=0), strict=True)
    tr = tr.cuda()
    body = _model("synthetic")
    rs = np.random.RandomState(13)
    lengths = [40, 1, 75, 17]
    seqs = []
    for n in lengths:
        th = torch.from_numpy((rs.standard_normal((n, 22, 3)) * 0.3).astype(np.float32)).cuda()
        t = torch.from_numpy(rs.standard_normal((n, 3)).astype(np.float32)).cuda()
        seqs.append(SU.keypoints(th, body, rs.standard_normal(10) * 1.5, t).cpu().numpy())
    poses = inference.run_inference_batch(tr, seqs)
    kp = torch.from_numpy(np.concatenate(seqs)).cuda()
    init = torch.from_numpy(np.concatenate(poses)).cuda()
    # One mu per sequence moves slowly from starts far from the targets (DESIGN.md section 9), so the network's poses
    # go through the per-frame fit first, at the mean shape; the shape fit starts there.  Its starting E_s is the data
    # term of those poses (the pose prior is centred on them, beta = 0), so its final cost bounds its data term from above.
    base = SU.fit_keypoints(kp, body, init, n_iter=10)
    got = SU.fit_keypoints_shape(kp, body, base["poses"], lengths, None, base["transl"], n_iter=10)
    seq = torch.from_numpy(np.repeat(np.arange(len(lengths)), lengths)).cuda()

    def data_cost(p, t, b):
        kq = SU.keypoints(p, body, torch.repeat_interleave(b, torch.tensor(lengths, device="cuda"), dim=0), t).double()
        e = ((kq - kp.double()) ** 2).sum((1, 2))
        return torch.zeros(len(lengths), dtype=torch.float64, device="cuda").index_add_(0, seq, e)
    d_base = data_cost(base["poses"], base["transl"], torch.zeros(len(lengths), 10, device="cuda"))
    d_shape = data_cost(got["poses"], got["transl"], got["betas"])
    print("end to end: data cost with the shape fit", d_shape.tolist(), "fit_keypoints at beta = 0", d_base.tolist())
    assert got["betas"].shape == (4, 10)
    assert bool((got["cost"] < got["cost_init"]).all()) and bool((d_shape < d_base).all())
