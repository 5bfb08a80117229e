"""Keypoint fitting on the GPU (smpl_util.fit_keypoints / tik_fit_keypoints) against the fp64 reference of
tests/fit_reference.py and scipy, on a smplx_synth mesh model with pose-blended landmarks and on the synthetic full
skeleton: one iteration, the initial cost, monotone cost, n_iter = 0, a start at the solution, recovery from noise,
agreement with scipy at convergence, batch independence, zero weights, guard regions, F = 0, CUDA-graph replay, and the
network's poses fitted to their own keypoints."""
import ctypes as C

import numpy as np
import pytest
import torch

import fit_reference as FR
from oracle import smplx_synth
from temporal_inverse_kinematics_b200 import _lib as L
from temporal_inverse_kinematics_b200 import smpl_util as SU

pytestmark = pytest.mark.gpu

NAMES = SU.keypoint_names()
CUSTOM = ["nose", "left_wrist", "right_ankle", "left_ear", "spine3", "right_index3", "right_elbow", "left_foot", "nose"]
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


def _problem(kind, F, seed, select="coco", betas_mode="shared", noise=0.1, target_noise=0.01, pose_scale=0.4):
    """theta*, tau*, betas; targets = keypoints(theta*, tau*) + noise; a start theta* + N(0, noise)."""
    rs = np.random.RandomState(seed)
    n = len(SU.keypoint_indices(select))
    theta = (rs.standard_normal((F, 22, 3)) * pose_scale).astype(np.float32)
    tau = rs.standard_normal((F, 3)).astype(np.float32)
    betas = {"none": None, "shared": rs.standard_normal(10).astype(np.float32),
             "frame": rs.standard_normal((F, 10)).astype(np.float32)}[betas_mode]
    bt = _cuda(betas) if betas is not None and betas.ndim == 2 else betas
    y = SU.keypoints(_cuda(theta), _model(kind), bt, _cuda(tau), select).cpu().numpy()
    y = (y + rs.standard_normal(y.shape) * target_noise).astype(np.float32)
    init = (theta + rs.standard_normal(theta.shape) * noise).astype(np.float32)
    tau0 = (tau + rs.standard_normal(tau.shape) * 0.05).astype(np.float32)
    w = rs.uniform(0.5, 2.0, n).astype(np.float32)
    wf = rs.uniform(0.5, 2.0, (F, n)).astype(np.float32)
    return dict(theta=theta, tau=tau, betas=betas, bt=bt, y=y, init=init, tau0=tau0, w=w, wf=wf, n=n)


def _fit(kind, pr, select="coco", weights=None, fit_transl=True, n_iter=10, prior=1e-3, tau0=True):
    return SU.fit_keypoints(_cuda(pr["y"]), _model(kind), _cuda(pr["init"]), pr["bt"], _cuda(pr["tau0"]) if tau0 else None,
                            select, weights, prior, n_iter, fit_transl)


def _cost_torch(kind, pr, poses, transl, select, w, prior):
    kp = SU.keypoints(poses, _model(kind), pr["bt"], transl, select).double()
    r2 = ((kp - torch.from_numpy(pr["y"]).cuda().double()) ** 2).sum(-1)
    wt = torch.ones_like(r2) if w is None else torch.as_tensor(np.asarray(w), dtype=torch.float64, device="cuda").expand_as(r2)
    d = (poses.double() - torch.from_numpy(pr["init"]).cuda().double()) ** 2
    return (wt * r2).sum(-1) + prior * d.sum((1, 2))


# ------------------------------------------------------------------ 1. one iteration against the fp64 reference

# With prior_weight = 0.05 every eigenvalue of H + mu diag(H) is >= 0.05 and the largest is ~ sum_k w_k |lever|^2 < 100,
# so the condition number is < 2e3.  The kernel's points carry ~1e-6 m from fp32 and the SFU sin/cos of its Rodrigues;
# through H^-1 that moves the step by <= 1e-6 * |J| * sqrt(3n) / 0.05 ~ 2e-4 rad, and the fp32 Cholesky adds
# cond * 2^-24 * |delta| < 1e-4 * |delta|.  Bound: 1e-3 rad on theta and 1e-4 m on tau.
TOL_THETA, TOL_TAU = 1e-3, 1e-4


@pytest.mark.parametrize("kind", ["mesh", "synthetic"])
@pytest.mark.parametrize("betas_mode,fit_transl,wmode,select", [
    ("shared", True, "point", "coco"), ("frame", False, "frame", "custom"), ("none", True, None, "custom"),
    ("frame", True, "frame", "coco"), ("shared", False, None, "coco")])
def test_one_iteration_matches_reference(kind, betas_mode, fit_transl, wmode, select):
    sel = CUSTOM if select == "custom" else "coco"
    F, prior = 40, 0.05
    pr = _problem(kind, F, 11 + len(betas_mode), sel, betas_mode)
    w = {"point": pr["w"], "frame": pr["wf"], None: None}[wmode]
    got = _fit(kind, pr, sel, _cuda(w) if wmode == "frame" else w, fit_transl, 1, prior)
    p, t, e0, e = FR.fit(_model(kind), pr["y"], pr["init"], pr["betas"], pr["tau0"], sel, w, prior, 1, fit_transl)
    assert np.isfinite(e).all() and (e < e0).all()                   # the step was taken in the reference
    dth = np.abs(got["poses"].cpu().numpy() - p).max()
    dtau = np.abs(got["transl"].cpu().numpy() - t).max()
    print(f"one iteration {kind} {betas_mode} {fit_transl} {wmode} {select}: theta {dth:.2e} tau {dtau:.2e}")
    assert dth < TOL_THETA and dtau < TOL_TAU
    assert np.allclose(got["cost_init"].cpu().numpy(), e0, rtol=1e-5, atol=0)
    if not fit_transl:
        assert torch.equal(got["transl"], _cuda(pr["tau0"]))


# ------------------------------------------------------------------ 2-5. cost, monotonicity, n_iter = 0, the solution


@pytest.mark.parametrize("kind", ["mesh", "synthetic"])
def test_cost_init_and_monotone_cost(kind):
    F = 4099
    pr = _problem(kind, F, 21, "coco", "frame", noise=0.2)
    got = _fit(kind, pr, "coco", pr["w"], True, 10, 1e-3)
    want = _cost_torch(kind, pr, _cuda(pr["init"]), _cuda(pr["tau0"]), "coco", pr["w"], 1e-3)
    assert torch.allclose(got["cost_init"].double(), want, rtol=1e-5, atol=0)
    assert bool((got["cost"] <= got["cost_init"]).all())
    assert float((got["cost"] / got["cost_init"]).median()) < 0.1
    # the returned cost is E at the returned pose
    fin = _cost_torch(kind, pr, got["poses"], got["transl"], "coco", pr["w"], 1e-3)
    assert torch.allclose(got["cost"].double(), fin, rtol=1e-4, atol=1e-9)


@pytest.mark.parametrize("kind", ["mesh", "synthetic"])
def test_zero_iterations_is_the_identity(kind):
    pr = _problem(kind, 100, 3)
    got = _fit(kind, pr, n_iter=0)
    assert torch.equal(got["poses"], _cuda(pr["init"])) and torch.equal(got["transl"], _cuda(pr["tau0"]))
    assert torch.equal(got["cost"], got["cost_init"])
    got = SU.fit_keypoints(_cuda(pr["y"]), _model(kind), _cuda(pr["init"]).reshape(100, 66), pr["bt"], None, n_iter=0)
    assert torch.equal(got["transl"], torch.zeros(100, 3, device="cuda"))


@pytest.mark.parametrize("kind", ["mesh", "synthetic"])
def test_a_start_at_the_solution_stays(kind):
    pr = _problem(kind, 500, 4, noise=0.0, target_noise=0.0)
    pr["tau0"] = pr["tau"]
    got = _fit(kind, pr, n_iter=10)
    assert (got["poses"] - _cuda(pr["theta"])).abs().max().item() < 1e-5
    assert (got["transl"] - _cuda(pr["tau"])).abs().max().item() < 1e-5
    assert bool((got["cost"] <= got["cost_init"]).all()) and got["cost_init"].max().item() < 1e-10


# The synthetic skeleton only: on the mesh test model (random pose-blend directions that move the landmarks by several
# cm) some frames converge more slowly than the fp64 reference of the same schedule; DESIGN.md section 9 has the numbers.
@pytest.mark.parametrize("kind", ["synthetic"])
def test_recovery_from_noisy_starts(kind):
    F = 256
    pr = _problem(kind, F, 5, noise=0.15, target_noise=0.0, pose_scale=0.3)
    got = _fit(kind, pr, n_iter=30, prior=1e-6)
    kp = SU.keypoints(got["poses"], _model(kind), pr["bt"], got["transl"])
    err = (kp - _cuda(pr["y"])).norm(dim=-1).max(dim=1).values
    ratio = got["cost"] / got["cost_init"]
    print(f"recovery {kind}: max point error {err.max().item():.2e} m, max cost ratio {ratio.max().item():.2e}")
    assert err.max().item() <= 5e-4
    assert ratio.max().item() <= 1e-3


# ------------------------------------------------------------------ 7. scipy at convergence


@pytest.mark.parametrize("kind", ["mesh", "synthetic"])
def test_agrees_with_scipy_at_convergence(kind):
    from scipy.optimize import least_squares
    F, lam = 24, 1e-2
    pr = _problem(kind, F, 6, noise=0.1, target_noise=0.02)
    got = _fit(kind, pr, "coco", pr["w"], True, 50, lam)
    m = FR.model_arrays(_model(kind))
    sel = SU.keypoint_indices("coco")
    b = FR.betas_rows(pr["betas"], 1, 10)
    sw = np.repeat(np.sqrt(pr["w"].astype(np.float64)), 3)

    def res_many(X, f):                                              # X (k, 69) -> (k, 51 + 66) residual vectors
        st = FR.forward(m, X[:, :66], np.repeat(b, X.shape[0], 0), X[:, 66:])
        r = (st["points"][:, sel] - pr["y"][f].astype(np.float64)).reshape(X.shape[0], -1) * sw
        return np.concatenate([r, np.sqrt(lam) * (X[:, :66] - pr["init"][f].reshape(1, 66))], 1)

    worst_c, worst_p = 0.0, 0.0
    for f in range(F):
        x0 = np.concatenate([pr["init"][f].reshape(66), pr["tau0"][f]]).astype(np.float64)
        h = 1e-6

        def jac(x):                                                  # central differences, all columns in one forward
            E = np.eye(69) * h
            R = res_many(np.concatenate([x + E, x - E]), f)
            return (R[:69] - R[69:]).T / (2 * h)
        sol = least_squares(lambda x: res_many(x[None], f)[0], x0, jac=jac, method="lm", xtol=1e-15, ftol=1e-15,
                            gtol=1e-15, max_nfev=2000)
        c_ref = 2 * sol.cost
        c_gpu = float(got["cost"][f])
        worst_c = max(worst_c, abs(c_gpu - c_ref) / c_ref)
        worst_p = max(worst_p, np.abs(got["poses"][f].cpu().numpy().reshape(66) - sol.x[:66]).max())
    print(f"scipy {kind}: cost rel {worst_c:.2e}, pose {worst_p:.2e} rad")
    assert worst_c <= 1e-4 and worst_p <= 1e-3


# ------------------------------------------------------------------ 8. batch independence


def _raw(pack, y, w, wpf, pose0, b, bpf, tr, fit_transl, sel, prior, n_iter, F, pose_out, tr_out, cost):
    s = (C.c_int32 * len(sel))(*sel)
    return L.lib().tik_fit_keypoints(C.byref(pack.c), L.ptr(y), L.ptr(w), wpf, L.ptr(pose0), L.ptr(b), bpf, L.ptr(tr),
                                     fit_transl, s, len(sel), prior, n_iter, F, L.ptr(pose_out), L.ptr(tr_out), L.ptr(cost),
                                     L.stream_ptr())


def _unaligned(a):
    """A CUDA copy of ``a`` that starts 4 bytes past a 16-byte boundary."""
    t = torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).reshape(-1)
    buf = torch.zeros(t.numel() + 4, device="cuda")
    out = buf[1:1 + t.numel()]
    out.copy_(t)
    return out.view(a.shape)


@pytest.mark.parametrize("kind", ["mesh", "synthetic"])
@pytest.mark.parametrize("F", [1, 63, 64, 65, 4099])
def test_frames_do_not_depend_on_the_batch(kind, F):
    pr = _problem(kind, F, 7 + F, "coco", "frame")
    wf = _cuda(pr["wf"])
    full = SU.fit_keypoints(_cuda(pr["y"]), _model(kind), _cuda(pr["init"]), pr["bt"], _cuda(pr["tau0"]), "coco", wf, 1e-3, 10)
    for i in sorted({0, F // 2, F - 1}):
        one = SU.fit_keypoints(_cuda(pr["y"][i:i + 1]), _model(kind), _cuda(pr["init"][i:i + 1]), pr["bt"][i:i + 1],
                               _cuda(pr["tau0"][i:i + 1]), "coco", wf[i:i + 1], 1e-3, 10)
        for k in ("poses", "transl", "cost_init", "cost"):
            assert torch.equal(full[k][i:i + 1], one[k]), (i, k)
    # the same call from inputs and outputs at unaligned addresses
    pack = _model(kind).keypoint_pack(torch.device("cuda"))
    sel = SU.keypoint_indices("coco")
    pose, tr, cost = _unaligned(np.zeros((F, 22, 3))), _unaligned(np.zeros((F, 3))), _unaligned(np.zeros((F, 2)))
    L.check(_raw(pack, _unaligned(pr["y"]), _unaligned(pr["wf"]), 1, _unaligned(pr["init"]), _unaligned(pr["betas"]), 1,
                 _unaligned(pr["tau0"]), 1, sel, 1e-3, 10, F, pose, tr, cost))
    torch.cuda.synchronize()
    assert torch.equal(pose, full["poses"]) and torch.equal(tr, full["transl"])
    assert torch.equal(cost[:, 0], full["cost_init"]) and torch.equal(cost[:, 1], full["cost"])


# ------------------------------------------------------------------ 9. hygiene


@pytest.mark.parametrize("kind", ["mesh", "synthetic"])
def test_zero_weight_is_leaving_the_point_out(kind):
    pr = _problem(kind, 300, 8, CUSTOM)
    w = pr["w"].copy()
    w[[1, 4]] = 0
    keep = [k for k in range(len(CUSTOM)) if w[k] != 0]
    # A zero weight makes every FMA of its rows in H and g an exact no-op, so both calls take the same steps; only the
    # cost sums run in another order.  Near convergence a step whose cost change is below fp32 rounding of E may then be
    # accepted in one call and rejected in the other, so the comparison stops after three clearly decisive iterations.
    got = _fit(kind, pr, CUSTOM, w, True, 3)
    pr2 = dict(pr, y=pr["y"][:, keep])
    sub = _fit(kind, pr2, [CUSTOM[k] for k in keep], w[keep], True, 3)
    assert (got["poses"] - sub["poses"]).abs().max().item() < 1e-6
    assert (got["transl"] - sub["transl"]).abs().max().item() < 1e-6
    assert torch.allclose(got["cost"], sub["cost"], rtol=1e-5, atol=0)


def test_fit_writes_only_its_outputs():
    """Outputs carved out of sentinel-filled buffers, F around the 8-frame CTA and at 4-byte offsets."""
    GUARD, SENT = 4096, 12345.0
    kind = "mesh"
    pack = _model(kind).keypoint_pack(torch.device("cuda"))
    sel = SU.keypoint_indices("coco")
    for F in (1, 7, 8, 9, 100):
        pr = _problem(kind, F, 30 + F, "coco", "frame")
        for shift in (0, 1):
            bufs, outs = [], []
            for width in (66, 3, 2):
                buf = torch.full((GUARD + F * width + GUARD + 1,), SENT, device="cuda")
                bufs.append(buf)
                outs.append(buf[GUARD + shift:GUARD + shift + F * width])
            L.check(_raw(pack, _cuda(pr["y"]), _cuda(pr["w"]), 0, _cuda(pr["init"]), _cuda(pr["betas"]), 1,
                         _cuda(pr["tau0"]), 1, sel, 1e-3, 5, F, *outs))
            torch.cuda.synchronize()
            for buf, out in zip(bufs, outs):
                n = out.numel()
                assert bool((buf[:GUARD + shift] == SENT).all()) and bool((buf[GUARD + shift + n:] == SENT).all()), (F, shift)
                assert bool(torch.isfinite(out).all()) and not bool((out == SENT).any()), (F, shift)
            ref = _fit(kind, pr, "coco", pr["w"], True, 5)
            assert torch.equal(outs[0].view(F, 22, 3), ref["poses"]) and torch.equal(outs[2].view(F, 2)[:, 1], ref["cost"])


def test_zero_frames_cuda_graph_and_errors_before_launch():
    kind = "mesh"
    m = _model(kind)
    z = SU.fit_keypoints(torch.zeros(0, 17, 3, device="cuda"), m, torch.zeros(0, 66, device="cuda"), np.ones(10))
    assert z["poses"].shape == (0, 22, 3) and z["cost"].shape == (0,)
    F = 1000
    pr = _problem(kind, F, 9, "coco", "frame")
    pack = m.keypoint_pack(torch.device("cuda"))
    sel = SU.keypoint_indices("coco")
    args = (_cuda(pr["y"]), _cuda(pr["w"]), 0, _cuda(pr["init"]), _cuda(pr["betas"]), 1, _cuda(pr["tau0"]), 1, sel, 1e-3, 10, F)
    eager = [torch.empty(F, 22, 3, device="cuda"), torch.empty(F, 3, device="cuda"), torch.empty(F, 2, device="cuda")]
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
               dict(prior_weight=-1.0), dict(weights=-np.ones(17)), dict(weights=np.ones(16)),
               dict(weights=torch.ones(F, 16, device="cuda")), dict(n_iter=-1), dict(select=CUSTOM)):
        a = dict(target=y, model=m, init_pose=p)
        a.update(kw)
        with pytest.raises(ValueError):
            SU.fit_keypoints(**a)
    with pytest.raises(RuntimeError):
        SU.fit_keypoints(y, m, p, transl=torch.zeros(F, 3))
    with pytest.raises(RuntimeError):
        SU.fit_keypoints(y, m, p, weights=torch.ones(F, 17))


def test_nonfinite_start_is_returned_unchanged():
    kind = "synthetic"
    pr = _problem(kind, 10, 12)
    pr["y"][3, 2, 0] = np.nan
    got = _fit(kind, pr, n_iter=5)
    assert torch.equal(got["poses"][3], _cuda(pr["init"][3])) and bool(torch.isnan(got["cost"][3]))
    assert bool(torch.isfinite(got["cost"][np.r_[0:3, 4:10]]).all())


# ------------------------------------------------------------------ 10. end to end


def test_network_poses_fitted_to_their_own_keypoints():
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
        seqs.append(SU.keypoints(th, body, None, t).cpu().numpy())
    poses = inference.run_inference_batch(tr, seqs)
    kp = torch.from_numpy(np.concatenate(seqs)).cuda()
    init = torch.from_numpy(np.concatenate(poses)).cuda()                 # (sum F, 66), the packed frames
    got = SU.fit_keypoints(kp, body, init, n_iter=10)
    assert got["poses"].shape == (sum(lengths), 22, 3)
    assert bool((got["cost"] < got["cost_init"]).all())
