"""Kinematic optimiser (SURVEY.md 8(a) E1-E3) against golden vectors produced by the reference's OWN functions
(tests/golden/make_kinopt_golden.py runs optimize_trajectory.py from the reference tree on a synthetic 14-frame clip)."""
import os

import numpy as np
import pytest

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "kinopt")


@pytest.fixture(scope="module")
def data(chd):
    inp, sk, fj, run = (np.load(os.path.join(G, n + ".npz")) for n in ("inputs", "skeleton", "funjac", "run"))
    b = chd.prepare.load_bvh(os.path.join(G, "skeleton.bvh"))
    return dict(inp=inp, sk=sk, fj=fj, run=run, bvh=b, F=inp["poses3D"].shape[0])


def make_model(chd, d, contacts, normal, point):
    ko = chd.kinopt
    j2n, pw, dw = ko.make_weights(d["inp"]["poses2D"], d["inp"]["conf"], d["inp"]["pp"], d["inp"]["focal"])
    p = ko.Problem(d["bvh"].parents, d["sk"]["offsets"], d["inp"]["poses3D"], d["inp"]["root_pos"], j2n, pw, dw, contacts, normal, point)
    return ko._Model(p), (j2n, pw, dw)


def test_skeleton_fit_and_weights_match_reference(chd, data):
    ko = chd.kinopt
    targets = data["inp"]["poses3D"][:, ko.FORWARD] + data["inp"]["root_pos"][:, None]
    np.testing.assert_array_equal(targets, data["sk"]["targets"])
    np.testing.assert_allclose(ko.update_skeleton(data["bvh"].parents, data["bvh"].offsets, targets), data["sk"]["offsets"], atol=1e-12)
    _, (j2n, pw, dw) = make_model(chd, data, data["inp"]["vel"], np.zeros(3), np.zeros(3))
    np.testing.assert_allclose(j2n, data["fj"]["j2n"], atol=1e-15)
    np.testing.assert_allclose(pw, data["fj"]["pw"], atol=1e-15)
    np.testing.assert_allclose(dw, data["fj"]["dw"], atol=1e-15)
    assert [ko.FORWARD[k] for k in ko.BACKWARD] == list(range(28))


@pytest.mark.parametrize("tag,floor_w", [("a", 0.0), ("b", 10.0)])
def test_residual_and_jacobian_vs_reference(chd, data, tag, floor_w):
    import scipy.sparse
    import torch
    ko = chd.kinopt
    fj, F = data["fj"], data["F"]
    m, _ = make_model(chd, data, data["inp"]["vel"], fj["normal"], fj["point"])
    x = torch.as_tensor(fj["x_" + tag].reshape(F, -1))
    w = ko.StageWeights(floor=floor_w)
    f = m.residual_vector(x, w).numpy()
    assert f.shape == fj["f_" + tag].shape
    # the reference's quaternion path carries 1e-10 relative noise (axis / (|axis| + 1e-10)); projection weight 1000
    np.testing.assert_allclose(f, fj["f_" + tag], rtol=0, atol=2e-7)
    Jm, Jr = m.dense_jacobian(x, w).numpy(), scipy.sparse.load_npz(os.path.join(G, "jac_%s.npz" % tag)).toarray()
    assert Jm.shape == Jr.shape
    nproj = F * 28 * 2
    np.testing.assert_allclose(Jm[nproj:], Jr[nproj:], rtol=0, atol=1e-6)          # every group but the projection term
    # projection rows: exact derivative here (central differences); the reference's analytic rows are not (see kinopt.py)
    rng = np.random.default_rng(0)
    cols = np.concatenate([rng.choice(F * 87, 10, replace=False), [0, 1, 2, 87, 89]])
    eps, worst_ref = 1e-6, 0.0
    for c in cols:
        xp, xm = x.reshape(-1).clone(), x.reshape(-1).clone()
        xp[c] += eps
        xm[c] -= eps
        fd = (m.residual_vector(xp.reshape(F, -1), w) - m.residual_vector(xm.reshape(F, -1), w)).numpy() / (2 * eps)
        scale = max(1.0, np.abs(Jm[:, c]).max())
        assert np.abs(fd - Jm[:, c]).max() / scale < 1e-7
        worst_ref = max(worst_ref, np.abs(fd[:nproj] - Jr[:nproj, c]).max() / scale)
    assert worst_ref > 1e-3      # documents the reference's misplaced root-translation columns (optimize_trajectory.py:106-137)


def test_normal_equations_and_banded_solver(chd, data):
    import torch
    ko = chd.kinopt
    F = 6
    d = dict(data)
    d["inp"] = {k: (v[:F] if getattr(v, "ndim", 0) >= 1 and v.shape[0] == data["F"] else v) for k, v in data["inp"].items()}
    m, _ = make_model(chd, d, d["inp"]["vel"], data["fj"]["normal"], data["fj"]["point"])
    x = torch.as_tensor(data["fj"]["x_b"].reshape(data["F"], -1)[:F].copy())
    w = ko.StageWeights(floor=10.0)
    cost, H, g = m.normal_equations(x, w)
    J = m.dense_jacobian(x, w)
    r = m.residual_vector(x, w)
    assert abs(cost - 0.5 * float(r @ r)) < 1e-9 * cost
    Hd = (J.T @ J).numpy()
    n = ko.NV
    for f in range(F):
        np.testing.assert_allclose(H[0][f].numpy(), Hd[f * n:(f + 1) * n, f * n:(f + 1) * n], rtol=1e-10, atol=1e-6)
        if f + 1 < F:
            np.testing.assert_allclose(H[1][f].numpy(), Hd[(f + 1) * n:(f + 2) * n, f * n:(f + 1) * n], rtol=1e-10, atol=1e-6)
        if f + 2 < F:
            np.testing.assert_allclose(H[2][f].numpy(), Hd[(f + 2) * n:(f + 3) * n, f * n:(f + 1) * n], rtol=1e-10, atol=1e-6)
        if f + 3 < F:
            assert np.abs(Hd[(f + 3) * n:, f * n:(f + 1) * n]).max() == 0.0           # nothing outside the two block bands
    np.testing.assert_allclose(g.reshape(-1).numpy(), (J.T @ r).numpy(), rtol=1e-10, atol=1e-6)
    lam = 1e-3
    s = ko._banded_cholesky_solve(torch, H, g, lam).reshape(-1).numpy()
    A = Hd + lam * np.diag(np.diag(Hd))
    np.testing.assert_allclose(s, np.linalg.solve(A, g.reshape(-1).numpy()), rtol=1e-6, atol=1e-9)
    sd = ko._banded_cholesky_solve(torch, H, g, lam, dense=True).reshape(-1).numpy()      # the GPU path: one dense factorisation
    np.testing.assert_allclose(sd, s, rtol=1e-8, atol=1e-10)


def test_objective_at_reference_solution_and_own_run(chd, data):
    import torch
    ko = chd.kinopt
    run, inp, F = data["run"], data["inp"], data["F"]
    m, _ = make_model(chd, data, run["newvel"], run["plane_normal"], run["plane_point"])
    w = ko.StageWeights(floor=10.0)
    # same objective: the reference's own final point costs the same under this model
    assert abs(m.cost(torch.as_tensor(run["x_fin"].reshape(F, -1)), w) - float(run["cost"])) < 1e-6 * float(run["cost"])
    # like-for-like final stage: the reference's fitted floor given, same contacts, same evaluation budget (50 + 50)
    res = ko.optimize_trajectory(inp["poses2D"], inp["conf"], inp["poses3D"], inp["root_pos"], inp["joint_angles"], data["bvh"].parents,
                                 data["bvh"].offsets, inp["pp"][0], inp["pp"][1], inp["focal"], inp["vel"],
                                 plane_normal=run["plane_normal"], plane_point=run["plane_point"])
    anim, new3d, proj, pn, pp, vel, info = res
    assert info["stage2"]["nfev"] <= 50 and info["stage1"]["nfev"] <= 50
    assert info["stage2"]["cost"] <= float(run["cost"])              # matches or beats the reference's final objective (2774 vs ~1400)
    assert abs(m.cost(torch.as_tensor(info["x"]), w) - info["stage2"]["cost"]) < 1e-6 * info["stage2"]["cost"]
    np.testing.assert_array_equal(vel, inp["vel"])                   # given floor: labels untouched (optimize_trajectory.py:739)
    # re-projection error of the confident joints [px] no worse than the reference's
    on = inp["conf"][:, :25] > 0.3
    e_mine = np.linalg.norm(proj[:, :25] - inp["poses2D"][:, :25], axis=-1)[on].mean()
    e_ref = np.linalg.norm(run["projPose2D"][:, :25] - inp["poses2D"][:, :25], axis=-1)[on].mean()
    assert e_mine <= 1.05 * e_ref
    # outputs are consistent: positions in body-25 order from the returned animation
    np.testing.assert_allclose(anim.global_positions()[:, ko.BACKWARD], new3d, atol=1e-9)


def test_floor_fit_path_prunes_and_converges(chd, data):
    ko = chd.kinopt
    inp = data["inp"]
    res = ko.optimize_trajectory(inp["poses2D"], inp["conf"], inp["poses3D"], inp["root_pos"], inp["joint_angles"], data["bvh"].parents,
                                 data["bvh"].offsets, inp["pp"][0], inp["pp"][1], inp["focal"], inp["vel"], max_nfev=15, ik_iterations=50)
    anim, new3d, proj, pn, pp, vel, info = res
    assert abs(np.linalg.norm(pn) - 1.0) < 1e-12 and pp[0] == 0.0 and pp[2] == 0.0
    assert set(np.unique(vel)) <= {0.0, 1.0} and (vel <= inp["vel"]).all()     # pruning only removes labels
    assert info["stage1"]["cost"] < 2309.5                                        # below the reference's stage-1 objective on this clip


def test_huber_fit_matches_sklearn(chd):
    sk = pytest.importorskip("sklearn.linear_model")
    rng = np.random.default_rng(3)
    X = rng.uniform(-100, 100, (80, 2))
    y = 0.05 * X[:, 0] - 0.02 * X[:, 1] + 90.0 + rng.normal(0, 0.8, 80)
    y[:9] += rng.uniform(8, 25, 9)
    for eps in (1.5, 2.2):
        ref = sk.HuberRegressor(epsilon=eps).fit(X, y)
        wv, c, s, out = chd.kinopt.huber_fit(X, y, eps)
        np.testing.assert_allclose(wv, ref.coef_, atol=2e-4)
        assert abs(c - ref.intercept_) < 2e-2 and abs(s - ref.scale_) < 2e-2
        np.testing.assert_array_equal(out, ref.outliers_)


def test_ik_initialisation_matches_reference(chd, data):
    ko, rs = chd.kinopt, chd.results
    inp, sk = data["inp"], data["sk"]
    g = np.load(os.path.join(G, "ik_init.npz"))
    F = data["F"]
    aa = -inp["joint_angles"]
    ang = np.linalg.norm(aa, axis=2)
    ax = aa / (ang + 1e-10)[..., None]
    K = np.zeros(aa.shape[:2] + (3, 3))
    K[..., 0, 1], K[..., 0, 2], K[..., 1, 0], K[..., 1, 2], K[..., 2, 0], K[..., 2, 1] = -ax[..., 2], ax[..., 1], ax[..., 2], -ax[..., 0], -ax[..., 1], ax[..., 0]
    R0 = np.eye(3) + np.sin(ang)[..., None, None] * K + (1 - np.cos(ang))[..., None, None] * (K @ K)
    P0 = np.tile(sk["offsets"][None], (F, 1, 1))
    P0[:, 0] = inp["root_pos"]
    anim = rs.SkelAnim(["j%d" % i for i in range(28)], data["bvh"].parents, sk["offsets"], R0, P0)
    tm = {j: sk["targets"][:, j] for j in range(28) if j not in ko.SPINE_IDX}
    out = rs.ik_solve(anim, tm, iterations=5, smoothness=0.0, damping=7.0, translate=False)
    q = g["rot_q"]
    w, x, y, z = [q[..., i] for i in range(4)]
    Rr = np.stack([np.stack([1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)], -1),
                   np.stack([2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)], -1),
                   np.stack([2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)], -1)], -2)
    np.testing.assert_allclose(out.rotations, Rr, atol=1e-8)
    np.testing.assert_allclose(out.positions, g["pos"], atol=1e-9)
