"""Golden vectors for the kinematic optimiser (`src/optimize/optimize_trajectory.py`), produced by the REFERENCE'S OWN code
imported from /root/reference with the shims of make_towr_golden.py (numpy 2 aliases, plotting stubs).  Build container
only.  Writes tests/golden/kinopt/:

  inputs.npz      synthetic clip: 2D keypoints + confidences, root-relative 3D joints, root translation, initial joint
                  angles (axis-angle, SMPL-style), contact labels; the skeleton is tests/golden/kinopt/skeleton.bvh
  skeleton.npz    update_skeleton(...) of the reference: fitted offsets
  funjac.npz      fun_anim_for_projection of the reference at two points x_a, x_b (stage weights without and with the
                  floor term), with the weights and floor plane it was evaluated with
  jac_a.npz,      jac_anim_for_projection_sparse of the reference at x_a resp. x_b, stored as CSR matrices
  jac_b.npz       (scipy.sparse.save_npz: about 1 % of the entries are non-zero)
  run.npz         the reference's full optimize_trajectory(...) output on the clip: final x is not exposed by the
                  reference, so: final joint positions, re-projected 2D points, floor normal / point, refined contact labels,
                  and the objective 0.5 |f|^2 of the returned animation under the final-stage weights
"""
import os
import sys

import numpy as np
import scipy.sparse as sp

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
from make_towr_golden import ROOT, combined_skeleton, import_reference  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "kinopt")
F = 14


def synth_clip(chd, seed=0):
    """A short walking-like clip seen by the MTC camera (focal 2000 px, 1920x1080, y down, z forward, cm)."""
    from chd import prepare, results
    rng = np.random.default_rng(seed)
    names, parents, off, key = combined_skeleton()
    J = len(names)
    t = np.arange(F) / 30.0
    e = np.zeros((F, J, 3))                                   # Euler x, y, z (R = Rz Ry Rx), radians
    e[:, 0] = np.stack([0.05 * np.sin(5 * t), 0.3 + 0.2 * t, 0.04 * np.cos(4 * t)], 1)
    sw = 0.45 * np.sin(2 * np.pi * 0.9 * t)
    e[:, key["l_hip"], 0], e[:, key["r_hip"], 0] = sw, -sw
    e[:, key["l_knee"], 0], e[:, key["r_knee"], 0] = 0.35 + 0.3 * np.cos(2 * np.pi * 0.9 * t), 0.35 - 0.3 * np.cos(2 * np.pi * 0.9 * t)
    e[:, key["l_sh"], 0], e[:, key["r_sh"], 0] = -0.3 * np.sin(2 * np.pi * 0.9 * t), 0.3 * np.sin(2 * np.pi * 0.9 * t)
    e += np.cumsum(rng.normal(0, 0.01, e.shape), axis=0)
    root = np.stack([20.0 + 60.0 * t, 15.0 + 1.5 * np.sin(2 * np.pi * 1.8 * t), 380.0 + 40.0 * t], axis=1)
    R = results.rot_zyx(e)
    T = np.tile(np.asarray(off, dtype=np.float64)[None], (F, 1, 1))
    T[:, 0] = 0.0
    gp, _ = prepare.forward_kinematics(np.array(parents), R, T)                 # root-relative positions, skeleton order
    return names, parents, off, e, root, gp


def main():
    tu = import_reference()
    import chd
    from chd import prepare, results
    import optimize_trajectory as ot
    import BVH
    os.makedirs(OUT, exist_ok=True)
    rng = np.random.default_rng(42)
    names, parents, off, e_true, root_true, gp = synth_clip(chd)
    J = len(names)
    skel_path = os.path.join(OUT, "skeleton.bvh")
    prepare.write_bvh(skel_path, names, parents, off, np.zeros((1, 3 + 3 * J)), 1.0 / 30.0, order="ZXY")
    BACK = ot.BACKWARD_MAPPING
    poses3D = np.stack([gp[:, BACK[j]] for j in range(J)], axis=1) * (1.0 + 0.03 * rng.normal(size=(1, J, 1))) + rng.normal(0, 0.8, (F, J, 3))
    poses3D[:, ot.ROOT_IDX] = 0.0
    root_pos = root_true + rng.normal(0, 1.0, (F, 3))
    focal, pp = np.array([2000.0, 2000.0]), np.array([960.0, 540.0])
    absj = np.stack([gp[:, BACK[j]] for j in range(J)], axis=1) + root_true[:, None]
    poses2D = absj[:, :, :2] / absj[:, :, 2:3] * focal + pp + rng.normal(0, 1.5, (F, J, 2))
    conf = rng.uniform(0.3, 1.0, (F, J))
    conf[rng.uniform(size=(F, J)) < 0.05] = 0.0
    poses2D[:, 25:], conf[:, 25:] = 0.0, 0.0
    # initial joint angles: axis-angle of the true local rotations (the reference negates the axis), noisy
    Rl = results.rot_zyx(e_true)
    ang = np.arccos(np.clip((np.trace(Rl, axis1=-2, axis2=-1) - 1.0) / 2.0, -1.0, 1.0))
    ax = np.stack([Rl[..., 2, 1] - Rl[..., 1, 2], Rl[..., 0, 2] - Rl[..., 2, 0], Rl[..., 1, 0] - Rl[..., 0, 1]], -1)
    ax = ax / (np.linalg.norm(ax, axis=-1, keepdims=True) + 1e-12)
    joint_angles = -(ax * ang[..., None]) + rng.normal(0, 0.03, (F, J, 3))
    # contacts (body-25 order): left foot planted in the first half, right foot in the second; one spurious label
    vel = np.zeros((F, J))
    vel[:F // 2, [19, 20, 21]] = 1
    vel[F // 2:, [22, 23, 24]] = 1
    vel[2, 22] = 1
    np.savez(os.path.join(OUT, "inputs.npz"), poses2D=poses2D, conf=conf, poses3D=poses3D, root_pos=root_pos, joint_angles=joint_angles,
             vel=vel, focal=focal, pp=pp)

    skeleton, bnames, _ = BVH.load(skel_path)
    targets = np.stack([poses3D[:, ot.FORWARD_MAPPING[j]] for j in range(J)], axis=1) + root_pos[:, None]
    sk = ot.update_skeleton(skeleton, targets, bnames)
    np.savez(os.path.join(OUT, "skeleton.npz"), offsets=sk.offsets, targets=targets)

    # the initialisation IK of optimize_trajectory.py:566-617 (rotations only, 5 of its 200 iterations)
    from Quaternions import Quaternions
    from InverseKinematics import JacobianInverseKinematicsCK
    anim = sk.copy()
    anim.orients.qs = sk.orients.qs.copy()
    anim.offsets = sk.offsets.copy()
    anim.positions = sk.positions.repeat(F, axis=0)
    anim.positions[:, 0] = root_pos
    ang0 = np.linalg.norm(joint_angles, axis=2)
    anim.rotations = Quaternions.from_angle_axis(ang0, -joint_angles / (ang0 + 1e-10)[..., None])
    tm = {j: targets[:, j] for j in range(J) if j not in ot.SKEL_SPINE_IDX}
    JacobianInverseKinematicsCK(anim, tm, translate=False, iterations=5, smoothness=0.0, damping=7, silent=True)()
    np.savez(os.path.join(OUT, "ik_init.npz"), rot_q=anim.rotations.qs, pos=anim.positions)

    # residual / Jacobian of the reference at two points
    pw = np.ones((F, J)) * conf * ot.PROJ_WEIGHTS
    pw[:, 25:] = 0
    dw = (1.0 + conf) * ot.DATA_WEIGHTS
    dw[:, 25:] = (1.0 + 0.4) * ot.DATA_WEIGHTS[25:]
    j2n = poses2D.copy()
    j2n[:, :25] = (poses2D[:, :25] - pp) / focal
    normal = np.array([0.03, -1.0, 0.02])
    normal /= np.linalg.norm(normal)
    point = np.array([0.0, 95.0, 400.0])
    fj = {}
    for tag, fw, sd in (("a", 0.0, 1), ("b", 10.0, 2)):
        r2 = np.random.default_rng(sd)
        x = np.concatenate([root_pos + r2.normal(0, 2, (F, 3)), (e_true + r2.normal(0, 0.05, e_true.shape)).reshape(F, -1)], axis=1).reshape(-1)
        args = (sk, poses3D, root_pos, j2n, normal, point, pw, dw, np.arange(J), np.arange(J), ot.SMOOTH_WEIGHTS, vel, 1000.0, 0.1, 0.5, 0.3, 10.0, fw)
        fj["x_" + tag] = x
        fj["f_" + tag] = ot.fun_anim_for_projection(x, *args)
        jac = sp.csr_matrix(ot.jac_anim_for_projection_sparse(x, *args))
        jac.eliminate_zeros()
        sp.save_npz(os.path.join(OUT, "jac_%s.npz" % tag), jac)
    np.savez_compressed(os.path.join(OUT, "funjac.npz"), normal=normal, point=point, pw=pw, dw=dw, j2n=j2n, **fj)

    # the full run
    import time
    t0 = time.time()
    skeleton, bnames, _ = BVH.load(skel_path)
    anim, newPose3D, projPose2D, pn, ppnt, newvel = ot.optimize_trajectory(poses2D.copy(), conf.copy(), poses3D.copy(), root_pos.copy(), joint_angles.copy(),
                                                                           skeleton, bnames, pp[0], pp[1], focal, vel.copy(), save_dir=OUT)
    dt = time.time() - t0
    import Animation
    x_fin = np.concatenate([anim.positions[:, 0], anim.rotations.euler().reshape(F, -1)], axis=1).reshape(-1)
    sk2 = ot.update_skeleton(BVH.load(skel_path)[0], targets, bnames)
    args = (sk2, poses3D, root_pos, j2n, pn, ppnt, pw, dw, np.arange(J), np.arange(J), ot.SMOOTH_WEIGHTS, newvel, 1000.0, 0.1, 0.5, 0.3, 10.0, 10.0)
    cost = 0.5 * float(np.sum(ot.fun_anim_for_projection(x_fin, *args) ** 2))
    np.savez(os.path.join(OUT, "run.npz"), newPose3D=newPose3D, projPose2D=projPose2D, plane_normal=pn, plane_point=ppnt, newvel=newvel,
             x_fin=x_fin, cost=cost, gpos=Animation.positions_global(anim), seconds=dt)
    os.remove(os.path.join(OUT, "final_test.bvh"))
    print("reference optimize_trajectory: %.1f s, final cost %.6g" % (dt, cost))


if __name__ == "__main__":
    main()
