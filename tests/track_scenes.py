"""TEST INFRASTRUCTURE: scenes for rigid point-to-TSDF tracking (tests/test_track_host.py, tests/test_gpu_track.py).

The body mesh of synth.make_scene seen from cameras on a ring, in a world whose origin is the volume's centre (scale 1,
center 0: world = grid - R/2), fused by the oracle (oracle/tsdf.py:fuse_depth_rigid) and rendered by synth.render_depth."""
import numpy as np

from dynamicfusion_body_b200 import synth


class Ring:
    def __init__(self, res=64, rows=480, cols=640, tdist=3.0, seed=0):
        self.sc = synth.make_scene(res=res, k=4, n_nodes=300, seed=seed, n_views=1, rows=rows, cols=cols)
        self.res, self.rows, self.cols, self.tdist = res, rows, cols, float(tdist)
        self.K, self.Kinv = self.sc.K, self.sc.Kinv
        self.verts = self.sc.vertices.astype(np.float64) - res / 2.0
        self.target = np.full(3, (res - 1) / 2.0) - res / 2.0
        self.scale, self.center = 1.0, np.zeros(3)

    def pose(self, deg, dist=1.7):
        """World -> camera 3x4 of the ring camera at `deg` degrees, `dist` volume widths from the body."""
        a = np.deg2rad(deg)
        return synth.look_at_extrinsic(self.target + dist * self.res * np.array([np.sin(a), 0.1, -np.cos(a)]), self.target)

    def frame(self, lw):
        lw = np.asarray(lw, dtype=np.float64)
        return synth.render_depth(self.verts @ lw[:, :3].T + lw[:, 3], self.sc.faces, self.K, self.rows, self.cols)

    def fuse_oracle(self, poses):
        """(tsdf, weight) float32 (R,R,R) fused by the oracle from the frames of `poses`, in float32 storage between frames."""
        from oracle import tsdf as ot
        R = self.res
        vox = ot.voxel_grid((R, R, R))
        T = np.full(R ** 3, self.tdist)
        W = np.zeros(R ** 3)
        for lw in poses:
            T, W, _, _ = ot.fuse_depth_rigid(T, W, vox, self.frame(lw), lw, self.K, self.Kinv, self.tdist, R, self.scale, self.center)
            T, W = T.astype(np.float32).astype(np.float64), W.astype(np.float32).astype(np.float64)
        return T.reshape(R, R, R).astype(np.float32), W.reshape(R, R, R).astype(np.float32)


def perturb(lw, deg, trans, seed):
    """The pose whose camera is turned by `deg` degrees about a seeded axis through its own centre and moved by `trans`
    (world units) along a seeded direction."""
    from dynamicfusion_body_b200 import engine
    rng = np.random.default_rng(seed)
    ax = rng.normal(size=3)
    d = rng.normal(size=3)
    dR, _ = engine.se3_exp(np.concatenate([np.zeros(3), np.deg2rad(deg) * ax / np.linalg.norm(ax)]))
    lw = np.asarray(lw, dtype=np.float64)
    Rc, C = lw[:, :3].T, -lw[:, :3].T @ lw[:, 3]
    Rn, Cn = dR @ Rc, C + trans * d / np.linalg.norm(d)
    return np.concatenate([Rn.T, (-Rn.T @ Cn)[:, None]], 1)


def pose_error(lw, truth):
    """(rotation error in degrees, camera-centre error in world units)."""
    lw, truth = np.asarray(lw, dtype=np.float64), np.asarray(truth, dtype=np.float64)
    dR = lw[:, :3] @ truth[:, :3].T
    ang = float(np.degrees(np.arccos(np.clip((np.trace(dR) - 1.0) / 2.0, -1.0, 1.0))))
    return ang, float(np.linalg.norm(lw[:, :3].T @ lw[:, 3] - truth[:, :3].T @ truth[:, 3]))
