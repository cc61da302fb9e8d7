"""Float64 numpy restatement of the photometric + depth solver (PHOVO_MODE_BIOBJECTIVE).

TEST INFRASTRUCTURE.  The reference solver is CPhotoconsistencyOdometryBiObjective.h (BI:242-452 for one pass,
BI:567-579 for the target depth).  The C oracle has no such mode, so this module restates it on its own:

* Level images.  I0, D0, I1, Gx and Gy come from the C oracle (bit-pinned against OpenCV).  D1 is the target depth
  resized like D0, GxD / GyD are the Scharr derivatives of D1 / max_depth with the level's gradient scale, and the
  gain is mean(I1) / mean(D1) over every pixel of the level, zeros included.
* Validity.  The analytic rule (AN:279-303): strict depth bounds, round half away from zero, inside the image, no
  Z > 0 test.
* Residual slots.  Source pixel i, in raster order, writes slot t(i) with I1[t] - I0[i] and then slot 2 t(i) with
  gain (D1[t] - D0[i]); later writes win, so a slot holds the write with the largest key 2 i + 1 (intensity) or
  2 i + 2 (depth).
* Jacobian rows.  Pixel i writes row i (intensity) and then row 2 i (depth), later writes win.  A row is the
  reference's factored product [gx gy] . Jproj (2x3) . JRt (3x6), a depth row gain ([gxD gyD] . Jproj . JRt - JRt[2,:]),
  not the closed form the kernels use.

No cv2 and no Python loop over pixels: one evaluation at 640x480 takes well under a second.
"""
import numpy as np

import oracle_py

# variants of the two aliasing rules, for the negative tests that show the fixtures can tell the rules apart
RULES = ("reference", "no_row0_rule", "swapped_keys")


def depth_metres(depth, depth_scale=1.0):
    """A caller's depth frame in metres as the library reads it: u16 raw * depth_scale, f32 widened, f64 as given."""
    d = np.asarray(depth)
    if d.dtype == np.uint16:
        return d.astype(np.float64) * float(depth_scale)
    return d.astype(np.float64)


def _cfg_values(cfg):
    n = int(cfg.num_levels)
    return dict(num_levels=n, max_iters=[int(cfg.max_num_iterations[l]) for l in range(n)],
                lam=[float(cfg.lambda_step[l]) for l in range(n)], min_grad=[float(cfg.min_gradient_norm[l]) for l in range(n)],
                grad_scale=[float(cfg.grad_scale[l]) for l in range(n)], min_depth=float(cfg.min_depth), max_depth=float(cfg.max_depth))


class BiLevels:
    """The level images of one pair.  `cfg` is a Config of the library or of the oracle (same layout)."""

    def __init__(self, cfg, K, gray0, depth0, gray1, depth1, depth_scale=1.0, levels=None):
        self.cfg = _cfg_values(cfg)
        self.K = np.asarray(K, dtype=np.float64).reshape(3, 3)
        ocfg = oracle_py.Config.from_buffer_copy(bytes(cfg))
        ocfg.mode = 0                                            # the oracle builds the same pyramids in mode 0
        o = oracle_py.Oracle(ocfg, self.K)
        o.set_source(gray0, depth_metres(depth0, depth_scale))
        o.set_target(gray1)
        d1 = depth_metres(depth1, depth_scale)
        if levels is None:
            levels = [l for l in range(self.cfg["num_levels"]) if self.cfg["max_iters"][l] > 0]
        self.levels = {}
        inv_max = 1.0 / self.cfg["max_depth"]
        for l in levels:
            I0, D0, I1, Gx, Gy = (o.level_image(w, l) for w in range(5))
            D1 = oracle_py.resize_level(d1, l)
            assert D1.shape == I0.shape
            Ds = D1 * inv_max
            gs = self.cfg["grad_scale"][l]
            with np.errstate(all="ignore"):
                gain = I1.mean() / D1.mean()
            self.levels[l] = dict(I0=I0, D0=D0, I1=I1, Gx=Gx, Gy=Gy, D1=D1, GxD=oracle_py.scharr(Ds, 1, 0, gs),
                                  GyD=oracle_py.scharr(Ds, 0, 1, gs), gain=gain,
                                  min_depth=self.cfg["min_depth"], max_depth=self.cfg["max_depth"])


def rotation_and_derivatives(state):
    """eigenPose's R = Rz(yaw) Ry(pitch) Rx(roll) (CPhotoconsistencyOdometry.h:47-71) and dR / d(yaw, pitch, roll)."""
    yaw, pitch, roll = (float(v) for v in state[3:6])
    cz, sz, cy, sy, cx, sx = np.cos(yaw), np.sin(yaw), np.cos(pitch), np.sin(pitch), np.cos(roll), np.sin(roll)
    Rz = np.array([[cz, -sz, 0.], [sz, cz, 0.], [0., 0., 1.]])
    Ry = np.array([[cy, 0., sy], [0., 1., 0.], [-sy, 0., cy]])
    Rx = np.array([[1., 0., 0.], [0., cx, -sx], [0., sx, cx]])
    dRz = np.array([[-sz, -cz, 0.], [cz, -sz, 0.], [0., 0., 0.]])
    dRy = np.array([[-sy, 0., cy], [0., 0., 0.], [-cy, 0., -sy]])
    dRx = np.array([[0., 0., 0.], [0., -sx, -cx], [0., cx, -sx]])
    R = np.array([[cz * cy, cz * sy * sx - sz * cx, cz * sy * cx + sz * sx],     # eigenPose's own expressions
                  [sz * cy, sz * sy * sx + cz * cx, sz * sy * cx - cz * sx],
                  [-sy, cy * sx, cy * cx]])
    return R, (dRz @ Ry @ Rx, Rz @ dRy @ Rx, Rz @ Ry @ dRx)


def round_half_away(v):
    return np.sign(v) * np.floor(np.abs(v) + 0.5)


def pack_upper(H):
    iu = np.triu_indices(6)
    return H[iu]


def evaluate(lv, K, level, state, rules="reference"):
    """One pass of BI:242-452 at `state` on the level images `lv` (a BiLevels.levels entry, which also carries the
    configuration's depth bounds).  Returns a dict:
    H (6x6), g (6), num_valid (valid source pixels), cost = 0.5 |res|^2, res (2N), J (2N x 6), keys (2N: the winning
    write key of each residual slot, 0 for none), row_owner (2N: 2 i for pixel i's intensity row, 2 i + 1 for its depth
    row, -1 for a zero row), valid (N) and target (N: the slot t(i) of each valid pixel, -1 for the others).
    `rules` other than "reference" change one aliasing rule on purpose (see RULES)."""
    assert rules in RULES
    state = np.asarray(state, dtype=np.float64)
    I0 = lv["I0"]
    rows, cols = I0.shape
    N = rows * cols
    p2 = 2.0 ** level
    fx, fy, ox, oy = K[0, 0] / p2, K[1, 1] / p2, K[0, 2] / p2, K[1, 2] / p2
    inv_fx, inv_fy = 1. / fx, 1. / fy
    R, dR = rotation_and_derivatives(state)
    c, r = np.meshgrid(np.arange(cols, dtype=np.float64), np.arange(rows, dtype=np.float64))
    d, c, r = lv["D0"].ravel(), c.ravel(), r.ravel()
    min_depth, max_depth = lv["min_depth"], lv["max_depth"]
    # warp in the reference's operation order (AN:279-303)
    px = ((c - ox) * d) * inv_fx
    py = ((r - oy) * d) * inv_fy
    P = np.stack([px, py, d])
    q = [(R[a, 0] * px + R[a, 1] * py) + R[a, 2] * d for a in range(3)]
    X, Y, Z = q[0] + state[0], q[1] + state[1], q[2] + state[2]
    with np.errstate(all="ignore"):
        iz = 1. / Z
        tc = (X * fx) * iz + ox
        tr = (Y * fy) * iz + oy
        ti, tj = round_half_away(tr), round_half_away(tc)
        valid = (min_depth < d) & (d < max_depth) & (ti >= 0) & (ti < rows) & (tj >= 0) & (tj < cols)
    i = np.flatnonzero(valid)
    t = (ti[i] * cols + tj[i]).astype(np.int64)
    target = np.full(N, -1, np.int64)
    target[i] = t
    # residual slots: the write with the largest key wins
    ki, kd = (2 * i + 2, 2 * i + 1) if rules == "swapped_keys" else (2 * i + 1, 2 * i + 2)
    keys = np.zeros(2 * N, np.int64)
    np.maximum.at(keys, np.concatenate([t, 2 * t]), np.concatenate([ki, kd]))
    gain = lv["gain"]
    res = np.zeros(2 * N)
    k = np.flatnonzero(keys)
    src = (keys[k] - 1) >> 1
    is_depth = ((keys[k] - 1) & 1) == 1
    if rules == "swapped_keys":
        is_depth = ~is_depth
    ks, kd_ = k[~is_depth], k[is_depth]
    res[ks] = lv["I1"].ravel()[ks] - I0.ravel()[src[~is_depth]]
    with np.errstate(all="ignore"):
        res[kd_] = gain * (lv["D1"].ravel()[kd_ >> 1] - d[src[is_depth]])
    # factored Jacobian of the valid pixels: JRt (3x6), Jproj (2x3), gradient (1x2)
    m = len(i)
    JRt = np.zeros((m, 3, 6))
    JRt[:, 0, 0] = JRt[:, 1, 1] = JRt[:, 2, 2] = 1.
    for a in range(3):
        JRt[:, :, 3 + a] = (dR[a] @ P[:, i]).T
    Jp = np.zeros((m, 2, 3))
    with np.errstate(all="ignore"):
        Jp[:, 0, 0] = fx / Z[i]
        Jp[:, 1, 1] = fy / Z[i]
        Jp[:, 0, 2] = -fx * X[i] / Z[i] ** 2
        Jp[:, 1, 2] = -fy * Y[i] / Z[i] ** 2

        def rows_of(gx, gy):
            v = gx.ravel()[i, None] * Jp[:, 0, :] + gy.ravel()[i, None] * Jp[:, 1, :]      # [gx gy] . Jproj
            return np.einsum("nb,nbc->nc", v, JRt)
        JI = rows_of(lv["Gx"], lv["Gy"])
        JD = gain * (rows_of(lv["GxD"], lv["GyD"]) - JRt[:, 2, :])
    # rows in raster write order: pixel i writes row i (time 2 i), then row 2 i (time 2 i + 1); the last write wins
    owner = np.full(2 * N, -1, np.int64)
    np.maximum.at(owner, np.concatenate([i, 2 * i]), np.concatenate([2 * i, 2 * i + 1]))
    if rules == "no_row0_rule" and m and i[0] == 0:
        owner[0] = 0                                           # pixel 0's intensity row instead of its depth row
    pos = np.full(N, -1, np.int64)
    pos[i] = np.arange(m)
    J = np.zeros((2 * N, 6))
    kk = np.flatnonzero(owner >= 0)
    w = owner[kk]
    pix, dep = pos[w >> 1], (w & 1) == 1
    J[kk[~dep]] = JI[pix[~dep]]
    J[kk[dep]] = JD[pix[dep]]
    with np.errstate(all="ignore"):
        H = J.T @ J
        g = J.T @ res
        cost = 0.5 * (res @ res)
    return dict(H=H, g=g, num_valid=int(m), cost=float(cost), res=res, J=J, keys=keys, row_owner=owner, valid=valid,
                target=target)


def optimize(levels, state0, rules="reference"):
    """The Gauss-Newton loop of AN:500-563 / AN:376-392 with the per-level lambda, coarse to fine.  Returns the final
    state and a log with the library's fields (H packed upper-triangular, like IterationStats)."""
    cfg, K = levels.cfg, levels.K
    s = np.array(state0, dtype=np.float64).reshape(6)
    log = []
    for level in range(cfg["num_levels"] - 1, -1, -1):
        M = cfg["max_iters"][level]
        for it in range(M):
            e = evaluate(levels.levels[level], K, level, s, rules)
            with np.errstate(all="ignore"):
                try:
                    step = np.linalg.solve(e["H"], e["g"]) if np.isfinite(e["H"]).all() else np.full(6, np.nan)
                except np.linalg.LinAlgError:
                    step = np.full(6, np.nan)
                s_out = s - cfg["lam"][level] * step
                gn = float(np.sqrt(e["g"] @ e["g"]))
            log.append(dict(level=level, iteration=it, num_valid=e["num_valid"], H=pack_upper(e["H"]), g=e["g"], cost=e["cost"],
                            grad_norm=gn, state_in=s.copy(), state_out=s_out.copy()))
            s = s_out
            if gn < cfg["min_grad"][level]:                        # AN:383-392 (NaN compares false)
                break
    return s, log
