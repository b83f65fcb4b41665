"""Restatement of the voxel-grid SDF (include/kin_b200.h, KinGrid) in double arithmetic on the float32 samples, written
out per point in the order the header states, for the tests to compare the device against.  Every fused multiply-add
the header names is rounded once here too (exact rational arithmetic, then one correctly rounded conversion), so a point
on a cell face falls into the same cell as on the device.  Members of a union that are not grids are evaluated by the C
oracle (oracle/ref_model.py: RefSDF), one row at a time."""
from fractions import Fraction

import numpy as np

from oracle import ref_model as R

EPS = 1e-7


def _fma(a, b, c):
    return float(Fraction(float(a)) * Fraction(float(b)) + Fraction(float(c)))


def _lerp(a, b, t):
    return _fma(t, float(b) - float(a), a)


class RefGrid:
    """values: (nx, ny, nz) indexed [i, j, k]; stored as float32 like kin_grid_create; pose: 4x4 world pose."""

    def __init__(self, values, spacing, pose=None):
        self.v = np.asarray(values, dtype=np.float32)
        self.n = np.array(self.v.shape)
        self.s = float(spacing)
        self.pose = np.eye(4) if pose is None else np.asarray(pose, dtype=np.float64)
        Rm, t = self.pose[:3, :3], self.pose[:3, 3]
        self.inv_R = Rm.T.copy()                   # inv(tf) = (-R' t, R') as the library forms it (transform.jl:62-65)
        self.inv_t = np.array([(-Rm[0, r]) * t[0] + (-Rm[1, r]) * t[1] + (-Rm[2, r]) * t[2] for r in range(3)])

    def local(self, p):
        p = np.asarray(p, dtype=np.float64)
        r = self.inv_R
        return np.array([_fma(r[k, 0], p[0], _fma(r[k, 1], p[1], _fma(r[k, 2], p[2], self.inv_t[k]))) for k in range(3)])

    def eval_local(self, l):
        """-> (d, local gradient of d)."""
        inv_s = 1.0 / self.s
        top = (self.n - 1).astype(np.float64)
        u = np.array([_fma(l[k], inv_s, 0.5 * top[k]) for k in range(3)])
        c = np.minimum(np.maximum(u, 0.0), top)
        i0 = np.minimum(np.floor(c).astype(np.int64), self.n - 2)
        t = c - i0
        e = u - c
        V = self.v[i0[0]:i0[0] + 2, i0[1]:i0[1] + 2, i0[2]:i0[2] + 2].astype(np.float64)   # V[di, dj, dk]
        a00, a10 = _lerp(V[0, 0, 0], V[1, 0, 0], t[0]), _lerp(V[0, 1, 0], V[1, 1, 0], t[0])
        a01, a11 = _lerp(V[0, 0, 1], V[1, 0, 1], t[0]), _lerp(V[0, 1, 1], V[1, 1, 1], t[0])
        b0, b1 = _lerp(a00, a10, t[1]), _lerp(a01, a11, t[1])
        f = _lerp(b0, b1, t[2])
        o = np.sqrt(_fma(e[0], e[0], _fma(e[1], e[1], e[2] * e[2])))
        df = np.array([_lerp(_lerp(V[1, 0, 0] - V[0, 0, 0], V[1, 1, 0] - V[0, 1, 0], t[1]),
                             _lerp(V[1, 0, 1] - V[0, 0, 1], V[1, 1, 1] - V[0, 1, 1], t[1]), t[2]),
                       _lerp(a10 - a00, a11 - a01, t[2]),
                       b1 - b0])
        gl = np.where(e != 0.0, e / (o if o > 0 else 1.0), df * inv_s)
        return _fma(self.s, o, f), gl

    def __call__(self, p):
        return self.eval_local(self.local(p))[0]

    def gradient(self, p, analytic=False, f=None):
        if analytic:
            return self.pose[:3, :3] @ self.eval_local(self.local(p))[1]
        f = self(p) if f is None else f
        p = np.asarray(p, dtype=np.float64)
        return np.array([(self(p + EPS * np.eye(3)[i]) - f) / EPS for i in range(3)])

    def sample_points(self):
        """World positions of the samples, (nx, ny, nz, 3)."""
        ax = [(np.arange(n) - (n - 1) / 2.0) * self.s for n in self.n]
        L = np.stack(np.meshgrid(*ax, indexing="ij"), axis=-1)
        return L @ self.pose[:3, :3].T + self.pose[:3, 3]


class RefScene:
    """A union of grid rows (RefGrid) and oracle rows (poses, sizes, kinds of oracle.ref_model.RefSDF), first-minimum
    argmin in table order."""

    def __init__(self, rows):
        self.rows = [r if isinstance(r, RefGrid) else R.RefSDF([r[0]], [r[1]], [r[2]]) for r in rows]

    def eval(self, p, grad_mode=None):
        """-> (d, 1-based argmin, gradient on the argmin row or None); grad_mode 0/2 = FD, 1 = analytic."""
        vals = [float(r(p)) for r in self.rows]
        k = int(np.argmin(vals))                       # first minimum
        d = vals[k]
        if grad_mode is None:
            return d, k + 1, None
        row = self.rows[k]
        if isinstance(row, RefGrid):
            g = row.gradient(p, analytic=grad_mode == 1, f=d)
        else:
            row(p)
            g = row.gradient(p, analytic=grad_mode == 1)
        return d, k + 1, g
