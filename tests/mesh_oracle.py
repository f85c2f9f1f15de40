"""fp64 restatement of the triangle-mesh ground's query (DESIGN.md section 4, "Triangle-mesh ground") by brute force
over ALL triangles, without the kernel's bucket grid: a bucket that misses a triangle shows up as a disagreement."""
import numpy as np


def face_normals(P):
    """(T, 3, 3) world vertices -> (T, 3) unit normals of (b - a) x (c - a) and (T,) |cross| (twice the area)."""
    n = np.cross(P[:, 1] - P[:, 0], P[:, 2] - P[:, 0])
    ln = np.linalg.norm(n, axis=1)
    return n / np.where(ln > 0, ln, 1.0)[:, None], ln


def closest_points(P, c):
    """Closest point of each triangle of P (T, 3, 3) to the point c (3,): Ericson's Voronoi-region test, vectorised."""
    a, b, cc = P[:, 0], P[:, 1], P[:, 2]
    ab, ac, ap = b - a, cc - a, c - a
    d1, d2 = (ab * ap).sum(1), (ac * ap).sum(1)
    bp = c - b
    d3, d4 = (ab * bp).sum(1), (ac * bp).sum(1)
    cp = c - cc
    d5, d6 = (ab * cp).sum(1), (ac * cp).sum(1)
    vc, vb, va = d1 * d4 - d3 * d2, d5 * d2 - d1 * d6, d3 * d6 - d5 * d4
    with np.errstate(divide="ignore", invalid="ignore"):
        den = va + vb + vc
        out = a + (vb / den)[:, None] * ab + (vc / den)[:, None] * ac
        e_bc = (d4 - d3 >= 0) & (d5 - d6 >= 0) & (va <= 0)
        w = (d4 - d3) / ((d4 - d3) + (d5 - d6))
        out = np.where(e_bc[:, None], b + w[:, None] * (cc - b), out)
        e_ac = (vb <= 0) & (d2 >= 0) & (d6 <= 0)
        out = np.where(e_ac[:, None], a + (d2 / (d2 - d6))[:, None] * ac, out)
        e_ab = (vc <= 0) & (d1 >= 0) & (d3 <= 0)
        out = np.where(e_ab[:, None], a + (d1 / (d1 - d3))[:, None] * ab, out)
    out = np.where(((d6 >= 0) & (d5 <= d6))[:, None], cc, out)
    out = np.where(((d3 >= 0) & (d4 <= d3))[:, None], b, out)
    out = np.where(((d1 <= 0) & (d2 <= 0))[:, None], a, out)
    return out


class MeshOracle:
    """The query of a sphere (centre c, radius r) against a mesh: nearest triangle (ties: lowest index), signed distance
    s, normal n, gap s - r; None farther than `margin` from every triangle."""

    def __init__(self, vertices, triangles, origin=(0.0, 0.0, 0.0), margin=0.2):
        P = np.asarray(vertices, np.float64)[np.asarray(triangles, np.int64)] + np.asarray(origin, np.float64)
        nf, ln = face_normals(P)
        keep = ln > 1e-12
        self.P, self.nf, self.dropped, self.margin = P[keep], nf[keep], int((~keep).sum()), margin

    def query(self, c):
        c = np.asarray(c, np.float64)
        p = closest_points(self.P, c)
        d2 = ((c - p) ** 2).sum(1)
        k = int(np.argmin(d2))  # (first minimum: the lowest index)
        d = np.sqrt(d2[k])
        if d > self.margin:
            return None
        sg = 1.0 if np.dot(c - p[k], self.nf[k]) >= 0 else -1.0
        n = self.nf[k] if d < 1e-6 else sg * (c - p[k]) / d
        # second-nearest distance: how far from a tie between two triangles the query is
        rest = np.delete(d2, k)
        gap = np.sqrt(rest.min()) - d if len(rest) else np.inf
        return dict(s=sg * d, n=n, tri=k, p=p[k], tie_gap=gap)


# ---------------------------------------------------------------- the physics oracle on a mesh ground

from oracle.physics_oracle import MAX_ACTIVE_PTS  # noqa: E402
from tests.terrain_oracle import TerrainOracle  # noqa: E402

D_ALLOWANCE = 0.1  # m, the depth allowance of the query margin


def mesh_tangents(n):
    """t1 = normalize(n_z, 0, -n_x), or normalize(0, n_z, -n_y) where n_x^2 + n_z^2 < 1e-6; t2 = n x t1."""
    q = n[:, 2] ** 2 + n[:, 0] ** 2
    wall = q < 1e-6
    t1 = np.where(wall[:, None], np.stack([np.zeros(len(n)), n[:, 2], -n[:, 1]], -1),
                  np.stack([n[:, 2], np.zeros(len(n)), -n[:, 0]], -1))
    t1 = t1 / np.linalg.norm(t1, axis=-1, keepdims=True)
    return t1, np.cross(n, t1)


class MeshPhysicsOracle(TerrainOracle):
    """TerrainOracle with a triangle mesh in place of the heightfield: the sole rows and the penalty contacts use the
    brute-force query of MeshOracle (every triangle, no grid); the rest of the sub-step is TerrainOracle's, line for
    line. The margin is contact_offset + the model's largest point radius + D, as the library forms it."""

    def __init__(self, tables, params, vertices, triangles, origin=(0.0, 0.0, 0.0), mu=None):
        super().__init__(tables, params)
        margin = float(np.float32(np.float32(params.contact_offset) + np.float32(np.max(tables.pt_radius)) +
                                  np.float32(D_ALLOWANCE)))
        self.mesh = MeshOracle(vertices, triangles, origin, margin)
        self.ground = self.mesh  # (not None: TerrainOracle.substep takes the ground path)
        if mu is not None:
            self.p.mu = mu

    def query_many(self, c):
        """(n, 3) centres -> s (n,), n (n, 3), hit (n,)."""
        n = len(c)
        s, nrm, hit = np.zeros(n), np.tile([0.0, 0.0, 1.0], (n, 1)), np.zeros(n, bool)
        for k in range(n):
            q = self.mesh.query(c[k])
            if q is not None:
                s[k], nrm[k], hit[k] = q["s"], q["n"], True
        return s, nrm, hit

    def _field_sole_row(self, Rw, pw, x, rad, cnt, body):
        p = self.p
        c = pw + np.einsum("nij,j->ni", Rw, x)
        s, n, hit = self.query_many(c)
        phi = s - rad
        act = hit & (phi < p.contact_offset) & (cnt < MAX_ACTIVE_PTS)
        t1, t2 = mesh_tangents(n)
        dirs_w = np.stack([n, t1, t2], 1)
        dirs = np.einsum("nji,ndj->ndi", Rw, dirs_w)
        xs = x[None, :] - rad * dirs[:, 0, :]
        Jr = np.concatenate([np.cross(xs[:, None, :], dirs), dirs], -1)
        bias = np.where(phi >= 0, -phi / p.dt, np.minimum(-p.erp * phi / p.dt, p.max_depen_vel))
        return Jr, bias, act, body, dirs_w

    def _external_wrench(self, i, Rw, pw, v, contact, par, push, rb_force, rb_torque):
        t, p = self.t, self.p
        N = Rw.shape[0]
        out = np.zeros((N, 6))

        def add_point_n(xs_l, n_w, depth, body):
            vel_w = np.einsum("nij,nj->ni", Rw, v[:, 3:] + np.cross(v[:, :3], xs_l))
            on = depth > 0
            vn = np.einsum("ni,ni->n", vel_w, n_w)
            fn = np.clip(p.pen_k * depth - p.pen_c * vn, 0.0, p.pen_fmax)
            vt = vel_w - vn[:, None] * n_w
            coef = np.minimum(p.pen_c, p.mu * fn / np.maximum(np.linalg.norm(vt, axis=-1), 1e-6))
            Fw = (fn[:, None] * n_w - coef[:, None] * vt) * on[:, None]
            contact[:, body, :] += Fw
            fl = np.einsum("nji,nj->ni", Rw, Fw)
            out[:, :3] += np.cross(xs_l, fl)
            out[:, 3:] += fl

        nrm_l = Rw[:, 2, :]
        for k in self.link_pts[i]:
            x, rad = t.pt_pos[k], t.pt_radius[k]
            c = pw + np.einsum("nij,j->ni", Rw, x)
            s, n, hit = self.query_many(c)
            add_point_n(x[None, :] - rad * np.einsum("nji,nj->ni", Rw, n), n, np.where(hit, rad - s, -1.0), int(t.pt_body[k]))
        for k in self.link_cyls[i]:
            c, a, (rad, hh) = t.cyl_center[k], t.cyl_axis[k], t.cyl_size[k]
            az = np.einsum("nj,j->n", nrm_l, a)
            sg = np.where(az >= 0, -1.0, 1.0)
            d_l = -(nrm_l - az[:, None] * a[None, :])
            dn = np.linalg.norm(d_l, axis=-1)
            rim = c[None, :] + (sg * hh)[:, None] * a[None, :] + np.where(dn[:, None] > 1e-6, rad * d_l / np.maximum(dn, 1e-30)[:, None], 0.0)
            q = pw + np.einsum("nij,nj->ni", Rw, rim)
            s, n, hit = self.query_many(q)
            add_point_n(rim, n, np.where(hit, -s, -1.0), int(t.cyl_body[k]))
        for b in self.link_bodies[i]:
            F = np.zeros((N, 3))
            Tq = np.zeros((N, 3))
            if push is not None and b == 0:
                F = F + push
            if rb_force is not None:
                F = F + rb_force[:, b, :]
            if rb_torque is not None:
                Tq = Tq + rb_torque[:, b, :]
            if push is None and rb_force is None and rb_torque is None:
                continue
            com = par[:, b, 1:4] / np.maximum(par[:, b, 0:1], 1e-30)
            fl = np.einsum("nji,nj->ni", Rw, F)
            out[:, :3] += np.cross(com, fl) + np.einsum("nji,nj->ni", Rw, Tq)
            out[:, 3:] += fl
        return out
