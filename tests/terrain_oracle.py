"""TEST INFRASTRUCTURE ONLY -- the fp64 physics oracle (oracle/physics_oracle.py) on a heightfield ground.

TerrainOracle is PhysicsOracle with an optional `ground`: without one it IS the plane oracle (every call goes to the
parent class); with a HeightField the sub-step below replaces the plane z = 0 by the field in the two places the
ground enters -- the sole rows of the constraint-solved contact and the penalty contact of every other candidate --
and is otherwise the parent's sub-step line for line. The field's height / normal query is written here separately
from the kernel's (physics_roles.cuh field_query): the plane through the triangle's three vertices instead of the
kernel's per-triangle gradients. The ground model is stated in DESIGN.md section 4.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

from oracle.physics_oracle import MAX_ACTIVE_PTS, PhysicsOracle, PhysParams, crf_apply, crm_apply


@dataclass
class HeightField:
    """Heightfield ground (DESIGN.md section 4): vertex (i, j) at origin + (i row_scale, j column_scale,
    vertical_scale samples[i, j]); row i along x, column j along y; each cell split along its diagonal
    (i, j)-(i+1, j+1); no ground outside the field's x-y rectangle."""
    samples: np.ndarray
    row_scale: float
    column_scale: float
    vertical_scale: float
    origin: tuple = (0.0, 0.0, 0.0)

    def query(self, x, y):
        """Height (N,), unit upward normal (N, 3) and inside mask (N,) at world points (x, y), from the plane through the
        three vertices of the triangle that holds the point. The cell is (floor u, floor v) of the grid coordinates
        u, v (the last vertex row / column belongs to the cell before it); a point with fu >= fv takes the triangle
        (i, j), (i+1, j), (i+1, j+1), any other (i, j), (i+1, j+1), (i, j+1)."""
        s = np.asarray(self.samples, np.float64)
        nr, nc = s.shape
        ox, oy, oz = (float(c) for c in self.origin)
        u = (np.asarray(x, np.float64) - ox) / self.row_scale
        v = (np.asarray(y, np.float64) - oy) / self.column_scale
        inside = (u >= 0) & (v >= 0) & (u <= nr - 1) & (v <= nc - 1)
        uc, vc = np.where(inside, u, 0.0), np.where(inside, v, 0.0)
        i = np.minimum(np.floor(uc).astype(int), nr - 2)
        j = np.minimum(np.floor(vc).astype(int), nc - 2)
        lower = (uc - i) >= (vc - j)

        def vert(a, b):
            return np.stack([ox + a * self.row_scale, oy + b * self.column_scale, oz + self.vertical_scale * s[a, b]], -1)

        p0 = vert(i, j)
        p1 = np.where(lower[:, None], vert(i + 1, j), vert(i + 1, j + 1))
        p2 = np.where(lower[:, None], vert(i + 1, j + 1), vert(i, j + 1))
        n = np.cross(p1 - p0, p2 - p0)
        n = n / np.linalg.norm(n, axis=-1, keepdims=True)
        xw = np.stack([ox + uc * self.row_scale, oy + vc * self.column_scale], -1)
        h = p0[:, 2] - (n[:, 0] * (xw[:, 0] - p0[:, 0]) + n[:, 1] * (xw[:, 1] - p0[:, 1])) / n[:, 2]
        return h, n, inside


def tangents(n):
    """Row directions of a ground contact with unit normal n (N, 3): t1 = normalize(n_z, 0, -n_x), t2 = n x t1."""
    t1 = np.stack([n[:, 2], np.zeros(len(n)), -n[:, 0]], -1)
    t1 = t1 / np.linalg.norm(t1, axis=-1, keepdims=True)
    return t1, np.cross(n, t1)


class TerrainOracle(PhysicsOracle):
    def __init__(self, tables, params: PhysParams = None, solver_bodies=("L_Foot_Link", "R_Foot_Link"),
                 ground: HeightField = None):
        """ground: None = the plane z = 0 with normal +z (PhysicsOracle itself); or a HeightField."""
        super().__init__(tables, params, solver_bodies)
        self.ground = ground

    # ------------------------------------------------------------------ one sub-step
    def substep(self, root, q, qd, tau, damping, armature, mass_scale, push=None, rb_force=None, rb_torque=None):
        """PhysicsOracle.substep (same arguments and results) on the heightfield."""
        if self.ground is None:
            return super().substep(root, q, qd, tau, damping, armature, mass_scale, push, rb_force, rb_torque)
        t, p, nl, nd, nb = self.t, self.p, self.nl, self.nd, self.nb
        N = root.shape[0]
        dt = p.dt
        g = np.asarray(p.gravity, float)
        X, Rw, pw = self.kinematics(root, q)
        J = self.jacobians(X)
        I = self.link_inertias(mass_scale)
        R0 = Rw[0]
        v0 = np.concatenate([np.einsum("nji,nj->ni", R0, root[:, 10:13]), np.einsum("nji,nj->ni", R0, root[:, 7:10])], -1)
        vgen = np.concatenate([v0, qd], -1)
        v = [np.einsum("nij,nj->ni", Ji, vgen) for Ji in J]
        # velocity-product accelerations
        avp = [np.zeros((N, 6))]
        for i in range(1, nl):
            S = np.zeros(6)
            S[:3] = t.link_axis[i]
            c = crm_apply(v[i], S[None, :] * qd[:, t.link_dof[i], None])
            avp.append(np.einsum("nij,nj->ni", X[i], avp[int(t.link_parent[i])]) + c)
        contact = np.zeros((N, nb, 3))
        M = np.zeros((N, 6 + nd, 6 + nd))
        h = np.zeros((N, 6 + nd))
        par = t.body_inertia[None, :, :] * mass_scale[:, :, None]
        for i in range(nl):
            Ii = I[i]
            M += np.swapaxes(J[i], -1, -2) @ Ii @ J[i]
            ag = np.concatenate([np.zeros((N, 3)), np.einsum("nji,j->ni", Rw[i], g)], -1)
            fi = np.einsum("nij,nj->ni", Ii, avp[i] - ag) + crf_apply(v[i], np.einsum("nij,nj->ni", Ii, v[i]))
            fi = fi - self._external_wrench(i, Rw[i], pw[i], v[i], contact, par, push, rb_force, rb_torque)
            h += np.einsum("nji,nj->ni", J[i], fi)
        idx = np.arange(nd)
        stiff = np.asarray(getattr(t, "dof_stiffness", np.zeros(nd)), float)  # joint spring about q = 0, implicit
        M[:, 6 + idx, 6 + idx] += armature + dt * damping + dt * dt * stiff
        tq = tau.copy()
        if p.clamp_effort:
            tq = np.clip(tq, -t.dof_effort, t.dof_effort)
        rhs = -h
        rhs[:, 6:] += tq - damping * qd - stiff * (q + dt * qd)
        Minv = np.linalg.inv(M)
        acc = np.einsum("nij,nj->ni", Minv, rhs)
        vstar = vgen + dt * acc
        # ---- constraint-solved ground contact of the solver points (block-Jacobi between feet, Gauss-Seidel inside)
        feet = self.feet
        nF = len(feet)
        Jf = [J[f] for f in feet]
        Om = [[Jf[a] @ Minv @ np.swapaxes(Jf[b], -1, -2) for b in range(nF)] for a in range(nF)]
        V = [np.einsum("nij,nj->ni", Jf[a], vstar) for a in range(nF)]
        P = [np.zeros((N, 6)) for _ in range(nF)]
        rows = []  # per foot: list of (Jrow (N,3,6), bias (N,), active (N,), body, world directions (N,3,3))
        for a, f in enumerate(feet):
            cnt = np.zeros(N, int)
            pts = []
            for i in self.foot_pts[f]:
                pts.append(self._field_sole_row(Rw[f], pw[f], t.pt_pos[i], t.pt_radius[i], cnt, int(t.pt_body[i])))
                cnt += pts[-1][2]
            rows.append(pts)
        lam = [[np.zeros((N, 3)) for _ in rows[a]] for a in range(nF)]
        for _ in range(p.sweeps):
            dP = [np.zeros((N, 6)) for _ in range(nF)]
            for a in range(nF):
                Oaa = Om[a][a]
                for k, (Jr, bias, act, _b, _dirs) in enumerate(rows[a]):
                    for d in range(3):
                        Jd = Jr[:, d, :]
                        cvec = np.einsum("nij,nj->ni", Oaa, Jd)
                        w = np.einsum("ni,ni->n", Jd, cvec)
                        vrel = np.einsum("ni,ni->n", Jd, V[a])
                        if d == 0:
                            new = np.maximum(lam[a][k][:, 0] + (bias - vrel) / w, 0.0)
                        else:
                            lim = p.mu * lam[a][k][:, 0]
                            new = np.clip(lam[a][k][:, d] - vrel / w, -lim, lim)
                        delta = np.where(act, new - lam[a][k][:, d], 0.0)
                        lam[a][k][:, d] += delta
                        V[a] = V[a] + cvec * delta[:, None]
                        dP[a] = dP[a] + Jd * delta[:, None]
            for a in range(nF):
                for b in range(nF):
                    if b != a:
                        V[a] = V[a] + np.einsum("nij,nj->ni", Om[a][b], dP[b])
                P[a] = P[a] + dP[a]
        imp = np.zeros((N, 6 + nd))
        for a in range(nF):
            imp += np.einsum("nji,nj->ni", Jf[a], P[a])
            for k, (_Jr, _bias, _act, b, dirs_w) in enumerate(rows[a]):  # world force (lam_n n + lam_1 t1 + lam_2 t2) / dt
                contact[:, b, :] += np.einsum("nd,ndj->nj", lam[a][k], dirs_w) / dt
        vnew = vstar + np.einsum("nij,nj->ni", Minv, imp)
        # ---- joints: velocity cap, integrate, limit projection
        qdn = np.clip(vnew[:, 6:], -p.vel_limit, p.vel_limit)
        qn = q + dt * qdn
        over, under = qn > t.dof_upper, qn < t.dof_lower
        qdn = np.where(over, np.minimum(qdn, 0.0), np.where(under, np.maximum(qdn, 0.0), qdn))
        qn = np.clip(qn, t.dof_lower, t.dof_upper)
        # ---- base
        wb, vb = vnew[:, :3], vnew[:, 3:6] + dt * np.cross(v0[:, :3], v0[:, 3:])
        ww = np.einsum("nij,nj->ni", R0, wb)
        vw = np.einsum("nij,nj->ni", R0, vb)
        wn = np.linalg.norm(ww, axis=-1, keepdims=True)
        ww = np.where(wn > p.max_ang_vel, ww * (p.max_ang_vel / np.maximum(wn, 1e-30)), ww)
        rootn = root.copy()
        rootn[:, 0:3] = root[:, 0:3] + dt * vw
        qx = root[:, 3:7]
        dq = 0.5 * dt * np.stack([ww[:, 0] * qx[:, 3] + ww[:, 1] * qx[:, 2] - ww[:, 2] * qx[:, 1],
                                  -ww[:, 0] * qx[:, 2] + ww[:, 1] * qx[:, 3] + ww[:, 2] * qx[:, 0],
                                  ww[:, 0] * qx[:, 1] - ww[:, 1] * qx[:, 0] + ww[:, 2] * qx[:, 3],
                                  -ww[:, 0] * qx[:, 0] - ww[:, 1] * qx[:, 1] - ww[:, 2] * qx[:, 2]], -1)
        qq = qx + dq
        rootn[:, 3:7] = qq / np.linalg.norm(qq, axis=-1, keepdims=True)
        rootn[:, 7:10] = vw
        rootn[:, 10:13] = ww
        diag = {"M": M, "acc": acc, "vstar": vstar, "lam": lam, "J": J, "I": I, "v": v, "Rw": Rw, "pw": pw}
        return rootn, qn, qdn, contact, diag

    def _field_sole_row(self, Rw, pw, x, rad, cnt, body):
        """Heightfield: rows (N,3,6) in link coordinates, bias, active mask, body and world row directions (N,3,3) of one
        sole candidate: gap phi = (z_c - h) n_z - r, contact location c - r n, rows n, t1, t2."""
        p = self.p
        c = pw + np.einsum("nij,j->ni", Rw, x)
        h, n, inside = self.ground.query(c[:, 0], c[:, 1])
        phi = (c[:, 2] - h) * n[:, 2] - rad
        act = inside & (phi < p.contact_offset) & (cnt < MAX_ACTIVE_PTS)
        t1, t2 = tangents(n)
        dirs_w = np.stack([n, t1, t2], 1)
        dirs = np.einsum("nji,ndj->ndi", Rw, dirs_w)  # link coordinates
        xs = x[None, :] - rad * dirs[:, 0, :]
        Jr = np.concatenate([np.cross(xs[:, None, :], dirs), dirs], -1)
        bias = np.where(phi >= 0, -phi / p.dt, np.minimum(-p.erp * phi / p.dt, p.max_depen_vel))
        return Jr, bias, act, body, dirs_w

    def _external_wrench(self, i, Rw, pw, v, contact, par, push, rb_force, rb_torque):
        """PhysicsOracle._external_wrench on the heightfield: depth (h - z) n_z (+ r for a sphere), normal force along the
        ground normal n damped by v.n, friction on the tangential part of the velocity."""
        if self.ground is None:
            return super()._external_wrench(i, Rw, pw, v, contact, par, push, rb_force, rb_torque)
        t, p = self.t, self.p
        N = Rw.shape[0]
        out = np.zeros((N, 6))

        def add_point_n(xs_l, n_w, depth, body):
            """xs_l (N,3) contact location in link coords, n_w (N,3) world ground normal, depth (N,) > 0 where
            penetrating."""
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

        nrm_l = Rw[:, 2, :]  # world z in link coords
        gnd = self.ground
        for k in self.link_pts[i]:
            x, rad = t.pt_pos[k], t.pt_radius[k]
            c = pw + np.einsum("nij,j->ni", Rw, x)
            h, n, inside = gnd.query(c[:, 0], c[:, 1])
            depth = np.where(inside, (h - c[:, 2]) * n[:, 2] + rad, -1.0)
            add_point_n(x[None, :] - rad * np.einsum("nji,nj->ni", Rw, n), n, depth, int(t.pt_body[k]))
        for k in self.link_cyls[i]:
            c, a, (rad, hh) = t.cyl_center[k], t.cyl_axis[k], t.cyl_size[k]
            az = np.einsum("nj,j->n", nrm_l, a)  # world z component of the axis
            s = np.where(az >= 0, -1.0, 1.0)
            d_l = -(nrm_l - az[:, None] * a[None, :])  # downward radial direction, link coords
            dn = np.linalg.norm(d_l, axis=-1)
            rim = c[None, :] + (s * hh)[:, None] * a[None, :] + np.where(dn[:, None] > 1e-6, rad * d_l / np.maximum(dn, 1e-30)[:, None], 0.0)
            # the rim point lowest in world z (as on the plane), against the ground below it
            q = pw + np.einsum("nij,nj->ni", Rw, rim)
            h, n, inside = gnd.query(q[:, 0], q[:, 1])
            add_point_n(rim, n, np.where(inside, (h - q[:, 2]) * n[:, 2], -1.0), int(t.cyl_body[k]))
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

