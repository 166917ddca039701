"""TEST INFRASTRUCTURE ONLY -- CPU restatement of the reference's `World.step_dt` for circle scenes WITH joints and
no-contact pairs: `OracleCircleWorld` (oracle/world_oracle.py) extended by

  * constraints.py:13-173 (Joint, FixedJoint, X / Y / RotConstraint: J, move, update_pos)
  * world.py:85, :101-107 (the joints' rot1 restarts with the positions when dt is halved), :117-118 (post-stab move)
  * world.py:156-170 (Je, recomputed before every solve: the pins' rows first, then the joints' in list order)
  * bodies.py:104-106 + contacts.py:60-61 (no_contact pairs never produce a contact)

Only `tests/` imports this module. PARITY PIN: `tests/test_joint_world_oracle.py` checks it against trajectories
recorded from the unmodified reference (`tests/golden/bworld_joints.npz`).
"""
import math

import torch

from .world_oracle import OracleCircleWorld


def _cart_to_polar(v):                                   # utils.py:75-82
    theta = torch.atan2(v[1], v[0])
    if theta.item() < 0:
        theta = theta + 2 * math.pi
    return v.norm(), theta


class OracleJointWorld(OracleCircleWorld):
    def __init__(self, pos, rad, vel, mass, restitution, fric_coeff, gravity=100.0, static=(0,), dt=1.0 / 30,
                 eps=0.1, tol=1e-6, post_stab=False, max_iter=10, joints=(), no_contact=()):
        """joints: specs of lcp_physics_b200.constraints (a Joint's pos is [2]); their rows follow the pins'.
        no_contact: pairs of bodies that never produce a contact."""
        self.no_contact = {frozenset((int(i), int(j))) for i, j in no_contact}
        super().__init__(pos, rad, vel, mass, restitution, fric_coeff, gravity=gravity, static=static, dt=dt, eps=eps,
                         tol=tol, post_stab=post_stab, max_iter=max_iter)
        f64 = torch.float64
        self.joints = []
        for spec in joints:
            kind = type(spec).__name__
            j = dict(kind=kind, i1=spec.i1, i2=spec.i2)
            if kind == "Joint":                          # constraints.py:16-27
                j["pos"] = torch.as_tensor(spec.pos, dtype=f64).reshape(2).clone()
                j["pos1"] = j["pos"] - self.p[spec.i1, 1:]
                j["r1"], j["rot1"] = _cart_to_polar(j["pos1"])
                if spec.i2 is not None:
                    j["pos2"] = j["pos"] - self.p[spec.i2, 1:]
            elif kind == "FixedJoint":                   # constraints.py:58-68
                j["pos"] = self.p[spec.i1, 1:]
                j["pos1"] = j["pos"] - self.p[spec.i1, 1:]
                j["pos2"] = j["pos"] - self.p[spec.i2, 1:]
            self.joints.append(j)
        self.Je = self._je()

    def _je(self):
        """world.py:156-170 with the pins first."""
        f64 = torch.float64
        blocks = [(torch.eye(3, dtype=f64), k, None, None) for k in self.static]
        for j in self.joints:
            kind = j["kind"]
            if kind in ("Joint", "FixedJoint"):          # constraints.py:29-36, :70-77
                p1 = j["pos1"]
                J1 = torch.stack([torch.stack([-p1[1], p1.new_tensor(1.0), p1.new_tensor(0.0)]),
                                  torch.stack([p1[0], p1.new_tensor(0.0), p1.new_tensor(1.0)])])
                J2 = None
                if j["i2"] is not None:
                    p2 = j["pos2"]
                    J2 = torch.stack([torch.stack([p2[1], p2.new_tensor(-1.0), p2.new_tensor(0.0)]),
                                      torch.stack([-p2[0], p2.new_tensor(0.0), p2.new_tensor(-1.0)])])
                if kind == "FixedJoint":
                    J1 = torch.cat([J1, J1.new_tensor([[1.0, 0.0, 0.0]])])
                    J2 = torch.cat([J2, J2.new_tensor([[-1.0, 0.0, 0.0]])])
                blocks.append((J1, j["i1"], J2, j["i2"]))
            else:
                q = {"XConstraint": [0.0, 1.0, 0.0], "YConstraint": [0.0, 0.0, 1.0], "RotConstraint": [1.0, 0.0, 0.0],
                     "TotalConstraint": None}[kind]
                J1 = torch.eye(3, dtype=f64) if q is None else torch.tensor([q], dtype=f64)
                blocks.append((J1, j["i1"], None, None))
        Je = torch.zeros(sum(b[0].shape[0] for b in blocks), self.n, dtype=f64)
        r = 0
        for J1, i1, J2, i2 in blocks:
            Je[r:r + J1.shape[0], 3 * i1:3 * i1 + 3] = J1
            if J2 is not None:
                Je[r:r + J2.shape[0], 3 * i2:3 * i2 + 3] = J2
            r += J1.shape[0]
        return Je

    def _move_joints(self, v, dt):
        """joint.move(dt) (constraints.py:38-45, :79-87): a revolute joint turns with body 1, then update_pos."""
        for j in self.joints:
            if j["kind"] == "Joint":
                j["rot1"] = j["rot1"] + v[3 * j["i1"]] * dt
                j["pos1"] = torch.cat([torch.cos(j["rot1"]).unsqueeze(0),
                                       torch.sin(j["rot1"]).unsqueeze(0)]).squeeze() * j["r1"]
                j["pos"] = self.p[j["i1"], 1:] + j["pos1"]
                if j["i2"] is not None:
                    j["pos2"] = j["pos"] - self.p[j["i2"], 1:]
            elif j["kind"] == "FixedJoint":
                j["pos"] = self.p[j["i1"], 1:]
                j["pos1"] = j["pos"] - self.p[j["i1"], 1:]
                j["pos2"] = j["pos"] - self.p[j["i2"], 1:]

    def find_contacts(self):
        cs = []
        for i in range(self.nb):
            for j in range(i + 1, self.nb):
                if frozenset((i, j)) in self.no_contact:          # `if geom1 in geom2.no_contact: return`
                    continue
                nrm = self.p[i, 1:] - self.p[j, 1:]
                dist = nrm.norm()
                pen = self.rad[i] + self.rad[j] - dist
                if pen.item() < -self.eps:
                    continue
                nrm = nrm / dist
                cs.append((nrm, -nrm * (self.rad[i] - pen / 2), nrm * (self.rad[j] - pen / 2), pen, i, j))
        self.contacts = cs

    def solve_dynamics(self, dt):
        self.Je = self._je()
        return super().solve_dynamics(dt)

    def post_stabilization(self):
        self.Je = self._je()
        return super().post_stabilization()

    def step(self):
        dt = self.dt
        start_p = self.p.clone()
        start_rot = [j.get("rot1") for j in self.joints]                   # world.py:85
        self.v = self.solve_dynamics(dt)
        while True:
            self.p = start_p + self.v.reshape(self.nb, 3) * dt
            self._move_joints(self.v, dt)
            self.find_contacts()
            if all(c[3].item() <= self.tol for c in self.contacts):
                break
            dt /= 2
            for j, r in zip(self.joints, start_rot):                       # world.py:104-107
                if r is not None:
                    j["rot1"] = r
        if self.post_stab:
            dp = self.post_stabilization() / 2
            self.p = self.p + dp.reshape(self.nb, 3) * dt
            self._move_joints(dp, dt)
            self.find_contacts()
        self.t += dt
