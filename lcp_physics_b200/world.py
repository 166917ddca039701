"""`BatchedWorld`: B independent 2-D worlds of circles stepped in lock-step on one GPU (SURVEY.md f-1).

The reference steps ONE scene per `World` object on the host (physics/world.py:72-122) and calls the
LCP with batch = 1 (SURVEY.md F3); `run_world` already anticipates a list of worlds (world.py:250-252).
Here the state of B scenes lives in structure-of-arrays tensors on the GPU and one step is

    new_v           <- -LCP(contact list)            lcpb200_engine_forward, mode 0   (engines.py:50-76)
    p               <- p + new_v dt_s                bodies.py:80-96, per-scene dt halving on penetration
                                                      (world.py:88-107)
    dp              <- -LCP_poststab(contact list)/2 lcpb200_engine_forward, mode 1   (engines.py:80-116,
                                                      world.py:109-120), optional

with contact generation for circle pairs (contacts.py:68-80: normal = (pos1 - pos2)/dist, penetration =
r1 + r2 - dist, contact when penetration >= -eps, p1 = -n (r1 - pen/2), p2 = n (r2 - pen/2)) on the device:
the pair test and the ordered compaction of all nb (nb - 1) / 2 pairs by lcpb200_find_contacts
(csrc/lcp_contacts.cuh), pair order (i < j, lexicographic) as the reference's broadphase callback visits
them, the geometry of the selected pairs by torch ops (differentiable). Every scene keeps its OWN contact count: the fused kernels take a per-scene count, and a scene
without contacts gets the equality-constrained solve of engines.py:35-49 inside the same kernel.

Scope (what the reference's demos use that this class mirrors): `Circle` bodies (bodies.py:114-140),
`Gravity` (forces.py), `TotalConstraint` pins (constraints.py:176-192), joints (`joints=`: revolute `Joint`,
`FixedJoint`, X / Y / Rot / TotalConstraint, lcp_physics_b200/constraints.py) and pairs that never touch
(`no_contact=`, bodies.py:104-106), restitution / friction as the mean of the two bodies (world.py:144-151,
:213-224), `eps`, `tol`, `post_stab`, `strict_no_penetration`. Hulls (`Rect`, `Hull`) and the renderer are not
mirrored (SURVEY.md section 8f). Everything is differentiable through torch autograd (the LCP through
lcpb200_engine_backward). Scenes with 3 nb + e <= 128 (e equality rows) use the condensed-KKT kernels
(fp32 / fp64); larger scenes (BASELINE config 4: a 512-ball pile) the banded large-scene kernels
(csrc/lcp_banded.cuh), float64 with e <= 16.

Joint rows depend on the positions (a revolute joint's lever turns with its body), so they are rebuilt before
every solve: lcpb200_joint_rows writes the dense A[B,e,3nb] the engine kernels take (and ge = A v for
post-stabilisation), lcpb200_joint_move advances the revolute joints' state with the bodies. When something
upstream requires grad, the same rows and state come from torch ops (`joint_rows_torch`, `move_joints_torch`),
which are also the reference the kernels are tested against.
"""
import ctypes
import math

import torch

from . import _lib
from .constraints import UNIT, LEVER_X, LEVER_Y, ROT, TotalConstraint, pair_mask, row_table
from .engines import engine_solve


class BatchedWorld:
    def __init__(self, pos, rad, vel=None, mass=1.0, restitution=0.5, fric_coeff=0.9, gravity=10.0,
                 static=(), gravity_mask=None, dt=1.0 / 30, eps=0.1, tol=1e-6, post_stab=False,
                 strict_no_penetration=True, max_iter=10, contact_capacity=None, device=None, joints=(),
                 no_contact=()):
        """pos [B,nb,2], rad [B,nb] (or [nb] / scalar), vel [B,nb,3] (rot, x, y) or None, mass / restitution /
        fric_coeff [B,nb] (or broadcastable), `static`: indices of bodies pinned by a TotalConstraint,
        `gravity`: g of the `Gravity` force (forces.py) applied to the bodies in gravity_mask
        (default: every non-static body), `joints`: constraint specs of lcp_physics_b200.constraints, shared by
        the batch (a revolute Joint's anchor may be [B,2]); their rows follow the pins', so the reference world
        is World(bodies, [TotalConstraint(s) for s in static] + joints). `no_contact`: pairs (i, j) of bodies
        that never produce a contact."""
        _lib.require_cuda()
        self.device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        pos = torch.as_tensor(pos)
        self.dtype = pos.dtype if pos.dtype in (torch.float32, torch.float64) else torch.float64
        to = lambda t: torch.as_tensor(t, dtype=self.dtype).to(self.device)
        pos = to(pos)
        B, nb, _ = pos.shape
        self.B, self.nb, self.n = B, nb, 3 * nb
        bc = lambda t: to(t).expand(B, nb).contiguous() if torch.as_tensor(t).dim() < 2 else to(t)
        self.rad, self.mass = bc(rad), bc(mass)
        self.restitution, self.fric_coeff = bc(restitution), bc(fric_coeff)
        self.inertia = self.mass * self.rad * self.rad / 2                          # bodies.py:126
        self.p = torch.cat([pos.new_zeros(B, nb, 1), pos], 2)                       # (rot, x, y)  bodies.py:27-33
        self.v = to(vel).reshape(B, self.n).clone() if vel is not None else pos.new_zeros(B, self.n)
        self.static = [int(k) for k in static]
        gm = torch.ones(nb, dtype=torch.bool)
        gm[self.static] = False
        if gravity_mask is not None:
            gm = torch.as_tensor(gravity_mask, dtype=torch.bool)
        self.fext = pos.new_zeros(B, self.n)
        if gravity is not None:
            self.fext[:, 2::3] = self.mass * float(gravity) * gm.to(self.device).to(self.dtype)   # Gravity: DOWN * m * g
        self.joints = list(joints)
        self.nj, self.dynamic_rows = 0, False
        self.ne = 3 * len(self.static)
        if self.joints:
            self._init_joints(pos)
        elif self.ne:
            A = pos.new_zeros(self.ne, self.n)
            for r, k in enumerate(self.static):
                for q in range(3):
                    A[3 * r + q, 3 * k + q] = 1.0                                  # TotalConstraint.J = eye(3)
            self.A = A.unsqueeze(0).expand(B, -1, -1).contiguous()
        else:
            self.A = None
        self.dt, self.eps, self.tol = float(dt), float(eps), float(tol)
        self.post_stab, self.strict_no_pen, self.max_iter = post_stab, strict_no_penetration, max_iter
        ii, jj = torch.triu_indices(nb, nb, 1)
        self.pi, self.pj = ii.to(self.device), jj.to(self.device)                   # pair (i, j), i < j, lexicographic
        self.no_contact = [tuple(pr) for pr in no_contact]
        if self.no_contact:
            mask, words = pair_mask(self.no_contact, nb)
            self.skip_mask, self.skip_words = mask.to(self.device), words.to(self.device)
        else:
            self.skip_mask = self.skip_words = None
        self.cap = int(contact_capacity) if contact_capacity else min(int(self.pi.numel()), 3 * nb)
        # 3 nb + e <= 128 and <= 256 contacts: condensed-KKT kernels (fp32 / fp64, differentiable);
        # larger scenes: the banded large-scene kernels (fp64, <= 16 equality rows; lcp_banded.cuh)
        self.large = self.n + self.ne > 128 or 4 * self.cap > 1024
        if self.large and (self.dtype != torch.float64 or self.ne > 16):
            raise ValueError("BatchedWorld: scenes with 3 nb + e > 128 (or > 256 contacts) need float64 and at most "
                             "16 equality rows; this one has 3 nb = %d, e = %d equality rows (%d pinned bodies), "
                             "%s" % (self.n, self.ne, len(self.static), self.dtype))
        if self.large and self.joints:
            # the banded kernel keeps every body with an equality row and the rows themselves in a border of 16
            nbb = len({int(b) for b in self._r_b1.tolist() + self._r_b2.tolist() if b >= 0})
            if 3 * nbb + self.ne > 16:
                raise ValueError("BatchedWorld: on the banded large-scene kernel 3 x (bodies with equality rows) + e must "
                                 "be <= 16 (its border); this scene has %d such bodies and e = %d rows" % (nbb, self.ne))
        self.t = pos.new_zeros(B)
        self.find_contacts()
        if self.strict_no_pen and bool((self.max_penetration() > self.tol).any()):
            raise AssertionError("Interpenetration at start")                      # world.py:66-68

    # ------------------------------------------------------------------ joints (constraints.py, world.py:156-170)
    def _init_joints(self, pos):
        """Row table and revolute-joint state (constraints.py:16-27): pos1 = anchor - p_b1, r1 = |pos1|,
        rot1 = atan2(y1, x1) (+ 2 pi when negative, utils.cart_to_polar)."""
        B, dev = self.B, self.device
        rows, revolute = row_table([TotalConstraint(k) for k in self.static] + self.joints, self.nb)
        self.ne, self.nj = len(rows), len(revolute)
        self.dynamic_rows = any(r[0] != UNIT for r in rows)
        self.row_table = torch.tensor(rows, dtype=torch.int32).to(dev)                      # [e, 4]
        rt = self.row_table.long()
        self._r_kind, self._r_b1, self._r_b2, self._r_aux = rt[:, 0], rt[:, 1], rt[:, 2], rt[:, 3]
        if self.nj:
            self.joint_body = torch.tensor([j.i1 for j in revolute], dtype=torch.int32).to(dev)
            anchor = torch.stack([j.pos.to(self.dtype).to(dev).expand(B, 2) for j in revolute], 1)   # [B, nj, 2]
            self.j_pos1 = anchor - pos[:, self.joint_body.long()]
            self.j_r1 = self.j_pos1.norm(dim=2)
            rot = torch.atan2(self.j_pos1[..., 1], self.j_pos1[..., 0])
            self.j_rot1 = torch.where(rot < 0, rot + 2 * math.pi, rot)
        else:
            self.joint_body = self.j_pos1 = self.j_r1 = self.j_rot1 = None
        self.A = None if self.dynamic_rows else self.joint_rows()[0]

    def _joint_needs_graph(self, *ts):
        return torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in ts)

    def joint_rows(self, v=None):
        """(A [B,e,3nb], ge = A v [B,e] or None) at the current positions and joint state: lcpb200_joint_rows, or
        joint_rows_torch when something upstream requires grad."""
        if self._joint_needs_graph(self.p, self.j_pos1, v):
            return self.joint_rows_torch(v)
        lib = _lib.load()
        dev = self.device
        pos_c = self.p[:, :, 1:].detach().contiguous()
        A = torch.empty(self.B, self.ne, self.n, dtype=self.dtype, device=dev)
        ge = torch.empty(self.B, self.ne, dtype=self.dtype, device=dev) if v is not None else None
        pos1 = self.j_pos1.detach().contiguous() if self.nj else None
        with torch.cuda.device(dev):
            _lib.check(lib.lcpb200_joint_rows(
                _lib.dtype_code(self.dtype), self.B, self.nb, self.ne, self.nj, _lib.ptr(self.row_table), _lib.ptr(pos_c),
                _lib.ptr(pos1), _lib.ptr(v.detach().contiguous() if v is not None else None), _lib.ptr(A), _lib.ptr(ge),
                ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
        return A, ge

    def joint_rows_torch(self, v=None):
        """The rows of joint_rows with torch ops (differentiable w.r.t. positions, anchors and v)."""
        B, e, n = self.B, self.ne, self.n
        pos = self.p[:, :, 1:]
        kind, b1, b2, aux = self._r_kind, self._r_b1, self._r_b2, self._r_aux
        lever = (kind == LEVER_X) | (kind == LEVER_Y)
        if self.nj:
            p1 = self.j_pos1[:, aux.clamp(min=0)]
            p1 = torch.where((lever & (aux >= 0)).reshape(1, e, 1), p1, torch.zeros_like(p1))
        else:
            p1 = pos.new_zeros(B, e, 2)
        p2 = (pos[:, b1] + p1) - pos[:, b2.clamp(min=0)]                                      # pos2 = p_b1 + pos1 - p_b2
        eye = torch.eye(3, dtype=self.dtype, device=self.device)
        c1 = torch.where((kind == UNIT).unsqueeze(1), eye[aux.clamp(0, 2)], torch.zeros_like(eye[aux.clamp(0, 2)]))
        c1 = c1 + eye[1] * (kind == LEVER_X).unsqueeze(1) + eye[2] * (kind == LEVER_Y).unsqueeze(1) \
            + eye[0] * (kind == ROT).unsqueeze(1)
        c2 = -(eye[1] * (kind == LEVER_X).unsqueeze(1) + eye[2] * (kind == LEVER_Y).unsqueeze(1)
               + eye[0] * (kind == ROT).unsqueeze(1))
        lx, ly = (kind == LEVER_X).reshape(1, e), (kind == LEVER_Y).reshape(1, e)
        c1 = c1.expand(B, e, 3)
        c2 = c2.expand(B, e, 3)
        j1 = torch.cat([torch.where(lx, -p1[..., 1], torch.where(ly, p1[..., 0], c1[..., 0])).unsqueeze(2), c1[..., 1:]], 2)
        j2 = torch.cat([torch.where(lx, p2[..., 1], torch.where(ly, -p2[..., 0], c2[..., 0])).unsqueeze(2), c2[..., 1:]], 2)
        q = torch.arange(3, device=self.device)
        idx1 = (3 * b1.unsqueeze(1) + q).expand(B, e, 3)
        idx2 = torch.where((b2 >= 0).unsqueeze(1), 3 * b2.unsqueeze(1) + q, n + q).expand(B, e, 3)   # no body 2: pad
        A = pos.new_zeros(B, e, n + 3).scatter(2, idx1, j1).scatter(2, idx2, j2)[:, :, :n].contiguous()
        ge = torch.bmm(A, v.unsqueeze(2)).squeeze(2) if v is not None else None
        return A, ge

    def move_joints(self, rot_start, v, dts, done=None):
        """Joint.move (constraints.py:38-45) of every revolute joint: rot1 = rot_start + v[3 b1] dts,
        pos1 = r1 (cos, sin)(rot1); scenes flagged done keep their state. lcpb200_joint_move, or move_joints_torch
        when something upstream requires grad."""
        if self._joint_needs_graph(rot_start, v, self.j_r1, self.j_rot1, self.j_pos1):
            return self.move_joints_torch(rot_start, v, dts, done)
        if self.j_rot1.requires_grad or self.j_pos1.requires_grad:     # the kernel updates the state in place
            self.j_rot1, self.j_pos1 = self.j_rot1.detach().clone(), self.j_pos1.detach().clone()
        lib = _lib.load()
        dev = self.device
        rs = self.j_rot1 if rot_start is self.j_rot1 else rot_start.detach().contiguous()
        with torch.cuda.device(dev):
            _lib.check(lib.lcpb200_joint_move(
                _lib.dtype_code(self.dtype), self.B, self.nb, self.nj, _lib.ptr(self.joint_body), _lib.ptr(rs),
                _lib.ptr(self.j_r1.detach().contiguous()), _lib.ptr(v.detach().contiguous()),
                _lib.ptr(dts.contiguous()), _lib.ptr(done.contiguous() if done is not None else None),
                _lib.ptr(self.j_rot1), _lib.ptr(self.j_pos1),
                ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))

    def move_joints_torch(self, rot_start, v, dts, done=None):
        """move_joints with torch ops (differentiable)."""
        rot = rot_start + v[:, 3 * self.joint_body.long()] * dts.unsqueeze(1)
        pos1 = torch.stack([torch.cos(rot), torch.sin(rot)], 2) * self.j_r1.unsqueeze(2)
        if done is not None:
            rot = torch.where(done.unsqueeze(1), self.j_rot1, rot)
            pos1 = torch.where(done.reshape(-1, 1, 1), self.j_pos1, pos1)
        self.j_rot1, self.j_pos1 = rot, pos1

    # ------------------------------------------------------------------ contacts.py:68-80, batched
    def find_contacts(self):
        """Pair test + ordered compaction on the GPU (lcpb200_find_contacts: all nb (nb - 1) / 2 pairs of every
        scene, lexicographic order = the reference's contact order), then the contact geometry of the selected
        pairs with torch ops (differentiable w.r.t. the positions)."""
        lib = _lib.load()
        B, cap, dev = self.B, self.cap, self.device
        pos = self.p[:, :, 1:]
        pos_c = pos.detach().contiguous()
        b1 = torch.empty(B, cap, dtype=torch.int32, device=dev)
        b2 = torch.empty(B, cap, dtype=torch.int32, device=dev)
        counts = torch.empty(B, dtype=torch.int32, device=dev)
        with torch.cuda.device(dev):
            if self.skip_words is None:
                _lib.check(lib.lcpb200_find_contacts(_lib.dtype_code(self.dtype), B, self.nb, cap, self.eps, _lib.ptr(pos_c),
                                                     _lib.ptr(self.rad), _lib.ptr(b1), _lib.ptr(b2), _lib.ptr(counts),
                                                     ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
            else:
                _lib.check(lib.lcpb200_find_contacts_masked(
                    _lib.dtype_code(self.dtype), B, self.nb, cap, self.eps, _lib.ptr(pos_c), _lib.ptr(self.rad),
                    _lib.ptr(self.skip_words), _lib.ptr(b1), _lib.ptr(b2), _lib.ptr(counts),
                    ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
        if int(counts.max()) > cap:
            raise RuntimeError("BatchedWorld: a scene has %d contacts, capacity %d" % (int(counts.max()), cap))
        self.c_b1, self.c_b2, self.counts = b1, b2, counts
        needs_graph = torch.is_grad_enabled() and any(t.requires_grad for t in (self.p, self.rad, self.fric_coeff, self.restitution))
        if not needs_graph:
            # nothing to differentiate: the geometry of the selected pairs in one kernel as well
            new = lambda *s_: torch.empty(B, cap, *s_, dtype=self.dtype, device=dev)
            self.c_normal, self.c_p1, self.c_p2 = new(2), new(2), new(2)
            self.c_pen, self.c_mu, self.c_rest = new(), new(), new()
            with torch.cuda.device(dev):
                _lib.check(lib.lcpb200_contact_geometry(
                    _lib.dtype_code(self.dtype), B, self.nb, cap, _lib.ptr(pos_c), _lib.ptr(self.rad.detach().contiguous()),
                    _lib.ptr(self.fric_coeff.detach().contiguous()), _lib.ptr(self.restitution.detach().contiguous()),
                    _lib.ptr(b1), _lib.ptr(b2), _lib.ptr(counts),
                    *[_lib.ptr(t) for t in (self.c_normal, self.c_p1, self.c_p2, self.c_pen, self.c_mu, self.c_rest)],
                    ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
            return
        i1, i2 = b1.long(), b2.long()
        take = lambda t, idx: torch.gather(t, 1, idx)
        d = torch.gather(pos, 1, i1.unsqueeze(2).expand(-1, -1, 2)) - torch.gather(pos, 1, i2.unsqueeze(2).expand(-1, -1, 2))
        dist = d.norm(dim=2)                                                       # b1.pos - b2.pos   contacts.py:69-71
        r1, r2 = take(self.rad, i1), take(self.rad, i2)
        pen_c = r1 + r2 - dist
        normal = d / dist.unsqueeze(2)
        valid = torch.arange(cap, device=dev).unsqueeze(0) < counts.unsqueeze(1)
        self.c_normal = normal
        self.c_p1 = -normal * (r1 - pen_c / 2).unsqueeze(2)                        # contacts.py:75-77
        self.c_p2 = normal * (r2 - pen_c / 2).unsqueeze(2)
        self.c_pen = torch.where(valid, pen_c, pen_c.new_full((), -1e30))
        self.c_b1, self.c_b2 = b1, b2
        self.c_mu = 0.5 * (take(self.fric_coeff, i1) + take(self.fric_coeff, i2))              # world.py:213-224
        self.c_rest = 0.5 * (take(self.restitution, i1) + take(self.restitution, i2))          # world.py:144-151
        self.counts = counts

    def find_contacts_torch(self):
        """The same contact list with torch ops only (O(nb^2) tensors, a stable sort for the compaction): the
        independent implementation tests/test_gpu_world.py checks lcpb200_find_contacts against. Returns
        (counts, b1, b2)."""
        pos = self.p[:, :, 1:]
        d = pos[:, self.pi] - pos[:, self.pj]
        pen = self.rad[:, self.pi] + self.rad[:, self.pj] - d.norm(dim=2)
        active = pen >= -self.eps                                                  # `if penetration < -eps: return`
        if self.skip_mask is not None:
            active = active & ~self.skip_mask                                      # no_contact pairs
        counts = active.sum(1)
        order = torch.sort((~active).to(torch.int8), dim=1, stable=True)[1][:, :self.cap]   # active pairs first, in pair order
        return counts.to(torch.int32), self.pi[order].to(torch.int32), self.pj[order].to(torch.int32)

    def max_penetration(self):
        return self.c_pen.max(dim=1)[0]

    # ------------------------------------------------------------------ engine calls
    def _lcp(self, mode, dt, b):
        z, status = engine_solve(self.mass, self.inertia, self.v, self.fext, self.c_normal, self.c_p1, self.c_p2,
                                 self.c_mu, self.c_rest, self.c_b1, self.c_b2, dt, A=self.A, b=b, mode=mode,
                                 max_iter=self.max_iter if mode == 0 else 10, counts=self.counts)
        if bool((status == _lib.STATUS_SINGULAR_Q).any()):
            from .lcp import SINGULAR_Q_MSG
            raise RuntimeError(SINGULAR_Q_MSG)
        if bool((status == -100).any()):
            raise RuntimeError("BatchedWorld: a scene's contact topology is not supported by the fused kernel")
        return z

    def solve_dynamics(self, dt):
        """engines.py:26-78 for every scene: new_v = -zhat."""
        if self.dynamic_rows:
            self.A = self.joint_rows()[0]
        b = self.v.new_zeros(self.B, self.ne) if self.ne else None
        return -self._lcp(0, dt, b)

    def post_stabilization(self):
        """engines.py:80-116 for every scene: -zhat with b = Je v."""
        if self.dynamic_rows:
            self.A, b = self.joint_rows(self.v)
        else:
            b = torch.bmm(self.A, self.v.unsqueeze(2)).squeeze(2) if self.ne else None
        return -self._lcp(1, 0.0, b)

    # ------------------------------------------------------------------ world.py:72-122
    def step(self):
        self.step_dt(self.dt)

    def step_dt(self, dt):
        start_p = self.p.clone()
        start_rot = self.j_rot1.clone() if self.nj else None                      # world.py:85
        self.v = self.solve_dynamics(dt)
        dts = self.v.new_full((self.B,), float(dt))
        done = torch.zeros(self.B, dtype=torch.bool, device=self.device)
        while True:
            moved = start_p + self.v.reshape(self.B, self.nb, 3) * dts.reshape(self.B, 1, 1)      # body.move(dt)
            self.p = torch.where(done.reshape(self.B, 1, 1), self.p, moved)
            if self.nj:
                self.move_joints(start_rot, self.v, dts, done)                     # joint.move(dt), world.py:93
            self.find_contacts()
            ok = self.max_penetration() <= self.tol
            if not self.strict_no_pen:
                ok = ok | (dts < self.dt / 4)                                      # world.py:98-100
            done = done | ok
            if bool(done.all()):
                break
            dts = torch.where(done, dts, dts / 2)                                  # world.py:101 (positions reset: start_p)
        if self.post_stab:
            tmp_v = self.v
            dp = self.post_stabilization() / 2                                     # world.py:111-112
            self.p = self.p + dp.reshape(self.B, self.nb, 3) * dts.reshape(self.B, 1, 1)
            if self.nj:
                self.move_joints(self.j_rot1, dp, dts)                             # world.py:117-118
            self.v = tmp_v
            self.find_contacts()
        self.t = self.t + dts

    def get_v(self):
        return self.v

    def get_p(self):
        return self.p.reshape(self.B, self.n)
