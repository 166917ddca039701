"""Seeded synthetic batched contact scenes (SURVEY.md section 8(d)).

Builds exactly what `PdipmEngine.solve_dynamics` hands to `LCPFunction`
(reference `lcp_physics/physics/engines.py:50-76`) for `B` independent 2-D
scenes of `nb` circles with `nc` contacts and `fd` friction directions:

    Q = blockdiag(1/2 m r^2, m, m)                  (bodies.py:44-47,126)
    Jc rows  [r1 x n, n | -(r2 x n), -n]            (world.py:172-184)
    Jf rows  +-left_orthogonal(n), same lever arms  (world.py:186-211)
    G = [Jc; Jf; 0],  F = [[0,0,0],[0,0,E],[mu,-E^T,0]],
    p = M v + dt f,   h = [(Jc v) * restitution, 0, 0]
    A = identity rows pinning body 0 (a TotalConstraint, constraints.py:176-192)

Everything is generated on the CPU with a `torch.Generator`: the random draws are
reproducible across hosts, the derived arithmetic (normals, Jacobians) only to the
last bit or two (different BLAS code paths) -- fixtures that must be exact store
their inputs (tests/golden/make_seeded_golden.py).
Also exposes the contact/body structure-of-arrays the assembly kernel consumes.
"""
import math

import torch


def pile_layout(nb, nc):
    """Bodies on a W x H grid (a settled pile); contact c joins grid neighbours:
    horizontal, vertical, the two diagonals, then distance-2 pairs, in that order.
    Returns (W, H, body1[nc], body2[nc])."""
    W = int(math.ceil(math.sqrt(nb)))
    while nb % W:
        W += 1
    H = nb // W
    if W < H:
        W, H = H, W
    pairs = []
    for dx, dy in ((1, 0), (0, 1), (1, 1), (-1, 1), (2, 0), (0, 2), (2, 1), (1, 2)):
        for k in range(nb):
            x2, y2 = k % W + dx, k // W + dy
            if 0 <= x2 < W and 0 <= y2 < H:
                pairs.append((k, y2 * W + x2))
    if len(pairs) < nc:
        raise ValueError("pile of %d bodies has only %d candidate contacts (< %d)"
                         % (nb, len(pairs), nc))
    i1 = torch.tensor([p[0] for p in pairs[:nc]])
    i2 = torch.tensor([p[1] for p in pairs[:nc]])
    return W, H, i1, i2


def make_contact_soa(B, nb, nc, seed=0, dtype=torch.float64, jitter=0.2, vscale=1.0):
    """Random bodies + a geometrically consistent contact list (SoA) for B scenes.

    SURVEY.md 8(d) pairs contact c with bodies (c mod nb, (7c+1) mod nb) and
    draws the normal at random; that gives mutually inconsistent constraints and
    the reference solver DIVERGES on it (residual 1e13 by iteration 8), which makes
    parity meaningless. We keep every other rule of 8(d) but take pairs and normals
    from a jittered grid pile, using the reference's circle-circle convention
    (contacts.py:68-80): normal = (pos1 - pos2)/|.|, p1 = -r1 n, p2 = r2 n.
    On these scenes the reference reaches residual 1e-4..1e-8 in 10 iterations."""
    g = torch.Generator().manual_seed(seed)
    f64 = torch.float64
    W, H, i1, i2 = pile_layout(nb, nc)
    mass = torch.rand(B, nb, generator=g, dtype=f64) + 0.5
    rad = torch.rand(B, nb, generator=g, dtype=f64) * 0.2 + 0.9
    k = torch.arange(nb)
    grid = torch.stack([(k % W).to(f64) * 2, (k // W).to(f64) * 2], -1)
    pos = grid.unsqueeze(0) + (torch.rand(B, nb, 2, generator=g, dtype=f64) - 0.5) * (2 * jitter)
    mu = torch.rand(B, nc, generator=g, dtype=f64) * 0.8 + 0.1
    v = torch.randn(B, 3 * nb, generator=g, dtype=f64) * vscale
    normal = pos[:, i1] - pos[:, i2]
    normal = normal / normal.norm(dim=-1, keepdim=True)
    p1 = -rad[:, i1].unsqueeze(-1) * normal
    p2 = rad[:, i2].unsqueeze(-1) * normal
    inertia = 0.5 * mass * rad * rad
    soa = dict(mass=mass, inertia=inertia, normal=normal, p1=p1, p2=p2,
               body1=i1.to(torch.int32), body2=i2.to(torch.int32),
               mu=mu, restitution=torch.full((B, nc), 0.5, dtype=f64), v=v)
    return {k: (t.to(dtype) if t.is_floating_point() else t) for k, t in soa.items()}


def _cross2(a, b):
    return a[..., 0] * b[..., 1] - a[..., 1] * b[..., 0]


def assemble_dense(soa, fd=2, e=0, dt=1.0 / 30, gravity=10.0, seed=0):
    """Plain-torch dense assembly of (Q, p, G, h, A, b, F) from the SoA --
    host-side reference used to create inputs; the CUDA assembly kernel is
    tested against it."""
    mass, inertia = soa["mass"], soa["inertia"]
    B, nb = mass.shape
    dtype = mass.dtype
    normal, p1, p2 = soa["normal"], soa["p1"], soa["p2"]
    nc = normal.shape[1]
    i1, i2 = soa["body1"].long(), soa["body2"].long()
    n = 3 * nb
    m = nc * (2 + fd)

    Mdiag = torch.stack([inertia, mass, mass], -1).reshape(B, n)
    Q = torch.diag_embed(Mdiag)

    def rows(direction, sign2=-1.0):
        # one Jacobian row per contact for a given direction field [B,nc,2]
        J = torch.zeros(B, nc, n, dtype=dtype)
        c1 = _cross2(p1, direction)
        c2 = _cross2(p2, direction)
        ar = torch.arange(nc)
        J[:, ar, 3 * i1 + 0] += c1
        J[:, ar, 3 * i1 + 1] += direction[..., 0]
        J[:, ar, 3 * i1 + 2] += direction[..., 1]
        J[:, ar, 3 * i2 + 0] += sign2 * c2
        J[:, ar, 3 * i2 + 1] += sign2 * direction[..., 0]
        J[:, ar, 3 * i2 + 2] += sign2 * direction[..., 1]
        return J

    Jc = rows(normal)
    d1 = torch.stack([normal[..., 1], -normal[..., 0]], -1)            # left_orthogonal
    dirs = [d1, -d1]
    if fd == 3:
        # non-physical third row (SURVEY.md F9): independent random direction
        g = torch.Generator().manual_seed(seed + 7919)
        a3 = torch.rand(B, nc, generator=g, dtype=torch.float64) * (2 * math.pi)
        dirs.append(torch.stack([torch.cos(a3), torch.sin(a3)], -1).to(dtype))
    elif fd != 2:
        raise ValueError("fd must be 2 or 3")
    Jf = torch.stack([rows(d) for d in dirs], 2).reshape(B, nc * fd, n)
    G = torch.cat([Jc, Jf, torch.zeros(B, nc, n, dtype=dtype)], 1)

    E = torch.zeros(nc * fd, nc, dtype=dtype)
    for k in range(fd):
        E[torch.arange(nc) * fd + k, torch.arange(nc)] = 1
    F = torch.zeros(B, m, m, dtype=dtype)
    F[:, nc:nc + nc * fd, nc + nc * fd:] = E
    F[:, nc + nc * fd:, :nc] = torch.diag_embed(soa["mu"])
    F[:, nc + nc * fd:, nc:nc + nc * fd] = -E.t()

    v = soa["v"]
    fvec = torch.zeros(B, n, dtype=dtype)
    fvec[:, 2::3] = gravity * mass
    p = Mdiag * v + dt * fvec
    h = torch.cat([torch.bmm(Jc, v.unsqueeze(2)).squeeze(2) * soa["restitution"],
                   torch.zeros(B, nc * fd + nc, dtype=dtype)], 1)
    if e > 0:
        A = torch.zeros(B, e, n, dtype=dtype)
        A[:, torch.arange(e), torch.arange(e)] = 1
        b = torch.zeros(B, e, dtype=dtype)
    else:
        A = torch.tensor([], dtype=dtype)
        b = torch.tensor([], dtype=dtype)
    return Q, p, G, h, A, b, F


def make_scenes(B, nb, nc, fd=2, e=0, dtype=torch.float32, seed=0):
    """(Q, p, G, h, A, b, F) for B scenes; n = 3 nb, m = nc (2 + fd)."""
    soa = make_contact_soa(B, nb, nc, seed=seed, dtype=torch.float64)
    out = assemble_dense(soa, fd=fd, e=e, seed=seed)
    return tuple(t.to(dtype).contiguous() for t in out)


def make_dense_random(B, n, m, e=0, dtype=torch.float64, seed=0):
    """Generic dense LCP (no contact structure): SPD Q, random G/A, F = L L^T-ish
    PSD + skew part. Exercises the solver on fully dense inputs."""
    g = torch.Generator().manual_seed(seed)
    f64 = torch.float64
    L = torch.randn(B, n, n, generator=g, dtype=f64)
    Q = torch.bmm(L, L.transpose(1, 2)) / n + torch.eye(n, dtype=f64)
    G = torch.randn(B, m, n, generator=g, dtype=f64)
    z0 = torch.rand(B, n, generator=g, dtype=f64)
    s0 = torch.rand(B, m, generator=g, dtype=f64) + 0.1
    h = torch.bmm(G, z0.unsqueeze(2)).squeeze(2) + s0
    p = torch.randn(B, n, generator=g, dtype=f64)
    W = torch.randn(B, m, m, generator=g, dtype=f64) * 0.1
    F = torch.bmm(W, W.transpose(1, 2)) * 0.1 + 0.2 * (W - W.transpose(1, 2))
    if e > 0:
        A = torch.randn(B, e, n, generator=g, dtype=f64)
        b = torch.bmm(A, z0.unsqueeze(2)).squeeze(2)
    else:
        A = torch.tensor([], dtype=f64)
        b = torch.tensor([], dtype=f64)
    return tuple(t.to(dtype).contiguous() for t in (Q, p, G, h, A, b, F))


def make_ball_drop(B, nballs=24, cols=6, seed=0, dtype=torch.float64, r_floor=2000.0):
    """Initial conditions of B `BatchedWorld` scenes: `nballs` balls (radius 20) in a loose cols-wide cluster,
    dropped onto a huge pinned ball (radius r_floor, body 0) that plays the floor -- the circle-only analogue of
    the reference's ball-pile demos (demos/demo.py). Returns a dict of [B, ...] tensors for BatchedWorld."""
    g = torch.Generator().manual_seed(seed)
    f64 = torch.float64
    nb = nballs + 1
    k = torch.arange(nballs)
    x = 300.0 - 21.0 * (cols - 1) + 42.0 * (k % cols).to(f64)
    y = 470.0 - 43.0 * (k // cols).to(f64)
    pos = torch.zeros(B, nb, 2, dtype=f64)
    pos[:, 0] = torch.tensor([300.0, 500.0 + r_floor], dtype=f64)
    pos[:, 1:, 0] = x + torch.rand(B, nballs, generator=g, dtype=f64) * 0.8
    pos[:, 1:, 1] = y - torch.rand(B, nballs, generator=g, dtype=f64) * 3.0
    vel = torch.zeros(B, nb, 3, dtype=f64)
    vel[:, 1:] = torch.randn(B, nballs, 3, generator=g, dtype=f64) * torch.tensor([0.2, 5.0, 5.0], dtype=f64)
    rad = torch.full((B, nb), 20.0, dtype=f64)
    rad[:, 0] = r_floor
    mass = torch.ones(B, nb, dtype=f64)
    mass[:, 1:] = 0.5 + torch.rand(B, nballs, generator=g, dtype=f64)
    fric = torch.full((B, nb), 0.9, dtype=f64)
    fric[:, 1:] = 0.2 + 0.7 * torch.rand(B, nballs, generator=g, dtype=f64)
    rest = torch.full((B, nb), 0.5, dtype=f64)
    rest[:, 1:] = 0.2 + 0.5 * torch.rand(B, nballs, generator=g, dtype=f64)
    return {k_: t.to(dtype) for k_, t in dict(pos=pos, vel=vel, rad=rad, mass=mass, fric=fric, rest=rest).items()}


def make_ball_pile(B, nballs=512, cols=32, seed=0, dtype=torch.float64, r=10.0, r_floor=1.0e5, gap=0.5):
    """BASELINE config 4 ("World.step() loop: 512-body ball pile"): `nballs` balls of radius r stacked in a
    hexagonal grid `cols` wide, `gap` apart, resting just above a huge pinned ball (radius r_floor, body 0)
    that plays the floor -- the circle-only analogue of the reference's Rect floor (BatchedWorld mirrors
    circle-circle contacts, contacts.py:68-80). y grows downwards (Gravity is +y, forces.py)."""
    g = torch.Generator().manual_seed(seed)
    f64 = torch.float64
    nb = nballs + 1
    k = torch.arange(nballs)
    row, col = k // cols, k % cols
    pitch = 2 * r + gap
    x = 500.0 + pitch * (col.to(f64) - (cols - 1) / 2) + (row % 2).to(f64) * (pitch / 2)
    y = 500.0 - r - gap - row.to(f64) * (pitch * math.sqrt(3) / 2)
    pos = torch.zeros(B, nb, 2, dtype=f64)
    pos[:, 0] = torch.tensor([500.0, 500.0 + r_floor], dtype=f64)
    pos[:, 1:, 0] = x + (torch.rand(B, nballs, generator=g, dtype=f64) - 0.5) * (gap / 4)
    pos[:, 1:, 1] = y - torch.rand(B, nballs, generator=g, dtype=f64) * (gap / 4)
    vel = torch.zeros(B, nb, 3, dtype=f64)
    rad = torch.full((B, nb), r, dtype=f64)
    rad[:, 0] = r_floor
    mass = torch.ones(B, nb, dtype=f64)
    fric = torch.full((B, nb), 0.9, dtype=f64)               # utils.py:22-24 defaults
    rest = torch.full((B, nb), 0.5, dtype=f64)
    return {k_: t.to(dtype) for k_, t in dict(pos=pos, vel=vel, rad=rad, mass=mass, fric=fric, rest=rest).items()}


JOINT_CHAIN_LINKS = 5


def make_joint_chain(B, seed=0, dtype=torch.float64, links=JOINT_CHAIN_LINKS):
    """Initial conditions of B jointed `BatchedWorld` scenes (the circle analogue of the reference's chain_demo,
    demos/demo.py:62-90): body 0 a huge pinned ball that plays the floor (radius 2000), bodies 1..links a chain of
    overlapping circles (radius 15, 25 apart) hung from a world Joint, each link jointed to the one above it at their
    midpoint (Joint(k + 1, k, ...), i1 > i2 as in chain_demo), then a ball thrown at the chain, a ball held by X and
    Rot constraints falling onto the floor, and a FixedJoint pair falling onto the floor. Each scene has its own
    velocities, masses, friction, restitution and anchor jitter. Returns a dict of [B, ...] tensors; `anchor`
    [B, links, 2] are the joint anchors (joint_chain_specs turns them into constraint specs)."""
    g = torch.Generator().manual_seed(seed)
    L = links
    nb = L + 5
    u = lambda *s: torch.rand(B, *s, generator=g, dtype=torch.float64)
    pos = torch.zeros(B, nb, 2, dtype=torch.float64)
    rad = torch.full((B, nb), 15.0, dtype=torch.float64)
    pos[:, 0] = torch.tensor([300.0, 2500.0])
    rad[:, 0] = 2000.0
    for k in range(L):
        pos[:, 1 + k] = torch.tensor([300.0, 130.0 + 25.0 * k])
    anchor = torch.stack([torch.tensor([300.0, 105.0 + 25.0 * k]) for k in range(L)]).expand(B, L, 2) \
        + (u(L, 2) - 0.5)
    pos[:, L + 1] = torch.tensor([180.0, 190.0])                                      # striker
    pos[:, L + 2] = torch.tensor([470.0, 440.0])                                      # X + Rot constrained
    rad[:, L + 2] = 20.0
    pos[:, L + 3] = torch.tensor([120.0, 455.0])                                      # FixedJoint pair
    pos[:, L + 4] = torch.tensor([155.0, 455.0])
    vel = torch.zeros(B, nb, 3, dtype=torch.float64)
    vel[:, 1:L + 1, 1] = (u(L) - 0.5) * 4.0
    vel[:, L + 1] = torch.stack([(u() - 0.5) * 0.4, 140.0 + 20.0 * u(), -30.0 - 10.0 * u()], 1)
    vel[:, L + 2, 2] = 40.0 + 10.0 * u()
    vel[:, L + 3:, 2] = (30.0 + 10.0 * u()).unsqueeze(1)
    vel[:, L + 3:, 1] = ((u() - 0.5) * 10.0).unsqueeze(1)
    mass = 0.5 + u(nb)
    mass[:, 0] = 1.0
    fric = 0.2 + 0.7 * u(nb)
    rest = 0.2 + 0.5 * u(nb)
    out = dict(pos=pos, vel=vel, rad=rad, mass=mass, fric=fric, rest=rest, anchor=anchor)
    return {k_: t.to(dtype) for k_, t in out.items()}


def joint_chain_specs(anchor, joints=True):
    """(joints, no_contact) of make_joint_chain's scene for anchor [B, links, 2] (BatchedWorld) or [links, 2] (one
    world). joints=False: no joints or constraints (the pins only), the same no-contact pairs."""
    from .constraints import FixedJoint, Joint, RotConstraint, XConstraint
    L = anchor.shape[-2]
    if not joints:
        return [], [(k, k + 1) for k in range(1, L)]
    js = [Joint(1, None, anchor[..., 0, :])]
    js += [Joint(k + 1, k, anchor[..., k, :]) for k in range(1, L)]
    js += [XConstraint(L + 2), RotConstraint(L + 2), FixedJoint(L + 3, L + 4)]
    return js, [(k, k + 1) for k in range(1, L)]
