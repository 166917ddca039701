"""Constraint specs for `BatchedWorld(joints=...)`: index-based counterparts of the reference's constraint classes
(physics/constraints.py). Bodies are indices into the world's body axis; one list describes the topology of every
scene of the batch, and only a revolute `Joint`'s anchor may differ between scenes.

Rows, in the order of World.Je() (physics/world.py:156-170), with pos1 = (x1, y1) the lever of a revolute joint on
body 1 and pos2 = (x2, y2) = p_b1 + pos1 - p_b2:

    Joint(i1, i2, pos)    2 rows   J1 = [[-y1, 1, 0], [x1, 0, 1]],  J2 = [[y2, -1, 0], [-x2, 0, -1]]  (:29-36)
    FixedJoint(i1, i2)    3 rows   the same with pos1 = 0, plus J1 = [1, 0, 0], J2 = [-1, 0, 0]       (:70-77)
    XConstraint(i)        1 row    [0, 1, 0]
    YConstraint(i)        1 row    [0, 0, 1]
    RotConstraint(i)      1 row    [1, 0, 0]
    TotalConstraint(i)    3 rows   eye(3)
"""
import torch

# row kinds of the row table (csrc/lcp_joints.cuh)
UNIT, LEVER_X, LEVER_Y, ROT = 0, 1, 2, 3


def _index(i, what):
    if isinstance(i, bool) or not isinstance(i, int) or i < 0:
        raise ValueError("%s: body index must be a non-negative int, got %r" % (what, i))
    return i


class _Single:
    rows = ()                         # dofs of body 1 the unit rows constrain

    def __init__(self, i):
        self.i1 = _index(i, type(self).__name__)
        self.i2 = None

    def bodies(self):
        return (self.i1,)

    def __repr__(self):
        return "%s(%d)" % (type(self).__name__, self.i1)


class XConstraint(_Single):
    """Prevents motion along x (constraints.py:122-146)."""
    rows = (1,)


class YConstraint(_Single):
    """Prevents motion along y (constraints.py:95-119)."""
    rows = (2,)


class RotConstraint(_Single):
    """Prevents rotation (constraints.py:149-173)."""
    rows = (0,)


class TotalConstraint(_Single):
    """Prevents all motion (constraints.py:176-192); `BatchedWorld(static=...)` pins are these."""
    rows = (0, 1, 2)


class Joint:
    """Revolute joint between body i1 and body i2 (or the world, i2 = None) at `pos`: [2], or [B, 2] for an anchor per
    scene (constraints.py:13-53). Differentiable w.r.t. `pos` when it requires grad."""

    def __init__(self, i1, i2, pos):
        self.i1 = _index(i1, "Joint")
        self.i2 = None if i2 is None else _index(i2, "Joint")
        if self.i2 == self.i1:
            raise ValueError("Joint: a joint of body %d with itself" % self.i1)
        self.pos = pos if isinstance(pos, torch.Tensor) else torch.as_tensor(pos, dtype=torch.float64)
        if self.pos.shape[-1:] != (2,) or self.pos.dim() not in (1, 2):
            raise ValueError("Joint: pos must be [2] or [B, 2], got shape %s" % (tuple(self.pos.shape),))

    def bodies(self):
        return (self.i1,) if self.i2 is None else (self.i1, self.i2)

    def __repr__(self):
        return "Joint(%d, %s)" % (self.i1, self.i2)


class FixedJoint:
    """Welds body i2 to body i1 (constraints.py:56-92)."""

    def __init__(self, i1, i2=None):
        self.i1 = _index(i1, "FixedJoint")
        if i2 is None:
            raise ValueError("FixedJoint: needs a second body")
        self.i2 = _index(i2, "FixedJoint")
        if self.i2 == self.i1:
            raise ValueError("FixedJoint: a joint of body %d with itself" % self.i1)

    def bodies(self):
        return (self.i1, self.i2)

    def __repr__(self):
        return "FixedJoint(%d, %d)" % (self.i1, self.i2)


SPECS = (Joint, FixedJoint, XConstraint, YConstraint, RotConstraint, TotalConstraint)


def row_table(specs, nb):
    """Host-side row descriptor of a constraint list: (rows, revolute) with rows a list of
    (kind, body1, body2 or -1, aux) -- aux = the dof of a UNIT row, the revolute-joint index of a LEVER row (-1: the
    FixedJoint's pos1 = 0) -- in World.Je() order, and revolute the list of `Joint` specs in the order of their
    state. Raises ValueError for an unknown spec or a body index >= nb."""
    rows, revolute = [], []
    for s in specs:
        if not isinstance(s, SPECS):
            raise ValueError("unknown constraint spec %r" % (s,))
        for i in s.bodies():
            if i >= nb:
                raise ValueError("%r: body index %d out of range (nb = %d)" % (s, i, nb))
        b2 = -1 if s.i2 is None else s.i2
        if isinstance(s, Joint):
            k = len(revolute)
            revolute.append(s)
            rows += [(LEVER_X, s.i1, b2, k), (LEVER_Y, s.i1, b2, k)]
        elif isinstance(s, FixedJoint):
            rows += [(LEVER_X, s.i1, b2, -1), (LEVER_Y, s.i1, b2, -1), (ROT, s.i1, b2, -1)]
        else:
            rows += [(UNIT, s.i1, -1, q) for q in s.rows]
    return rows, revolute


def pair_mask(pairs, nb):
    """Skip mask of `no_contact` pairs over the lexicographic pair index q of (i < j) (the order of
    torch.triu_indices(nb, nb, 1)): (bool [nb (nb - 1) / 2], packed int32 words for lcpb200_find_contacts_masked)."""
    npairs = nb * (nb - 1) // 2
    mask = torch.zeros(npairs, dtype=torch.bool)
    for pr in pairs:
        i, j = (_index(x, "no_contact") for x in pr)
        if i == j or max(i, j) >= nb:
            raise ValueError("no_contact: bad pair (%d, %d) for nb = %d" % (i, j, nb))
        i, j = min(i, j), max(i, j)
        mask[i * (2 * nb - i - 1) // 2 + j - i - 1] = True
    nwords = (npairs + 31) // 32
    bits = torch.zeros(nwords * 32, dtype=torch.int64)
    bits[:npairs] = mask.long()
    words = (bits.reshape(nwords, 32) << torch.arange(32)).sum(1)          # < 2^32
    words = torch.where(words >= 2 ** 31, words - 2 ** 32, words).to(torch.int32)
    return mask, words
