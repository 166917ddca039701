"""Records trajectories of B independent UNMODIFIED reference `World`s with joints (ode/pygame stubbed,
oracle/ref_shim.py) for `lcp_physics_b200.world.BatchedWorld(joints=..., no_contact=...)` to reproduce:

    python tests/golden/make_joint_world_golden.py        (build container only)

Scene (lcp_physics_b200.scenes.make_joint_chain): a huge pinned floor ball, a chain of overlapping circles hung from
a world `Joint` with neighbouring links jointed (i1 > i2, as in chain_demo) and marked no-contact, a ball thrown at
the chain, a ball held by XConstraint + RotConstraint and a FixedJoint pair falling onto the floor. Constraints in
the order [TotalConstraint(floor)] + joint_chain_specs. Stored per variant (post_stab off / on): the initial
state, the anchors, and p, v, the contact count after every step and the final t.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import ref_shim  # noqa: E402

ref_shim.install_world_stubs()
import lcp_physics.physics.engines as ref_engines  # noqa: E402
from lcp_physics.physics import constraints as rc  # noqa: E402
from lcp_physics.physics.bodies import Circle  # noqa: E402
from lcp_physics.physics.forces import Gravity  # noqa: E402
from lcp_physics.physics.world import World  # noqa: E402

from lcp_physics_b200.scenes import joint_chain_specs, make_joint_chain  # noqa: E402

ref_engines.LCPFunction = ref_shim.ReferenceLCPFunction
OUT = os.path.dirname(os.path.abspath(__file__))
B, STEPS = 5, 40


def run(ic, w, post_stab):
    nb = ic["pos"].shape[1]
    bodies = []
    for k in range(nb):
        c = Circle([float(x) for x in ic["pos"][w, k]], float(ic["rad"][w, k]), vel=tuple(float(x) for x in ic["vel"][w, k]),
                   mass=float(ic["mass"][w, k]), restitution=float(ic["rest"][w, k]), fric_coeff=float(ic["fric"][w, k]))
        if k > 0:
            c.add_force(Gravity(g=100))
        bodies.append(c)
    specs, no_contact = joint_chain_specs(ic["anchor"][w])
    cons = [rc.TotalConstraint(bodies[0])]
    for s in specs:
        kind = type(s).__name__
        if kind == "Joint":
            cons.append(rc.Joint(bodies[s.i1], bodies[s.i2] if s.i2 is not None else None, [float(x) for x in s.pos]))
        elif kind == "FixedJoint":
            cons.append(rc.FixedJoint(bodies[s.i1], bodies[s.i2]))
        else:
            cons.append(getattr(rc, kind)(bodies[s.i1]))
    for i, j in no_contact:
        bodies[i].add_no_contact(bodies[j])
    world = World(bodies, cons, dt=1.0 / 30, post_stab=post_stab)
    P, V, NC, T = [], [], [], []
    for _ in range(STEPS):
        world.step()
        P.append(torch.stack([b.p for b in world.bodies]).detach().numpy().copy())
        V.append(world.v.detach().numpy().reshape(-1, 3).copy())
        NC.append(len(world.contacts))
        T.append(float(world.t))
    return np.stack(P), np.stack(V), np.array(NC), np.array(T)


def main():
    ic = make_joint_chain(B, seed=7)
    blob = {k: v.numpy() for k, v in ic.items()}
    for tag, ps in (("nops", False), ("ps", True)):
        res = [run(ic, w, ps) for w in range(B)]
        blob[tag + "_p"] = np.stack([r[0] for r in res], 1)          # [steps, B, nb, 3]
        blob[tag + "_v"] = np.stack([r[1] for r in res], 1)
        blob[tag + "_nc"] = np.stack([r[2] for r in res], 1)
        blob[tag + "_t"] = np.stack([r[3] for r in res], 1)          # [steps, B]
        halved = int((np.abs(np.diff(np.concatenate([np.zeros((1, B)), blob[tag + "_t"]]), axis=0) - 1.0 / 30) > 1e-12).sum())
        print(tag, "contacts per step (world 0):", res[0][2].tolist(), "steps with dt halving:", halved)
    path = os.path.join(OUT, "bworld_joints.npz")
    np.savez_compressed(path, **blob)
    print("->", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
