"""World-steps/s of `BatchedWorld` with joints on the GPU, next to the same bodies without them.

    python scripts/bench_joint_world.py [--B 1024] [--steps 20] [--warmup 5] [--reps 3]
    python scripts/bench_joint_world.py --profile DIR      # torch.profiler trace + the joint kernels' share

Scene: lcp_physics_b200.scenes.make_joint_chain (the scene of tests/golden/bworld_joints.npz): a pinned floor ball,
a 5-link chain hung from a world Joint, a thrown ball, an X + Rot constrained ball and a FixedJoint pair (18
equality rows, 10 bodies). "pins" is the same bodies and no-contact pairs with only the floor pin (3 rows), so the
difference is the cost of the joints: the row kernels, the rows in the solve and the different motion. Both run with
grad off, in fp64 and fp32; each repetition builds both worlds afresh, steps them `warmup` steps untimed and then
times `steps` steps (host clock around work that ends in a device synchronise), alternating the two.
Prints one JSON line per dtype, with the card's name and power limit.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from lcp_physics_b200.scenes import joint_chain_specs, make_joint_chain  # noqa: E402
from lcp_physics_b200.world import BatchedWorld  # noqa: E402


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        idx = torch.cuda.current_device()
        name, power = [s.strip() for s in out[idx].split(",")]
        return name, power
    except Exception as e:                       # the number is still reported, with what could be read
        return torch.cuda.get_device_name(), "unknown (%s)" % type(e).__name__


def make_world(B, dtype, joints, seed=0):
    ic = make_joint_chain(B, seed=seed, dtype=dtype)
    js, nc = joint_chain_specs(ic["anchor"], joints=joints)
    return BatchedWorld(ic["pos"], ic["rad"], vel=ic["vel"], mass=ic["mass"], restitution=ic["rest"],
                        fric_coeff=ic["fric"], gravity=100.0, static=[0], joints=js, no_contact=nc, post_stab=True)


def timed(w, steps):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        w.step()
    torch.cuda.synchronize()
    return time.perf_counter() - t0


def bench(args, dtype):
    rates = {"joints": [], "pins": []}
    for rep in range(args.reps):
        for name in ("joints", "pins") if rep % 2 == 0 else ("pins", "joints"):
            w = make_world(args.B, dtype, name == "joints", seed=rep)
            for _ in range(args.warmup):
                w.step()
            rates[name].append(args.B * args.steps / timed(w, args.steps))
    med = {k: sorted(v)[len(v) // 2] for k, v in rates.items()}
    return dict(dtype=str(dtype).replace("torch.", ""), B=args.B, steps=args.steps, warmup=args.warmup, reps=args.reps,
                joints_world_steps_per_s=round(med["joints"], 1), pins_world_steps_per_s=round(med["pins"], 1),
                joints_over_pins=round(med["joints"] / med["pins"], 3),
                all_joints=[round(x, 1) for x in rates["joints"]], all_pins=[round(x, 1) for x in rates["pins"]])


def profile(args, dtype):
    from torch.profiler import ProfilerActivity, profile as tprof
    w = make_world(args.B, dtype, True)
    for _ in range(args.warmup):
        w.step()
    torch.cuda.synchronize()
    with tprof(activities=[ProfilerActivity.CUDA, ProfilerActivity.CPU]) as prof:
        for _ in range(args.steps):
            w.step()
        torch.cuda.synchronize()
    os.makedirs(args.profile, exist_ok=True)
    tag = str(dtype).replace("torch.", "")
    prof.export_chrome_trace(os.path.join(args.profile, "joint_world_%s.pt.trace.json" % tag))
    kern = {}
    for ev in prof.events():
        if ev.device_type == torch.autograd.DeviceType.CUDA:
            kern[ev.name] = kern.get(ev.name, 0.0) + ev.device_time
    total = sum(kern.values())
    joint = sum(t for k, t in kern.items() if "joint_" in k)
    top = sorted(kern.items(), key=lambda kv: -kv[1])[:8]
    return dict(dtype=tag, B=args.B, steps=args.steps, kernel_time_us=round(total, 1), joint_kernel_time_us=round(joint, 1),
                joint_kernel_share=round(joint / total, 4) if total else None,
                top_kernels=[(k[:60], round(t, 1)) for k, t in top])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--B", type=int, default=1024)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--profile", default=None, help="write torch.profiler traces here and report the joint kernels' share")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_joint_world: needs a CUDA device")
    name, power = card()
    with torch.no_grad():
        for dtype in (torch.float64, torch.float32):
            res = profile(args, dtype) if args.profile else bench(args, dtype)
            res.update(gpu=name, power_limit=power)
            print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
