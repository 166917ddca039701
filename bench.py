#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 LCP contact solver.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json `metric`, config "LCPFunction fwd+bwd (implicit diff):
batch=4096, 64 contacts, fp32, 1 GPU"): one STEP = one forward + one backward
(all seven gradients) of `LCPFunction` over a batch of 4096 synthetic contact
scenes per GPU (32 bodies, 64 contacts, 2 friction directions: n = 96,
m = 256, neq = 0, max_iter = 10, fp32). N GPUs: scene-sharded, 4096 scenes per
rank (weak scaling; N = 8 is BASELINE's 32768-scene config), no collective on
the data path, one all_gather of the per-rank loss gradients per step.

Prints ONE JSON line (rank 0). `value` = solves/s with inputs resident in HBM;
`e2e` = same metric through the public API with pinned HOST buffers (H2D of all
inputs and D2H of all results inside the timed region); `roofline` for the
dominant kernel (forward); `cpu_baseline` = the oracle port of the reference's
CPU algorithm on a bounded sample, timed on this box's host cores.

`--impl reference`: times the reference's own CPU implementation (the oracle
port, as-is semantics incl. the per-row Python pivot loop of util.py:86-90) on
rank 0. The Python reference cannot travel to the GPU box; see DESIGN.md.

`--dump-outputs DIR`: after the timed steps, rank 0 writes the results of the
last timed step as DIR/<name>.npy (float32 / float64), so that two builds run
with the same arguments (hence the same seeded inputs) can be compared output
for output. Outputs larger than 64 MB in all are written for a fixed, seeded
sample of the scenes (the same scenes in every array).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

if os.environ.get("OMP_NUM_THREADS") == "1" and "TORCHELASTIC_RUN_ID" in os.environ:
    del os.environ["OMP_NUM_THREADS"]      # torchrun's per-rank default; see use_all_host_threads()
import torch  # noqa: E402

NB, NC, FD, NEQ = 32, 64, 2, 0
N_DOF, M_INEQ = 3 * NB, NC * (2 + FD)
MAX_ITER = 10
METRIC = "LCP solves/sec (LCPFunction fwd+bwd, batch=4096 x 64 contacts, fp32)"
UNIT = "solves/s"

# BASELINE.json configs[1] (--config cfg2): LCPFunction forward only, batch=1024, 32 contacts, 3 friction dirs, fp64
CFG2 = dict(nb=16, nc=32, fd=3, e=0, batch=1024)
METRIC_CFG2 = "LCP solves/sec (LCPFunction forward only, batch=1024 x 32 contacts x 3 fric dirs, fp64)"


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# FP32 / FP64 FMA pipe peaks measured on this pool with scripts/ubench/pipes.cu (record:
# profiles/r02_ubench_pipes_latencies.txt): FFMA 70.5 TFLOP/s (121 FMA/clk/SM), DFMA 36.6 TFLOP/s (63 FMA/clk/SM)
FFMA_PEAK_TFLOPS = 70.5
DFMA_PEAK_TFLOPS = 36.6


def condensed_fp64_flops(n, m_blocks, cs, ucols, iters_mean):
    """FP64 flops the condensed-KKT kernel needs per solve (DESIGN.md section 3): per factorisation an n x n LU
    (2/3 n^3), the block inverses (2 cs^3 each) and the assembly of K (2 cs^2 ucols + 2 cs ucols^2 per block);
    per solve two triangular substitutions (2 n^2) and two block mat-vecs. K + 1 factorisations, 2K + 1 solves."""
    fact = 2.0 / 3 * n ** 3 + m_blocks * (2.0 * cs ** 3 + 2.0 * cs * cs * ucols + 2.0 * cs * ucols * ucols)
    solve = 2.0 * n * n + m_blocks * (4.0 * cs * cs + 4.0 * cs * ucols)
    return (iters_mean + 1) * fact + (2 * iters_mean + 1) * solve


def algorithmic(n, m, e, w, iters_mean):
    """SURVEY.md 8(d): flops and bytes per solve for the dense formulation."""
    K = iters_mean
    W_pre = 2.0 / 3 * n ** 3 + 2.0 * n * n * m + 2.0 * m * m * n
    W_iter = 2.0 / 3 * m ** 3 + 6.0 * m * m + 12.0 * m * n + 10.0 * n * n
    W_init = 2.0 / 3 * m ** 3 + 4.0 * n * n + 4.0 * m * n + 2.0 * m * m
    W_fwd = W_pre + W_init + K * W_iter
    W_bwd = W_pre + 2.0 / 3 * m ** 3 + 4.0 * n * n + 4.0 * m * n + 2.0 * m * m + 2 * (2.0 * m * n + m * m + n * n)
    b_in = (n * n + m * n + m * m + n + m) * w
    b_fwd_resident = b_in + (n + 2 * m) * w
    b_fwd_stream = (K + 1) * (m * m + m * n + n * n) * w      # north_star: block streamed once per factorisation
    b_bwd = b_in + (2 * n + 2 * m) * w + (n * n + m * n + m * m + n + m) * w
    return dict(W_fwd=W_fwd, W_bwd=W_bwd, b_fwd_resident=b_fwd_resident, b_fwd_stream=b_fwd_stream, b_bwd=b_bwd)


class ClockSampler:
    """Samples SM clocks / throttle reasons with nvidia-smi during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.samples, self.stop_flag, self.th = index, [], False, None

    def _run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5)
                parts = [p.strip() for p in out.stdout.strip().split(",")]
                if len(parts) >= 6:
                    self.samples.append(parts)
            except Exception:
                pass
            time.sleep(0.2)

    def start(self):
        self.th = threading.Thread(target=self._run, daemon=True)
        self.th.start()

    def stop(self):
        self.stop_flag = True
        if self.th:
            self.th.join(timeout=6)
        sm = sorted(int(s[0]) for s in self.samples if s[0].isdigit())
        mx = [int(s[1]) for s in self.samples if s[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for s in self.samples for i in range(4) if s[2 + i].lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


DUMP_BYTES = 60 * 10 ** 6           # array data of --dump-outputs; leaves room for the .npy headers under 64 MB


def dump_outputs(path, arrays):
    """Writes `arrays` (name -> tensor with the scene index first, or None) as path/<name>.npy. Integer outputs
    become float64 (exact). When every scene does not fit in DUMP_BYTES, all arrays keep the same scenes: a sorted
    sample drawn with a fixed seed."""
    import numpy as np
    arrays = {k: v.detach() for k, v in arrays.items() if v is not None}
    arrays = {k: (v if v.dtype in (torch.float32, torch.float64) else v.double()) for k, v in arrays.items()}
    B = next(iter(arrays.values())).shape[0]
    per_scene = sum(v[0].numel() * v.element_size() for v in arrays.values())
    k = min(B, DUMP_BYTES // per_scene)
    idx = torch.randperm(B, generator=torch.Generator().manual_seed(0))[:k].sort().values if k < B else None
    os.makedirs(path, exist_ok=True)
    for name, v in arrays.items():
        v = v.cpu() if idx is None else v.index_select(0, idx.to(v.device)).cpu()
        np.save(os.path.join(path, name + ".npy"), v.numpy())
    print("bench: wrote %d arrays of %d of %d scenes to %s" % (len(arrays), k, B, path), file=sys.stderr, flush=True)


WORKLOAD = ("LCPFunction fwd+bwd (all 7 gradients), batch=%d scenes/GPU x 64 contacts x 2 fric dirs "
            "(n=96, m=256, neq=0), fp32, max_iter=10, pile scenes (lcp_physics_b200/scenes.py)")


def use_all_host_threads():
    """Threads the CPU legs run with. torchrun exports OMP_NUM_THREADS=1 for every rank; that default is
    dropped at the top of this file (before torch is imported) so that the CPU legs get torch's own
    default = all host cores, exactly as in a plain `python bench.py` run. (Calling
    torch.set_num_threads() after import instead dead-locked MKL's threaded SLASWP in this image.)"""
    return torch.get_num_threads()


def cpu_reference_leg(B_sample, dtype, seed, reps=1, cfg2=False, unpack="loop"):
    """Oracle port of the reference CPU path on B_sample scenes: fwd+bwd (cfg3) or forward (cfg2). unpack="loop": as-is
    semantics (the reference's per-row Python pivot loop, util.py:86-90); "vec": the same arithmetic with that loop
    vectorised over the batch (the "modern torch" restatement SURVEY.md section 8d asks to report next to it)."""
    from oracle import pdipm_oracle as po
    from lcp_physics_b200.scenes import make_scenes
    nb, nc, fd, e = (CFG2["nb"], CFG2["nc"], CFG2["fd"], CFG2["e"]) if cfg2 else (NB, NC, FD, NEQ)
    inp = make_scenes(B_sample, nb, nc, fd=fd, e=e, dtype=dtype, seed=seed)
    g = torch.randn(B_sample, 3 * nb, dtype=dtype, generator=torch.Generator().manual_seed(seed))
    small = tuple(t[:4] if t.dim() > 1 else t for t in inp)
    po.lcp_backward(po.lcp_forward(*small, max_iter=MAX_ITER, unpack=unpack), g[:4])   # warm-up
    t0 = time.perf_counter()
    for _ in range(reps):
        res = po.lcp_forward(*inp, max_iter=MAX_ITER, unpack=unpack)
        if not cfg2:
            po.lcp_backward(res, g)
    dt = (time.perf_counter() - t0) / reps
    return B_sample / dt, dt


def run_reference(args, rank, world):
    if rank != 0:
        return
    if args.config == "cfg4":
        ow = cfg4_oracle_world(cfg4_initial(1, 0))
        for _ in range(min(args.warmup, 1)):                      # ~20 s per step on 8 cores: one warm-up step at most
            ow.step()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            ow.step()
        dt = time.perf_counter() - t0
        val = args.steps / dt
        print(json.dumps({"impl": "reference", "metric": METRIC_CFG4, "value": val, "unit": "steps/s", "n_gpus": world,
                          "steps": args.steps, "warmup": min(args.warmup, 1), "ms_per_step": dt / args.steps * 1e3,
                          "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                          "config": {"workload": WORKLOAD_CFG4, "worlds": 1, "parallelism": "host CPU, rank 0 only"},
                          "cpu_baseline": {"value": val, "unit": "steps/s", "cores": use_all_host_threads(), "kind": "port",
                                           "sample": "%d steps of the 512-ball pile (oracle/world_oracle.py: restatement of "
                                                     "World.step_dt, LCP by the oracle port, m = 4 x %d contacts)"
                                                     % (args.steps, len(ow.contacts))},
                          "e2e": {"value": val, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                          "gpu_launches": 0}), flush=True)
        return
    if args.config == "world":
        from oracle.world_oracle import OracleCircleWorld
        ic = world_initial(1, 0)
        ow = OracleCircleWorld(ic["pos"][0], ic["rad"][0], ic["vel"][0], ic["mass"][0], ic["rest"][0], ic["fric"][0],
                               gravity=100.0, static=(0,), dt=1.0 / 30)
        for _ in range(args.warmup):
            ow.step()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            ow.step()
        dt = time.perf_counter() - t0
        val = args.steps / dt
        print(json.dumps({"impl": "reference", "metric": METRIC_WORLD, "value": val, "unit": "world-steps/s", "n_gpus": world,
                          "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
                          "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                          "config": {"workload": "one world (pile of 24 balls in contact on a pinned floor ball) stepped on the host"},
                          "cpu_baseline": {"value": val, "unit": "world-steps/s", "cores": use_all_host_threads(), "kind": "port",
                                           "sample": "1 world, %d steps (oracle/world_oracle.py)" % args.steps},
                          "e2e": {"value": val, "unit": "world-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                          "gpu_launches": 0}), flush=True)
        return
    cores = use_all_host_threads()
    Bs = args.ref_batch
    cfg2 = args.config == "cfg2"
    rdt = torch.float64 if cfg2 else torch.float32
    full_batch = args.batch or (CFG2["batch"] if cfg2 else 4096)
    for _ in range(args.warmup and 1):
        cpu_reference_leg(8, rdt, 1, cfg2=cfg2)
    t0 = time.perf_counter()
    for k in range(args.steps):
        cpu_reference_leg(Bs, rdt, 100 + k, cfg2=cfg2)
    dt = time.perf_counter() - t0
    val = Bs * args.steps / dt
    vec_val, _ = cpu_reference_leg(Bs, rdt, 100, cfg2=cfg2, unpack="vec")
    line = {
        "impl": "reference", "metric": METRIC_CFG2 if cfg2 else METRIC, "value": val, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64" if cfg2 else "f32", "data": "synthetic",
        "config": {"workload": (METRIC_CFG2 if cfg2 else WORKLOAD % full_batch), "global_batch": world * full_batch,
                   "parallelism": "host CPU, rank 0 only", "sample_batch": Bs,
                   "note": "each step times a bounded sample of the workload (sample_batch scenes) on the host cores"},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": "%d scenes per step (of the %d-scene batch), %s, as-is reference "
                                   "semantics incl. util.py:86-90 pivot loop" % (Bs, full_batch, "forward" if cfg2 else "fwd+bwd"),
                         "vectorised_restatement_value": vec_val,
                         "vectorised_note": "same arithmetic with the per-row Python pivot loop vectorised over the batch "
                                            "(oracle unpack='vec'), one %d-scene sample" % Bs},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def parity_sample(inp_host, g_host, fo_dev, bo_dev, n_sample, dtype, max_iter, with_backward):
    """Real parity on the first n_sample scenes of the TIMED batch (rank 0): the oracle port of the reference in
    the run's dtype (the reference's own answer) and in fp64 (the truth), against what the GPU returned.
    Also returns the CPU timing of the as-is oracle run (the cpu_baseline of the same scenes)."""
    from oracle import pdipm_oracle as po
    sub = tuple(t[:n_sample].clone() if t.dim() > 1 else t for t in inp_host)
    g = g_host[:n_sample]
    t0 = time.perf_counter()
    res = po.lcp_forward(*sub, max_iter=max_iter, unpack="loop")          # as-is reference semantics
    rg = po.lcp_backward(res, g) if with_backward else None
    dt = time.perf_counter() - t0
    sub64 = tuple(t.double() for t in sub)
    res64 = po.lcp_forward(*sub64, max_iter=max_iter)

    def rel(a, b_):
        a = a.double().reshape(a.shape[0], -1); b_ = b_.double().reshape(b_.shape[0], -1)
        return (a - b_).norm(dim=1) / b_.norm(dim=1).clamp_min(1e-300)

    def stats(e):
        return {"frac_within_tol": float((e < TOL[dtype]).float().mean()), "median": float(e.median()),
                "p90": float(e.quantile(0.9)), "max": float(e.max())}

    z = fo_dev[0][:n_sample].cpu()
    out = {"n": n_sample, "tol": TOL[dtype],
           "zhat_vs_reference": stats(rel(z, res.zhat)),
           "zhat_vs_fp64": stats(rel(z, res64.zhat)),
           "reference_vs_fp64": stats(rel(res.zhat, res64.zhat))}
    if with_backward:
        # gradient truth: the fp64 oracle on the state the GPU forward returned (the backward map itself)
        st = [None if t is None else t[:n_sample].double().cpu() for t in (fo_dev[0], fo_dev[1], fo_dev[2], fo_dev[3])]
        truth = po.lcp_backward_from_saved(sub64, st[0], st[1], st[2], st[3], g.double())
        out["dp_vs_fp64_same_state"] = stats(rel(bo_dev[1][:n_sample].cpu(), truth[1]))
        out["dQ_vs_fp64_same_state"] = stats(rel(bo_dev[0][:n_sample].cpu(), truth[0]))
        out["dG_vs_fp64_same_state"] = stats(rel(bo_dev[2][:n_sample].cpu(), truth[2]))
        out["reference_dp_vs_fp64_own_state"] = stats(rel(rg[1], po.lcp_backward(res64, g.double())[1]))
    return out, n_sample / dt, dt


TOL = {torch.float32: 1e-3, torch.float64: 1e-6}

METRIC_WORLD = "sim steps/sec (World.step: pile of 24 balls on a pinned floor ball, 2 fric dirs, fp64; B worlds in lock-step)"


def world_initial(B, seed):
    """--config world: B piles of 24 balls (6 wide, hexagonal, 0.05 apart: ~55 contacts per world from step 0,
    m ~ 220) on a pinned floor ball; every world has its own jitter."""
    from lcp_physics_b200.scenes import make_ball_pile
    return make_ball_pile(B, nballs=24, cols=6, seed=2000 + seed, gap=0.05)


def run_world(args, rank, world, local_rank):
    """--config world: `BatchedWorld.step()` (contact generation + fused engine kernels + dt halving) over B worlds
    per GPU; value = world-steps per second. CPU baseline: the oracle restatement of the reference's World.step_dt
    (oracle/world_oracle.py, one world) on the first world of the batch, which also gives the parity figure."""
    import torch.distributed as dist
    from lcp_physics_b200 import _lib
    from lcp_physics_b200.world import BatchedWorld
    _lib.require_cuda()
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    B = args.batch or 1024
    ic = world_initial(B, rank)

    def mk():
        return BatchedWorld(ic["pos"], ic["rad"], vel=ic["vel"], mass=ic["mass"], restitution=ic["rest"],
                            fric_coeff=ic["fric"], gravity=100.0, static=[0], dt=1.0 / 30, device=dev)

    w_ = mk()
    for _ in range(args.warmup):
        w_.step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    ncs = []
    for _ in range(args.steps):
        w_.step()
        ncs.append(w_.counts.float().mean())
    e1.record()
    torch.cuda.synchronize()
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"p": w_.p, "v": w_.v, "t": w_.t, "contacts": w_.counts})
    ms = e0.elapsed_time(e1)
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = t.item()
    # e2e: initial conditions in (pinned) host memory every step-block: upload, K steps, positions back
    hp = {k: v.pin_memory() for k, v in ic.items()}
    t0 = time.perf_counter()
    w2 = BatchedWorld(hp["pos"], hp["rad"], vel=hp["vel"], mass=hp["mass"], restitution=hp["rest"], fric_coeff=hp["fric"],
                      gravity=100.0, static=[0], dt=1.0 / 30, device=dev)
    out_p = torch.empty(B, w_.nb, 3, dtype=torch.float64).pin_memory()
    for _ in range(args.steps):
        w2.step()
        out_p.copy_(w2.p)                                         # the step's result back to the host, every step
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    if rank != 0:
        return
    line = {"metric": METRIC_WORLD, "value": world * B * args.steps / (ms * 1e-3), "unit": "world-steps/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "BatchedWorld.step(): %d worlds/GPU x (pile of 24 balls in contact + pinned floor ball), n=75, <= 75 contacts, "
                                   "fp64, max_iter=10, per-scene contact sets and dt halving" % B,
                       "global_batch": world * B, "parallelism": "world-sharded x%d" % world,
                       "mean_contacts_per_world": float(torch.stack(ncs).mean())},
            "e2e": {"value": world * B * args.steps / e2e_s, "unit": "world-steps/s",
                    "h2d_bytes_per_step": sum(v.numel() * 8 for v in ic.values()) // max(1, args.steps),
                    "d2h_bytes_per_step": out_p.numel() * 8,
                    "api": "BatchedWorld(pinned host tensors) once, then every step: step() + positions of all bodies "
                           "back to pinned host memory"},
            "gpu_launches": 2 * args.steps, "clocks": clocks}
    if world == 1 and not args.no_cpu_baseline:
        from oracle.world_oracle import OracleCircleWorld
        ow = OracleCircleWorld(ic["pos"][0], ic["rad"][0], ic["vel"][0], ic["mass"][0], ic["rest"][0], ic["fric"][0],
                               gravity=100.0, static=(0,), dt=1.0 / 30)
        wg = mk()
        nst = min(args.warmup + args.steps, 40)
        t0 = time.perf_counter()
        worst = 0.0
        for _ in range(nst):
            ow.step()
        dt_cpu = time.perf_counter() - t0
        for _ in range(nst):
            wg.step()
        worst = float((wg.p[0].cpu() - ow.p).abs().max())
        line["parity"] = {"n": 1, "steps": nst, "max_abs_position_error_vs_oracle_world": worst}
        line["cpu_baseline"] = {"value": nst / dt_cpu, "unit": "world-steps/s", "cores": use_all_host_threads(), "kind": "port",
                                "sample": "world 0 of the batch, %d steps, %.1f s (oracle/world_oracle.py: restatement of "
                                          "World.step_dt, LCP by the oracle port)" % (nst, dt_cpu)}
    print(json.dumps(line), flush=True)


# BASELINE.json configs[3] (--config cfg4): "World.step() loop: 512-body ball pile, 2 friction dirs, 1000 steps, 1 GPU"
CFG4 = dict(nballs=512, cols=32, gap=0.05, gravity=100.0)
METRIC_CFG4 = "sim steps/sec (World.step() loop, 512-body ball pile, 2 friction dirs, fp64)"
WORKLOAD_CFG4 = ("BatchedWorld.step() on a pile of 512 balls (radius 10, hexagonal, 32 wide, 0.05 apart: in contact from "
                 "step 0) resting on a pinned floor ball: n = 1539, ~1450 contacts (m ~ 5800), 2 friction dirs, "
                 "max_iter = 10, dt = 1/30, fp64; contact generation + LCP + dt halving every step")


def cfg4_initial(B, seed):
    from lcp_physics_b200.scenes import make_ball_pile
    return make_ball_pile(B, nballs=CFG4["nballs"], cols=CFG4["cols"], seed=3000 + seed, gap=CFG4["gap"])


def cfg4_oracle_world(ic, k=0):
    from oracle.world_oracle import OracleCircleWorld
    return OracleCircleWorld(ic["pos"][k], ic["rad"][k], ic["vel"][k], ic["mass"][k], ic["rest"][k], ic["fric"][k],
                             gravity=CFG4["gravity"], static=(0,), dt=1.0 / 30)


def run_cfg4(args, rank, world, local_rank):
    """--config cfg4: the reference's `World.step()` loop on ONE large scene per GPU (`--batch B`: B such worlds per
    GPU, one CTA each). value = world steps per second (B x steps / time). Every step = batched contact
    generation (torch ops on the device), one banded-kernel LCP (csrc/lcp_banded.cuh) and the dt-halving loop of
    world.py:88-107. CPU arm: the oracle restatement of World.step_dt on the same initial condition (one step,
    ~20 s on 8 cores), which also gives the parity figure."""
    import torch.distributed as dist
    from lcp_physics_b200 import _lib
    from lcp_physics_b200 import engines as _eng
    from lcp_physics_b200.world import BatchedWorld
    _lib.require_cuda()
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    B = args.batch or 1
    ic = cfg4_initial(B, rank)

    def mk(src):
        return BatchedWorld(src["pos"], src["rad"], vel=src["vel"], mass=src["mass"], restitution=src["rest"],
                            fric_coeff=src["fric"], gravity=CFG4["gravity"], static=[0], dt=1.0 / 30, device=dev,
                            contact_capacity=4 * CFG4["nballs"])

    w_ = mk(ic)
    for _ in range(args.warmup):
        w_.step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    ncs, its = [], []
    for _ in range(args.steps):
        w_.step()
        ncs.append(w_.counts.float().mean())
        its.append(_eng.last_solve_info()["iters"].float().mean())
    e1.record()
    torch.cuda.synchronize()
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"p": w_.p, "v": w_.v, "t": w_.t, "contacts": w_.counts})
    ms = e0.elapsed_time(e1)
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = t.item()
    # the LCP kernel alone (one launch per step): solve_dynamics on the current state, CUDA events
    k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    w_.solve_dynamics(w_.dt)
    k0.record()
    for _ in range(5):
        w_.solve_dynamics(w_.dt)
    k1.record()
    torch.cuda.synchronize()
    kernel_ms = k0.elapsed_time(k1) / 5
    info = _eng.last_solve_info()
    iters_k = float(info["iters"].float().mean())
    hd = _lib.get_handle(torch.float64, w_.n, 4 * w_.cap, w_.ne, dev.index, torch.cuda.current_stream(dev).cuda_stream)
    hd.profile(True)
    w_.solve_dynamics(w_.dt)
    torch.cuda.synchronize()
    prof = hd.profile(False)
    bw = prof["c_gradients"] / B                                   # half bandwidth of the ordered condensed matrix (debug counter)
    # e2e: initial conditions in pinned host memory -> upload, K steps, positions back
    hp = {k: v.pin_memory() for k, v in ic.items()}
    out_p = torch.empty(B, CFG4["nballs"] + 1, 3, dtype=torch.float64).pin_memory()
    t0 = time.perf_counter()
    w2 = mk(hp)
    for _ in range(args.steps):
        w2.step()
        out_p.copy_(w2.p)                                         # the step's result (rot, x, y of every body) back to the host
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    if rank != 0:
        return
    N = w_.n + w_.ne
    wband = bw + 16                                               # band + border rows each pass touches
    nfac, nsub = iters_k + 1, 2 * iters_k + 1
    flops = nfac * 2.0 * N * wband * wband + nsub * 4.0 * N * wband      # banded LU (2 N w^2) + substitutions (4 N w)
    dense_flops = nfac * (2.0 / 3.0) * (4.0 * float(torch.stack(ncs).mean())) ** 3   # the reference's m x m LU, per solve
    sms = min(B, torch.cuda.get_device_properties(dev).multi_processor_count)
    ach = flops * B / (kernel_ms * 1e-3) / 1e12
    line = {"metric": METRIC_CFG4, "value": world * B * args.steps / (ms * 1e-3), "unit": "steps/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD_CFG4, "worlds_per_gpu": B, "global_worlds": world * B,
                       "parallelism": "replicas x%d (one scene does not shard)" % world,
                       "mean_contacts": float(torch.stack(ncs).mean()), "mean_pdipm_iters": float(torch.stack(its).mean()),
                       "contacts_min_max_over_steps": [float(torch.stack(ncs).min()), float(torch.stack(ncs).max())],
                       "n_m_e": [3 * (CFG4["nballs"] + 1), "4 x contacts", 3],
                       "l2": "working set per world (factors + band, ~8 MB) is L2 resident by design; inputs are 60 KB"},
            "kernel": {"name": "band_forward_kernel", "ms_per_launch": kernel_ms, "launches_per_step": 1,
                       "share_of_step": kernel_ms / (ms / args.steps), "half_bandwidth": bw, "order": N,
                       "pdipm_iters": iters_k},
            "roofline": {"bound": "fma", "achieved": ach, "peak": DFMA_PEAK_TFLOPS, "unit": "TFLOP/s", "frac": ach / DFMA_PEAK_TFLOPS,
                         "sms_used": sms, "frac_of_sms_used": ach / (DFMA_PEAK_TFLOPS * sms / 148.0),
                         "traffic": None,
                         "note": "achieved = executed banded fp64 flops (2 N w^2 per LU, 4 N w per substitution, w = half "
                                 "bandwidth + 16 border rows) / kernel time; one CTA per world, so one world uses one SM; "
                                 "peak = measured DFMA pipe peak of the whole GPU",
                         "reference_formulation_tflops": dense_flops * B / (kernel_ms * 1e-3) / 1e12},
            "e2e": {"value": world * B * args.steps / e2e_s, "unit": "steps/s",
                    "h2d_bytes_per_step": sum(v.numel() * 8 for v in ic.values()) // max(1, args.steps),
                    "d2h_bytes_per_step": out_p.numel() * 8,
                    "api": "BatchedWorld(pinned host tensors) once, then every step: step() + positions of all bodies "
                           "back to pinned host memory"},
            "gpu_launches": 2 * args.steps, "clocks": clocks}
    if world == 1 and not args.no_cpu_baseline:
        ow = cfg4_oracle_world(ic)
        wg = mk({k: v[:1] for k, v in ic.items()})
        t0 = time.perf_counter()
        ow.step()
        dt_cpu = time.perf_counter() - t0
        wg.step()
        line["parity"] = {"n": 1, "steps": 1, "contacts": [int(wg.counts[0]), len(ow.contacts)],
                          "max_abs_position_error_vs_oracle_world": float((wg.p[0].cpu() - ow.p).abs().max()),
                          "max_abs_velocity_error_vs_oracle_world": float((wg.v[0].cpu() - ow.v).abs().max())}
        line["cpu_baseline"] = {"value": 1.0 / dt_cpu, "unit": "steps/s", "cores": use_all_host_threads(), "kind": "port",
                                "sample": "1 step of world 0 (%d contacts), %.1f s (oracle/world_oracle.py: restatement of "
                                          "World.step_dt, LCP by the oracle port)" % (len(ow.contacts), dt_cpu)}
    print(json.dumps(line), flush=True)


def engine_path_leg(B, rank, dev, g, steps, warmup, barrier, world):
    """cfg 3's scenes (same seed, hence the same LCPs) solved from their contact structure-of-arrays:
    forward + backward (9 gradients w.r.t. the contact list). `value`: SoA resident in HBM; `e2e`: SoA in pinned
    host memory, H2D + D2H of every result inside the timed region (a few KB per scene instead of 0.8 MB)."""
    import torch.distributed as dist
    from lcp_physics_b200.engines import engine_solve
    from lcp_physics_b200.scenes import make_contact_soa
    soa = make_contact_soa(B, NB, NC, seed=1000 + rank, dtype=torch.float64)
    fext = torch.zeros(B, 3 * NB, dtype=torch.float64)
    fext[:, 2::3] = 10.0 * soa["mass"]
    names = ["mass", "inertia", "v", "fext", "normal", "p1", "p2", "mu", "restitution"]
    host = {k: (fext if k == "fext" else soa[k]).float().pin_memory() for k in names}
    b1, b2 = soa["body1"].to(dev), soa["body2"].to(dev)
    devt = {k: host[k].to(dev) for k in names}

    def step(src, to_host):
        lv = [src[k].to(dev, non_blocking=True).requires_grad_(True) for k in names]
        z, status = engine_solve(*lv, b1, b2, 1.0 / 30, max_iter=MAX_ITER)
        (z * g).sum().backward()
        if to_host:
            return [z.detach().cpu()] + [t.grad.cpu() for t in lv]
        return None

    for _ in range(max(1, warmup)):
        step(devt, False)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step(devt, False)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    step(host, True)
    barrier()
    n_e2e = max(1, min(steps, 3))
    t0 = time.perf_counter()
    for _ in range(n_e2e):
        step(host, True)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    t = torch.tensor([ms, e2e_s], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, e2e_s = t.tolist()
    per_scene = sum(host[k][0].numel() for k in names) * 4
    return {"api": "lcp_physics_b200.engines.engine_solve (lcpb200_engine_forward/_backward), fwd+bwd, same scenes as the headline",
            "value": world * B * steps / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms / steps,
            "e2e": {"value": world * B * n_e2e / e2e_s, "unit": UNIT,
                    "h2d_bytes_per_step": per_scene * B, "d2h_bytes_per_step": (per_scene + 3 * NB * 4) * B}}


def run_b200(args, rank, world, local_rank):
    import torch.distributed as dist
    from lcp_physics_b200 import _lib, solve_forward, solve_backward
    from lcp_physics_b200.scenes import make_scenes
    from lcp_physics_b200.sharding import gather_loss_gradients

    _lib.require_cuda()
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    cfg2 = args.config == "cfg2"
    if cfg2:
        nb, nc, fd, neq = CFG2["nb"], CFG2["nc"], CFG2["fd"], CFG2["e"]
        B = args.batch or CFG2["batch"]
        dtype, w, with_bwd, metric = torch.float64, 8, False, METRIC_CFG2
        workload = ("LCPFunction forward only, batch=%d scenes/GPU x 32 contacts x 3 fric dirs (n=48, m=160, neq=0), "
                    "fp64, max_iter=10, pile scenes (lcp_physics_b200/scenes.py)" % B)
    else:
        nb, nc, fd, neq = NB, NC, FD, NEQ
        B = args.batch or 4096
        dtype, w, with_bwd, metric = torch.float32, 4, True, METRIC
        workload = WORKLOAD % B
    n_dof, m_ineq = 3 * nb, nc * (2 + fd)

    inp_host = make_scenes(B, nb, nc, fd=fd, e=neq, dtype=dtype, seed=1000 + rank)
    g_host = torch.randn(B, n_dof, dtype=dtype, generator=torch.Generator().manual_seed(rank))
    inp = tuple(t.to(dev) for t in inp_host)
    g = g_host.to(dev)
    Q, p, G, h, A, b, F = inp

    def mk_fwd_out(device, pin=False):
        kw = dict(device=device, pin_memory=pin)
        return (torch.empty(B, n_dof, dtype=dtype, **kw), None, torch.empty(B, m_ineq, dtype=dtype, **kw),
                torch.empty(B, m_ineq, dtype=dtype, **kw), torch.empty(B, dtype=torch.int32, **kw),
                torch.empty(B, dtype=torch.int32, **kw), torch.empty(B, dtype=dtype, **kw))

    def mk_bwd_out(device, pin=False):
        kw = dict(device=device, pin_memory=pin, dtype=dtype)
        return (torch.empty(B, n_dof, n_dof, **kw), torch.empty(B, n_dof, **kw), torch.empty(B, m_ineq, n_dof, **kw),
                torch.empty(B, m_ineq, **kw), None, None, torch.empty(B, m_ineq, m_ineq, **kw))

    fo = mk_fwd_out(dev)
    bo = mk_bwd_out(dev) if with_bwd else None
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    kev = []

    def step(record=False):
        if record:
            e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
            e0.record()
        saved = {}
        solve_forward(Q, p, G, h, A, b, F, max_iter=MAX_ITER, out=fo, save=saved)
        if record:
            e1.record()
        if with_bwd:
            solve_backward(Q, G, A, F, fo[0], None, fo[2], fo[3], g, out=bo, saved=saved)   # as LCPFunction.backward does
        if record:
            e2.record()
            kev.append((e0, e1, e2))
        if world > 1 and with_bwd:
            # the path's only exchange: gather per-rank loss gradients (here d loss / d p and d h summed over scenes)
            local = torch.cat([bo[1].sum(0), bo[3].sum(0)])
            gather_loss_gradients(local)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ev[0].record()
    for _ in range(args.steps):
        step(record=True)
    ev[1].record()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        names = ("zhat", None, "lam", "slack", "status", "iters", "resid")
        outs = {n: t for n, t in zip(names, fo) if n}
        if with_bwd:
            outs.update(zip(("grad_Q", "grad_p", "grad_G", "grad_h", "grad_A", "grad_b", "grad_F"), bo))
        dump_outputs(args.dump_outputs, outs)
    ms_total = ev[0].elapsed_time(ev[1])
    t = torch.tensor([ms_total], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = t.item()
    fwd_ms = sum(a.elapsed_time(b_) for a, b_, _ in kev) / len(kev)
    bwd_ms = sum(b_.elapsed_time(c) for _, b_, c in kev) / len(kev)
    iters_mean = fo[5].float().mean().item()
    finite_ok = bool(torch.isfinite(fo[0]).all()) and bool((fo[4] >= 0).all())

    # ---- e2e: public API with pinned host buffers (H2D inputs + D2H results inside the timed region)
    pin = lambda t_: t_.pin_memory() if t_.numel() else t_
    hin = tuple(pin(t_) for t_ in inp_host)
    hg = pin(g_host)
    hfo = mk_fwd_out("cpu", pin=True)
    hbo = mk_bwd_out("cpu", pin=True) if with_bwd else None
    hsaved = {}

    def e2e_step():
        solve_forward(*hin, max_iter=MAX_ITER, out=hfo, save=hsaved)
        if with_bwd:
            solve_backward(hin[0], hin[2], hin[4], hin[6], hfo[0], None, hfo[2], hfo[3], hg, out=hbo, saved=hsaved)

    e2e_steps = max(1, min(args.steps, 3))
    e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    t = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_s = t.item()
    # the same through the same API with the gradients in FACTORED form: solve_backward(need=...) returns only
    # dp (= dx), dh (= -dlam), db (= -dnu); dQ, dG, dF, dA are outer products of these with the forward's
    # zhat / lam / nu (lcp.py:52-63), so a consumer that chains them further (like the engine's assembly adjoint)
    # never needs the 0.4 MB per scene of dense gradients on the host
    e2e_f_s = None
    if with_bwd:
        need_f = (False, True, False, True, False, neq > 0, False)
        hbo_f = [hbo[k] if need_f[k] else None for k in range(7)]

        def e2e_step_f():
            solve_forward(*hin, max_iter=MAX_ITER, out=hfo, save=hsaved)
            solve_backward(hin[0], hin[2], hin[4], hin[6], hfo[0], None, hfo[2], hfo[3], hg, need=need_f, out=hbo_f,
                           saved=hsaved)

        e2e_step_f()
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            e2e_step_f()
        torch.cuda.synchronize()
        t = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_f_s = t.item()
    in_bytes = sum(t_.numel() * w for t_ in inp_host)
    h2d = in_bytes + (n_dof * w * B if with_bwd else 0)     # the 7 inputs once (kept on the device) + dl_dzhat
    d2h = ((n_dof + 2 * m_ineq + 1) * w + 8) * B + (in_bytes if with_bwd else 0)   # zhat, lam, slack, resid, status, iters (+ the 7 gradients)

    # ---- the same scenes through the fused engine entry points (contact list in, gradients w.r.t. the contact
    # list out: lcpb200_engine_forward / _backward) -- what B200PdipmEngine calls; reported next to the headline
    eng = None
    if not cfg2:
        eng = engine_path_leg(B, rank, dev, g, args.steps, args.warmup, barrier, world)

    if rank != 0:
        return
    alg = algorithmic(n_dof, m_ineq, neq, w, iters_mean)
    peak, peak_src = load_peaks()
    stream_gbs = alg["b_fwd_stream"] * B / (fwd_ms * 1e-3) / 1e9
    dense_tflops = alg["W_fwd"] * B / (fwd_ms * 1e-3) / 1e12
    fma_peak = DFMA_PEAK_TFLOPS if cfg2 else FFMA_PEAK_TFLOPS
    c64 = condensed_fp64_flops(n_dof, nc, 2 + fd, 6, iters_mean) * B / (fwd_ms * 1e-3) / 1e12
    step_bytes = alg["b_fwd_resident"] + (alg["b_bwd"] if with_bwd else 0)
    kern = "cond_forward_kernel<%s, %d>" % ("double" if cfg2 else "float", 3 if cfg2 else 6)
    line = {
        "metric": metric, "value": world * B * args.steps / (ms_total * 1e-3), "unit": UNIT, "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_total / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64" if cfg2 else "f32 I/O and iterates; the condensed n x n KKT matrix is formed, factored and solved in f64",
        "data": "synthetic",
        "config": {"workload": workload,
                   "global_batch": world * B, "parallelism": "scene-sharded x%d" % world,
                   "l2": "inputs%s per step (%.1f GB) exceed the 126 MB L2, no flush needed"
                         % (" + gradients" if with_bwd else "", step_bytes * B / 1e9),
                   "mean_pdipm_iters": iters_mean, "finite_ok": finite_ok},
        "e2e": {"value": world * B * e2e_steps / e2e_s, "unit": UNIT, "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": d2h, "steps": e2e_steps,
                "api": "solve_forward%s on pinned CPU tensors -> lcpb200_forward_host%s"
                       % (("/solve_backward", "/backward_host") if with_bwd else ("", "")),
                "pcie_note": "dense host tensors: %.2f GB H2D + %.2f GB D2H per step bound this number, not the kernels"
                             % (h2d / 1e9, d2h / 1e9)},
        "gpu_launches": (4 if with_bwd else 2) * args.steps,
        "kernels": {"forward_ms (cond_forward_kernel + dual-form fallback launch)": fwd_ms,
                    "backward_ms (cond_backward_kernel + dual-form fallback launch)": bwd_ms if with_bwd else None},
        "roofline": {"bound": "fma", "kernel": kern,
                     "achieved": dense_tflops, "peak": fma_peak, "unit": "TFLOP/s", "frac": dense_tflops / fma_peak,
                     "traffic": measured_traffic(B, "cfg2" if cfg2 else "cfg3"),
                     "peak_source": "%s FMA pipe measured on this pool (scripts/ubench/pipes.cu, profiles/r02_ubench_pipes_latencies.txt)"
                                    % ("FP64" if cfg2 else "FP32"),
                     "definition": "ALGORITHMIC flops of the reference's dense dual formulation (SURVEY 8d: W_fwd, %.1f MFLOP/solve "
                                   "at the measured iteration count) / forward time / the FMA-pipe peak of the I/O dtype. The kernel "
                                   "reaches the same iterates through the condensed n x n system in fp64 and executes far fewer flops; "
                                   "see fp64_pipe for the executed work" % (alg["W_fwd"] / 1e6),
                     "fp64_pipe": {"achieved_tflops": c64, "peak_tflops": DFMA_PEAK_TFLOPS, "frac": c64 / DFMA_PEAK_TFLOPS,
                                   "note": "necessary fp64 flops of the condensed formulation (LU 2/3 n^3 per factorisation + block "
                                           "inverses + assembly + substitutions) / forward time / measured DFMA peak"},
                     "hbm_per_iteration": {"achieved_gbs": stream_gbs, "peak_gbs": peak, "frac": stream_gbs / peak,
                                           "peak_source": peak_src,
                                           "definition": "north_star per-iteration HBM roofline: (K+1) x (m^2+mn+n^2) x w bytes per "
                                                         "solve (the dense KKT block streamed once per factorisation) / forward time"},
                     "hbm_resident": {"achieved_gbs": alg["b_fwd_resident"] * B / (fwd_ms * 1e-3) / 1e9, "peak_gbs": peak,
                                      "definition": "every input read once, every output written once / forward time"}},
        "clocks": clocks,
    }
    if e2e_f_s is not None:
        line["e2e_factored_gradients"] = {
            "value": world * B * e2e_steps / e2e_f_s, "unit": UNIT, "h2d_bytes_per_step": h2d,
            "d2h_bytes_per_step": ((n_dof + 2 * m_ineq + 1) * w + 8) * B + (n_dof + m_ineq + neq) * w * B,
            "api": "solve_forward / solve_backward(need=(dp, dh, db)) on pinned CPU tensors: the dense dQ, dG, dF, dA are "
                   "outer products of the returned vectors with zhat / lam / nu (lcp.py:52-63) and are not shipped"}
    if not cfg2:
        line["engine_path"] = eng
    if world == 1 and not args.no_cpu_baseline:
        ncores = use_all_host_threads()
        par, val, dt = parity_sample(inp_host, g_host, fo, bo, args.cpu_sample, dtype, MAX_ITER, with_bwd)
        line["parity"] = par
        line["config"]["parity_ok"] = bool(par["zhat_vs_reference"]["frac_within_tol"] >= 0.9 and
                                           par["zhat_vs_fp64"]["p90"] <= 1.2 * par["reference_vs_fp64"]["p90"] + 1e-5)
        line["cpu_baseline"] = {"value": val, "unit": UNIT, "cores": ncores, "kind": "port",
                                "sample": "the first %d scenes of the timed batch, %s, %.1f s, as-is reference semantics "
                                          "(incl. util.py:86-90 pivot loop); the same scenes feed `parity`"
                                          % (args.cpu_sample, "fwd+bwd" if with_bwd else "forward", dt)}
    print(json.dumps(line), flush=True)


def measured_traffic(batch, cfg="cfg3"):
    """DRAM bytes per forward launch from the newest committed ncu capture (profiles/rNN_fwd_traffic[_cfg2].json)."""
    import glob
    pat = "r*_fwd_traffic.json" if cfg == "cfg3" else "r*_fwd_traffic_cfg2.json"
    files = sorted(glob.glob(os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", pat)))
    if not files:
        return None
    with open(files[-1]) as f:
        d = json.load(f)
    return d["dram_bytes_per_launch"] * batch / d["batch"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default 5; 20 for --config cfg4)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="cfg3", choices=["cfg3", "cfg2", "world", "cfg4"],
                    help="cfg3 (default, BASELINE's headline): fwd+bwd, 4096 x 64 contacts, fp32; "
                         "cfg2: forward only, 1024 x 32 contacts x 3 fric dirs, fp64; world: BatchedWorld.step() over 1024 "
                         "small worlds; cfg4: BASELINE configs[3], World.step() loop on one 512-ball pile (fp64, banded kernel)")
    ap.add_argument("--batch", type=int, default=0, help="scenes per GPU (default: the config's)")
    ap.add_argument("--cpu-sample", type=int, default=128)
    ap.add_argument("--ref-batch", type=int, default=256)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the results of the last timed step to DIR/<name>.npy (--impl b200)")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = 20 if args.config == "cfg4" and args.impl == "b200" else 5
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29500")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", local_rank))
    try:
        if args.config == "world":
            run_world(args, rank, world, local_rank)
        elif args.config == "cfg4":
            run_cfg4(args, rank, world, local_rank)
        else:
            run_b200(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
