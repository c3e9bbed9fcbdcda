#!/usr/bin/env python
"""Benchmark of the GN-ODE rollout hot path (BASELINE.json metric: rollout node-steps/s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    (N > 1: python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...)

Workload (config.workload): BASELINE.json configs[3] as written -- epinions-scale rollout inference of 4096 trials
(maxTime 20, deltaT 0.5: T = 40 grid points, 39 Euler steps). The epinions pickle is missing from the reference checkout,
so the graph is the synthetic stand-in BA(N=75,879, m=5, seed=0) (SURVEY 8d); trials are the synthetic (beta, gamma, I0)
draws of monitorer-sim.py:116-119; weights are the default nn.Linear init under seed 0.
One "step" = the whole job: all 4096 trials, streamed through the GPU(s) in chunks from COMPACT trial descriptors
(seeds, beta, gamma per trial: gnode_rollout_forward_trials, SURVEY 8f N4) -- the dense [N, 3+H] input block per trial
of the reference (83 GB for this job) is never built. Trials are independent -> the 4096 trials are sharded across the
ranks with the graph replicated, no collective on the data path; total work is fixed, so scaling is "strong".

Prints ONE JSON line (rank 0). value = node-steps/s with every descriptor resident in HBM and the probabilities of all T
grid points left in HBM; e2e = the same job through ODEBlock.forward_trials with the descriptors in pinned host memory
and the probabilities of the grid points the reference's test() consumes (get_sir_t_nodes_torch: rows int(i/deltaT),
20 of 40) copied back to pinned host memory inside the timed region.

--dump-outputs DIR writes what the last timed step of the device-resident measurement computed: the probabilities
[T, rows, 3] (S, I, R at every grid point) of DUMP_ROWS (trial, node) rows drawn with a fixed seed from the whole job, as
DIR/probs_sample.npy (float32), and their row ids trial * N + node as DIR/probs_sample_rows.npy (float64); under several
ranks each rank writes its own share with the suffix _rank<r>. The rows are gathered on the device after each chunk of
that step, one small index_select per chunk inside the timed window.
"""
import argparse
import atexit
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np    # noqa: E402
import torch          # noqa: E402

H = 64
MAXTIME, DELTAT = 20, 0.5
ALGO_BYTES_PER_NODE_STEP = 2060.0      # SURVEY 8d / BASELINE.md section 3 (fixed denominator)
R_STATE_NOTE = {
    1: "inference carries no R plane: S + I + R is conserved (dS + dI + dR = 0), so the decoder's R term is "
       "W3 (S_0 + I_0 + R_0) - W3 S_k - W3 I_k (4 floats per row written once + two terms the transform's GEMMs deliver); the "
       "64-float R plane is neither read nor written, i.e. 512 of the 2060 algorithmic bytes per node-step are not moved -- the "
       "roofline denominator stays 2060 B (SURVEY 8d); GNODE_R_STATE=full keeps the plane",
    0: "full 64-float R plane (GNODE_R_STATE=full)"}
JSON_OUT = sys.stdout
UNIT = "node-steps/s"
METRIC = "GN-ODE rollout node-steps/s (epinions)"
DUMP_ROWS = 65536                      # x T x 3 float32 = 31.5 MB for T = 40


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def traffic_file(workload):
    return "profiles/step_kernel_traffic.json" if workload == "epinions" else "profiles/step_kernel_traffic_%s.json" % workload


def ncu_traffic_per_launch(rows, workload="epinions"):
    """DRAM bytes per step-kernel launch: dram__bytes_read.sum + dram__bytes_write.sum of the committed
    `ncu --set full` capture of this workload (profiles/step_kernel_traffic*.json hold bytes per row of the capture)."""
    p = os.path.join(ROOT, traffic_file(workload))
    if os.path.exists(p):
        with open(p) as fh:
            return float(json.load(fh)["dram_bytes_per_row"]) * rows
    return None


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons of one GPU DURING the timed region."""
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.FIELDS,
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for r in self.rows:
            if len(r) < 7:
                continue
            try:
                sm.append(float(r[0])); smax.append(float(r[1]))
            except ValueError:
                continue
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "samples": len(sm), "reasons": sorted(reasons)}


WORKLOADS = {
    # name: (graph description, BASELINE.json config, total trials of the job, trials per chunk)
    "epinions": ("epinions stand-in BA(N=75879,m=5,seed=0)", "BASELINE.json configs[3]", 4096, 128),
    "ba2m": ("BA(N=2000000,m=10,seed=0) stress graph (chunked preferential attachment, ~20M edges)", "BASELINE.json configs[4]", 64, 8),
}


def build_graph(workload="epinions"):
    from gn_ode_sir_b200 import synth
    return synth.epinions_standin(seed=0) if workload == "epinions" else synth.ba_stress(seed=0)


def trial_descriptors(N, first, count):
    """(seeds, beta, gamma) of the trials first .. first+count-1: the draws of monitorer-sim.py:116-119."""
    from gn_ode_sir_b200 import synth
    seeds, beta, gamma = [], [], []
    for b in range(first, first + count):
        sd, be, ga = synth.trial_parameters(N, b)
        seeds.append(sd); beta.append(be); gamma.append(ga)
    return seeds, beta, gamma


def cpu_reference_sample(A, trials, n_points, repeats=1):
    """Times the oracle port of the reference's CPU path (torch ops, per-step host-side
    block_diag rebuild as at ode_nn_ngraph_sim.py:68-71) on a bounded sample. The only place
    where bench.py touches oracle/ (cpu_baseline leg and the --impl reference arm)."""
    import scipy.sparse
    from oracle import gnode_oracle as orc
    N = A.shape[0]
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    params = orc.default_params(H, seed=0)
    x = torch.cat([orc.synthetic_trial(N, H, b) for b in range(trials)])
    t = orc.time_grid(MAXTIME, DELTAT)[:n_points]

    def rebuild():
        bd = scipy.sparse.block_diag([A for _ in range(trials)])
        return torch.LongTensor(np.vstack((bd.row, bd.col)))

    best = float("inf")
    for _ in range(repeats):
        t0 = time.perf_counter()
        with torch.no_grad():
            orc.forward(x, params, None, t, rebuild_index=rebuild)
        best = min(best, time.perf_counter() - t0)
    units = trials * N * (n_points - 1)
    return units / best, cores, "%d trial(s) x %d Euler steps of the bench workload (%d node-steps, %.1f s)" % (
        trials, n_points - 1, units, best)


def run_reference_arm(args, rank, world):
    if rank != 0:
        return
    A = build_graph(args.workload)
    for _ in range(args.warmup):
        cpu_reference_sample(A, 1, 3)
    vals, times = [], []
    for _ in range(args.steps):
        t0 = time.perf_counter()
        v, cores, sample = cpu_reference_sample(A, args.ref_trials, args.ref_points)
        times.append(time.perf_counter() - t0)
        vals.append(v)
    value = float(np.mean(vals))
    out = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * float(np.mean(times)),
           "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": workload_config(args, world),
           "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
           "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    print(json.dumps(out), file=JSON_OUT, flush=True)


def job_size(args):
    total = args.trials if args.trials > 0 else WORKLOADS[args.workload][2]
    chunk = args.chunk if args.chunk > 0 else WORKLOADS[args.workload][3]
    return total, chunk


def workload_config(args, world):
    name, cfg, _, _ = WORKLOADS[args.workload]
    total, chunk = job_size(args)
    return {"workload": "%s rollout inference of %d trials, H=64, T=40 (maxTime=20, deltaT=0.5), streamed in chunks of %d trials "
                        "from compact (seeds, beta, gamma) descriptors (%s)" % (name, total, chunk, cfg),
            "global_trials": total, "trials_per_chunk": chunk,
            "nodes": 75879 if args.workload == "epinions" else 2000000,
            "euler_steps": int(len(np.arange(0, MAXTIME, DELTAT)) - 1),
            "parallelism": "trials sharded over %d rank(s), graph replicated, no data-path collective" % world,
            "l2_policy": "no flush: per-launch working set (state + I' of a chunk, >3 GB) exceeds the 126 MB L2"}


def run_train_mode(args, rank, world, dev, dist, gn, L):
    """Data-parallel training step on the five training graphs of BASELINE configs[2] (dolphins, fb-food, fb-social,
    openflights, wiki-vote: their CSR travels in tests/golden/ng_train5_b8.npz; real_graphs/ does not exist on the GPU
    box). Global batch = `--train-per-graph` instances of every graph (synthetic trials and labels), split across the
    ranks by node count; one step = forward with trajectory (only the unit-time grid points decoded) + fused L1 + reverse
    sweep + ONE flat all-reduce of the 4.6k-float gradient + Adam. Prints one JSON line (rank 0)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from _util import Golden
    from gn_ode_sir_b200 import harness, parallel, synth
    from gn_ode_sir_b200.rollout import l1_subsampled, unit_time_steps
    g = Golden("ng_train5_b8")
    names = ["dolphins", "fb-food", "fb-social", "openflights", "wiki-vote"]
    torch.manual_seed(0)
    of = gn.ode_ngraphs.ODEfunc(g.adjs, H, dev)
    blk = gn.ode_ngraphs.ODEBlock(MAXTIME, DELTAT, H, of, dev).to(dev)
    if dist is not None:
        parallel.broadcast_parameters(blk)
    T = len(np.arange(0, MAXTIME, DELTAT))
    gen = torch.Generator().manual_seed(1)
    items = []
    for gi, A in enumerate(g.adjs):
        n = A.shape[0]
        for k in range(args.train_per_graph):
            x = synth.synthetic_trial(n, H, 100 * gi + k)
            x[0, 5] = gi + 1
            y = torch.rand(n, MAXTIME, 3, generator=gen, dtype=torch.float64)
            items.append((x, y / y.sum(-1, keepdim=True), gi))
    sizes = [it[0].size(0) for it in items]
    mine = parallel.shard_instances(sizes, world)[rank] if world > 1 else list(range(len(items)))
    x = torch.cat([items[i][0] for i in mine]).to(dev)
    y = torch.cat([items[i][1] for i in mine]).to(dev)
    inst = [items[i][2] for i in mine]
    share = x.size(0) / float(sum(sizes))
    steps_sel = unit_time_steps(MAXTIME, DELTAT)
    opt = torch.optim.Adam(blk.parameters(), lr=1e-4)
    ar0, ar1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ar_ms = [0.0]

    def step(timed):
        opt.zero_grad()
        probs = blk.rollout_probs(x, out_steps=steps_sel, instances=inst)
        loss = l1_subsampled(probs, y, scale=share)
        loss.backward()
        if timed:
            ar0.record()
        parallel.allreduce_gradients(blk.parameters())
        if timed:
            ar1.record()
        opt.step()
        if timed:
            ar1.synchronize()
            ar_ms[0] += ar0.elapsed_time(ar1)
        return loss

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step(False)
    barrier()
    launches0 = int(L.gnode_launch_count())
    sampler = ClockSampler(int(os.environ.get("LOCAL_RANK", "0")))
    sampler.start()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    barrier()
    ev[0].record()
    for _ in range(args.steps):
        loss = step(True)
    ev[1].record()
    barrier()
    clocks = sampler.stop()
    ms = ev[0].elapsed_time(ev[1])
    if dist is not None:
        t = torch.tensor([ms, ar_ms[0]], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, ar = float(t[0]), float(t[1])
    else:
        ar = ar_ms[0]
    rows = sum(sizes)
    if rank == 0:
        out = {"metric": "GN-ODE multi-graph training node-steps/s (forward + backward)", "mode": "train",
               "value": rows * (T - 1) * args.steps / (ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
               "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong",
               "vs_baseline": None, "dtype": "f32", "data": "synthetic trials and labels on the shipped real graphs",
               "config": {"workload": "data-parallel training step on %s (BASELINE.json configs[2]): %d instances per graph, "
                                      "%d rows per global batch, adjoint gradients, Adam" % ("+".join(names), args.train_per_graph, rows),
                          "global_rows": rows, "euler_steps": T - 1,
                          "parallelism": "instances sharded over %d rank(s) by node count, one flat all-reduce of %d floats per step" % (world, 4553 + 256)},
               "allreduce": {"ms_per_step": ar / args.steps, "share_of_step": ar / ms, "backend": (dist.get_backend() if dist is not None else None)},
               "loss": float(loss.item()), "gpu_launches": int(L.gnode_launch_count()) - launches0, "clocks": clocks}
        print(json.dumps(out), file=JSON_OUT, flush=True)
    if dist is not None:
        dist.destroy_process_group()


def main():
    # stdout carries exactly ONE JSON line: everything else that libraries write to file descriptor 1 (NCCL prints its
    # version banner there under torchrun) is sent to stderr, and the JSON line goes to the saved descriptor.
    global JSON_OUT
    sys.stdout.flush()
    JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--mode", default="rollout", choices=["rollout", "train"],
                    help="rollout = the headline metric (default); train = data-parallel multi-graph training step "
                         "(BASELINE configs[2]): forward + fused L1 + reverse sweep + gradient all-reduce + Adam")
    ap.add_argument("--train-per-graph", type=int, default=8, help="--mode train: instances per graph in the global batch")
    ap.add_argument("--trials", type=int, default=0, help="total trials of the job (default: the workload's, 4096 for epinions)")
    ap.add_argument("--chunk", type=int, default=0, help="trials per chunk (default: the workload's, 128 for epinions)")
    ap.add_argument("--workload", default="epinions", choices=sorted(WORKLOADS),
                    help="epinions = the metric's configuration (default); ba2m = the 2M-node stress graph")
    ap.add_argument("--ref-trials", type=int, default=2)
    ap.add_argument("--ref-points", type=int, default=20)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write a fixed, seeded sample of what the last timed step computed to DIR/*.npy (--mode rollout)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.mode != "rollout"):
        ap.error("--dump-outputs needs --impl ours --mode rollout")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the GN-ODE rollout has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa_cpus = None
    if world > 1:
        # one process per GPU: host buffers next to the GPU (8 ranks x 28 GB/s of PCIe traffic must not cross sockets)
        from gn_ode_sir_b200.parallel import bind_to_gpu_numa_node
        numa_cpus = bind_to_gpu_numa_node(local_rank)
        print("bench.py: rank %d bound to %s" % (rank, ("%d CPUs near GPU %d" % (len(numa_cpus), local_rank)) if numa_cpus else "no CPU set (unchanged)"),
              file=sys.stderr, flush=True)
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        dist.init_process_group("nccl", device_id=dev)

    import gn_ode_sir_b200 as gn
    from gn_ode_sir_b200 import _build, _lib
    if "GNODE_B200_LIB" not in os.environ and _build.is_stale():
        # sources newer than the library build() left: rebuild into a temporary directory, never into the tree (which
        # may be read-only)
        tmp = tempfile.mkdtemp(prefix="gnode_b200_")
        atexit.register(shutil.rmtree, tmp, True)
        os.environ["GNODE_B200_LIB"] = _build.build_library(force=True, out=os.path.join(tmp, "libgnode_b200.so"))
    L = _lib.lib()

    from gn_ode_sir_b200.parallel import shard_trials
    from gn_ode_sir_b200.rollout import TrialSet, unit_time_steps
    if args.mode == "train":
        run_train_mode(args, rank, world, dev, dist, gn, L)
        return
    A = build_graph(args.workload)
    N = A.shape[0]
    T = len(np.arange(0, MAXTIME, DELTAT))
    total_trials, chunk = job_size(args)
    lo, hi = shard_trials(total_trials, world, rank)                 # this rank's trials [lo, hi)
    chunk = max(1, min(chunk, hi - lo))
    bounds = [(c, min(c + chunk, hi)) for c in range(lo, hi, chunk)]
    n_chunks = len(bounds)
    torch.manual_seed(0)
    of = gn.ode_sim.ODEfunc(A, 0.2, 0.1, H, dev)
    blk = gn.ode_sim.ODEBlock(MAXTIME, DELTAT, N, [0, 1], H, of, dev).to(dev).eval()
    units_per_step = total_trials * N * (T - 1)                      # whole job, all ranks
    # the job's inputs: one pinned-host descriptor set per chunk (a few KB each)
    host_sets = [TrialSet(*trial_descriptors(N, c0, c1 - c0), [N] * (c1 - c0)) for c0, c1 in bounds]
    rows_full = chunk * N
    ws_bytes = int(L.gnode_rollout_trials_workspace_bytes(of.batch_for(chunk).handle, 0))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if dist is None:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---------------- device-resident measurement (value, roofline): descriptors of every chunk in HBM, all T grid
    # points emitted into one reused [T, M_chunk, 3] buffer
    dev_sets = [hs.to(dev) for hs in host_sets]
    out_full = torch.empty((T, rows_full, 3), dtype=torch.float32, device=dev)
    dump, dump_rows = None, None
    if args.dump_outputs:
        # per chunk: (row indices within the chunk, [T, rows, 3] destination) of the job-wide seeded sample
        pick = np.random.default_rng(0).choice(total_trials * N, size=min(DUMP_ROWS, total_trials * N), replace=False)
        dump_rows = np.sort(pick[(pick >= lo * N) & (pick < hi * N)])
        dump = []
        for c0, c1 in bounds:
            sel = dump_rows[(dump_rows >= c0 * N) & (dump_rows < c1 * N)] - c0 * N
            dump.append((torch.from_numpy(sel).to(dev), torch.empty((T, len(sel), 3), dtype=torch.float32, device=dev)))

    def job_resident(capture=None):
        for k, ((c0, c1), ds) in enumerate(zip(bounds, dev_sets)):
            if c1 - c0 == chunk:
                blk.forward_trials(ds, None, None, probs_out=out_full, workspace=ws)
                probs = out_full
            else:                                                      # ragged last chunk: its own (smaller) buffers
                probs = blk.forward_trials(ds, None, None)
            if capture is not None:
                probs = probs if probs is out_full else torch.cat(probs, -1)
                torch.index_select(probs, 1, capture[k][0], out=capture[k][1])

    with torch.no_grad():
        for _ in range(args.warmup):
            job_resident()
        barrier()
        sampler = ClockSampler(local_rank)
        sampler.start()
        launches0 = int(L.gnode_launch_count())
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        barrier()
        ev[0].record()
        for i in range(args.steps):
            job_resident(dump if i == args.steps - 1 else None)
        ev[1].record()
        barrier()
        clocks = sampler.stop()
        launches = int(L.gnode_launch_count()) - launches0
        ms_local = ev[0].elapsed_time(ev[1])
        ms_total = max_over_ranks(ms_local)
    if dump is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        suffix = "_rank%d" % rank if world > 1 else ""
        np.save(os.path.join(args.dump_outputs, "probs_sample%s.npy" % suffix), torch.cat([d for _, d in dump], 1).cpu().numpy())
        np.save(os.path.join(args.dump_outputs, "probs_sample_rows%s.npy" % suffix), dump_rows.astype(np.float64))
        del dump
    ms_per_step = ms_total / args.steps
    value = units_per_step / (ms_per_step * 1e-3)
    # dominant kernel = the fused Euler-step kernel: (T-1) launches per chunk, each over the chunk's rows; the trial
    # expansion, encoder and final decode launches of a chunk are timed in the same stream window and are charged to
    # the step kernel (conservative: makes the per-launch time slightly larger).
    local_rows = (hi - lo) * N                                         # rows this rank pushes through one Euler step per job
    step_ms = ms_local / (args.steps * n_chunks * (T - 1))             # average launch (chunks of this rank)
    rows_per_launch = local_rows / n_chunks
    peak, peak_src = measured_peak()
    achieved = rows_per_launch * ALGO_BYTES_PER_NODE_STEP / (step_ms * 1e-3) / 1e9
    traffic = ncu_traffic_per_launch(rows_per_launch, args.workload)
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic,
                "kernel": "gnode::step_stream_kernel (fused Euler step: TMA-fed S tile, tcgen05 transform, CSR gather, SIR update; "
                          "the chunk's expansion, encoder and final decode launches are charged to it)",
                "launch_ms": step_ms, "rows_per_launch": rows_per_launch,
                "algorithmic_bytes_per_node_step": ALGO_BYTES_PER_NODE_STEP, "peak_source": peak_src,
                "traffic_source": "%s (ncu --set full dram bytes per row of the committed capture) x rows" % traffic_file(args.workload),
                "r_state": R_STATE_NOTE[int(L.gnode_get_r_state())]}
    del out_full, dev_sets

    # ---------------- end-to-end through the public API with host buffers
    # The caller's loop: descriptors of a chunk pinned host -> device (KBs), ODEBlock.forward_trials emitting the grid
    # points the reference's test() consumes (get_sir_t_nodes_torch: int(i/deltaT), 20 of 40), probabilities -> pinned host.
    # Three streams: the D2H of chunk c-1 overlaps the rollout of chunk c (plain PyTorch stream code around the drop-in
    # module; every byte is copied every step; the K timed steps form one continuous stream of chunks).
    sel = unit_time_steps(MAXTIME, DELTAT)
    n_sel = len(sel)
    out_pin = [torch.empty((n_sel, rows_full, 3), dtype=torch.float32).pin_memory() for _ in range(2)]
    out_dev = [torch.empty((n_sel, rows_full, 3), dtype=torch.float32, device=dev) for _ in range(2)]
    land = [host_sets[0].to(dev) for _ in range(2)]                    # device landing buffers of the descriptors
    h2d_bytes = sum(hs.h2d_bytes for hs in host_sets)
    d2h_bytes = n_sel * local_rows * 3 * 4
    s_in, s_cmp, s_out = torch.cuda.Stream(), torch.cuda.Stream(), torch.cuda.Stream()
    ev_free = [torch.cuda.Event() for _ in range(2)]                   # descriptors of buffer b consumed
    ev_in = [torch.cuda.Event() for _ in range(2)]
    ev_cmp = [torch.cuda.Event() for _ in range(2)]
    ev_out = [torch.cuda.Event() for _ in range(2)]                    # result buffer b copied out

    def e2e_steps(n_steps):
        main = torch.cuda.current_stream()
        for st in (s_in, s_cmp, s_out):
            st.wait_stream(main)
        for i in range(n_steps * n_chunks):
            c = i % n_chunks
            c0, c1 = bounds[c]
            buf = i % 2
            full = c1 - c0 == chunk
            with torch.cuda.stream(s_in):
                if i >= 2:
                    s_in.wait_event(ev_free[buf])
                tgt = land[buf] if full else host_sets[c].to(dev)
                if full:
                    tgt.copy_from(host_sets[c])
                ev_in[buf].record(s_in)
            with torch.cuda.stream(s_cmp):
                s_cmp.wait_event(ev_in[buf])
                if i >= 2:
                    s_cmp.wait_event(ev_out[buf])                       # out_dev[buf] has been copied to the host
                if full:
                    dst = out_dev[buf]
                    blk.forward_trials(tgt, None, None, out_steps=sel, probs_out=dst, workspace=ws)
                else:
                    dst = torch.cat(blk.forward_trials(tgt, None, None, out_steps=sel), -1)
                ev_free[buf].record(s_cmp)
                ev_cmp[buf].record(s_cmp)
            with torch.cuda.stream(s_out):
                s_out.wait_event(ev_cmp[buf])
                if full:
                    out_pin[buf].copy_(dst, non_blocking=True)
                else:
                    out_pin[buf][:, :(c1 - c0) * N].copy_(dst, non_blocking=True)
                    dst.record_stream(s_out)
                ev_out[buf].record(s_out)
        for st in (s_in, s_cmp, s_out):
            main.wait_stream(st)

    with torch.no_grad():
        e2e_steps(1)
        barrier()
        ev2 = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        ev2[0].record()
        e2e_steps(args.steps)
        ev2[1].record()
        barrier()
        e2e_ms = max_over_ranks(ev2[0].elapsed_time(ev2[1])) / args.steps
    e2e = {"value": units_per_step / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d_bytes,
           "d2h_bytes_per_step": d2h_bytes, "ms_per_step": e2e_ms, "chunks": n_chunks,
           "api": "ODEBlock.forward_trials(seeds, beta, gamma, out_steps=int(i/deltaT)): descriptors from pinned host memory, "
                  "probabilities of the %d grid points the reference's test() consumes to pinned host memory (per rank)" % n_sel}

    # ---------------- CPU baseline (oracle port of the reference's CPU path), rank 0, N=1 only
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        v, cores, sample = cpu_reference_sample(A, args.ref_trials, args.ref_points)
        cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample}

    if rank == 0:
        out = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
               "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
               "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(args, world),
               "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": launches, "clocks": clocks}
        print(json.dumps(out), file=JSON_OUT, flush=True)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
