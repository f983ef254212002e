#!/usr/bin/env python
"""bench.py -- MCTS node-expansions/s on Connect-Four (BASELINE.json metric), one rank per GPU.

A "step" = MCTS.explore! (600 simulations) on every one of the rank's 4096 concurrent game trees (fresh trees,
synthetic random Connect-Four positions), every new node evaluated by the 7-block ResNet: config[1] of BASELINE.json.
  value : expansions/s with the roots already resident in HBM (az_mcts_set_roots before the timed region)
  e2e   : the same through the host-buffer seam az_mcts_explore (H2D roots + eta, run, D2H N/W/P inside the timed region)
Trees are sharded over ranks with no data-path collective (weak scaling: 4096 trees per GPU).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
  --impl reference : the reference's algorithm on the host CPU cores (oracle port + torch-CPU fp32 network),
                     rank 0 only, on a bounded sample of the same workload.
  --dump-outputs   : after the timed steps, write the root statistics N, W, P [trees, 7] of the last device-resident step
                     and e2e_N, e2e_W, e2e_P of the last end-to-end step as DIR/<name>.npy (float64, P float32; suffix
                     _rank<r> with several ranks).  The inputs are seeded, so two builds can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SEED_POS = 0xA17A2E80          # SURVEY 8d
TREES_PER_GPU = 4096
NSIMS = 600
BLOCKS = 7
HP = dict(num_blocks=BLOCKS, num_filters=128, conv_kernel_size=(3, 3), num_policy_head_filters=32, num_value_head_filters=32)
CONV_MFLOP_PER_LEAF = 2 * 42 * 128 * 1152 / 1e6     # one 3x3 conv layer, valid positions only (SURVEY 8d: 12.39 MFLOP)
NET_MFLOP_PER_LEAF = 174.7                           # whole 7-block network (SURVEY 2a)
METRIC = "mcts_node_expansions_per_s"
# dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel (ncu --set full, cold caches)
NCU_TRAFFIC_BYTES = 401.4e6  # profiles/r02final_tower_ncu_summary.txt: 50.3 MB read + 351.1 MB written per launch of az_k_tower_yrow (ONE launch = all 14 layers; ncu, cold caches, ~3000 leaves)


def resnet_blob(dim, num_actions, hp, seed=1):
    """Random-init weights of a freshly constructed Flux ResNet (Glorot-uniform conv/dense weights, zero biases,
    BatchNorm gamma=1 beta=0 mu=0 sigma2=1) in the blob order az_net_load expects (include/azb200.h).  Kept here so that
    the product arm of the bench never imports oracle/."""
    W, H, C = dim
    nf, nb, npf, nvf = hp["num_filters"], hp["num_blocks"], hp["num_policy_head_filters"], hp["num_value_head_filters"]
    rng = np.random.default_rng(seed)
    parts = []

    def conv(k, ci, co):
        s = np.sqrt(6.0 / (k * k * ci + k * k * co))
        parts.extend([rng.uniform(-s, s, k * k * ci * co), np.zeros(co)])

    def bn(n):
        parts.extend([np.ones(n), np.zeros(n), np.zeros(n), np.ones(n)])

    def dense(out, inn):
        s = np.sqrt(6.0 / (inn + out))
        parts.extend([rng.uniform(-s, s, out * inn), np.zeros(out)])
    conv(3, C, nf); bn(nf)
    for _ in range(nb):
        conv(3, nf, nf); bn(nf); conv(3, nf, nf); bn(nf)
    conv(1, nf, nvf); bn(nvf); dense(nf, W * H * nvf); dense(1, nf)
    conv(1, nf, npf); bn(npf); dense(num_actions, W * H * npf)
    return np.concatenate(parts).astype(np.float32)


NCU_TREE_TRAFFIC_BYTES = 6.56e6   # profiles/r02final_tree_ncu_summary.txt: select 3.57 MB + expand_backup 2.99 MB of DRAM reads per tick (cold, tick ~550)


def hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f)["hbm_gbs"], "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def sum_ms(tp):
    return tp["select_ms"] + tp["expand_ms"] + tp["net_ms"]


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return p["bf16_tflops_sustained"], "measured (MEASURED_PEAKS.json bf16_tflops_sustained)"
    except Exception:
        return 1400.0, "fallback (B200_PROFILING.md sustained)"


class ClockSampler:
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu=0):
        self.gpu, self.rows, self.stop, self.th = gpu, [], False, None

    def _run(self):
        while not self.stop:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def __enter__(self):
        self.th = threading.Thread(target=self._run, daemon=True)
        self.th.start()
        return self

    def __exit__(self, *a):
        self.stop = True
        self.th.join(timeout=6)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = sorted(float(r[1]) for r in self.rows)
        reasons = []
        for i, name in enumerate(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]):
            if any(r[4 + i].lower().startswith("active") for r in self.rows):
                reasons.append(name)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.rows[0][2]), "reasons": reasons, "samples": len(sm)}


def make_eta(_unused, roots, A, seed):
    """Dirichlet(1) root noise per tree; generated with numpy here (bench input, not a parity path)."""
    rng = np.random.default_rng(seed)
    eta = np.zeros((len(roots), A))
    full = np.array([(r[35:42] == 0).sum() for r in roots])  # legal columns = empty top cells
    for i, n in enumerate(full):
        e = rng.exponential(size=n)
        eta[i, :n] = e / e.sum()
    return eta


DUMP_BYTES = 60 * 10**6   # all ranks together, .npy headers aside: a dump stays under 64 MB at any --trees


def dump_outputs(d, arrays, rank, world):
    """Writes `arrays` (one row per tree) as d/<name>.npy in float64 (float32 arrays stay float32).  Above this rank's share
    of DUMP_BYTES every array keeps the same fixed, seeded sample of rows (in tree order)."""
    arrays = {k: np.asarray(v, np.float32 if v.dtype == np.float32 else np.float64) for k, v in arrays.items()}
    n = len(next(iter(arrays.values())))
    keep = min(n, DUMP_BYTES // world // sum(a[0].nbytes for a in arrays.values()))
    rows = np.sort(np.random.default_rng(0).choice(n, keep, replace=False)) if keep < n else slice(None)
    os.makedirs(d, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(d, k + ("_rank%d" % rank if world > 1 else "") + ".npy"), a[rows])


def product_config(S, nsims, blocks, oracle_net, world):
    """The `config` object of a bench line (both arms print the same one for the same workload)."""
    return {"workload": "connect-four: %d concurrent game trees per GPU x %d sims/move, %s, synthetic random positions (0-30 plies), fresh trees per step"
                        % (S, nsims, ("%d-block ResNet 128 filters" % blocks) if not oracle_net else oracle_net + " oracle"),
            "trees_per_gpu": S, "nsims": nsims, "parallelism": "trees sharded over %d rank(s), no data-path collective" % world,
            "l2": "inputs larger than L2: tree tables %.0f MB + activations %.0f MB per GPU" % (S * 1024 * 128 / 1e6, S * 42 * 128 * 5 / 1e6)}


def cpu_reference_run(n_trees, nsims, threads, seed_offset=0, net="resnet"):
    """The reference's algorithm on host cores: CPU MCTS (oracle port, `threads` host threads over the independent trees
    like the reference's worker tasks) + either the batched torch-CPU fp32 7-block ResNet (net="resnet": the end-to-end
    figure) or the uniform oracle (net="uniform": the tree-only figure, MCTS.RandomOracle).  Every tick evaluates the
    pending leaves of all trees as ONE batch, the shape the product runs.  Returns (expansions, seconds, simulations)."""
    import torch
    from oracle import oracle as oz, netref
    torch.set_num_threads(threads)
    oz.set_threads(threads)
    gid = oz.game_id("connect-four")
    dim, A = (7, 6, 3), 7
    blob = netref.make_blob(dim, A, HP, seed=1, randomize=False) if net == "resnet" else None
    roots = oz.random_positions(gid, SEED_POS, n_trees, 30, first_stream=seed_offset)
    eta = make_eta(None, roots, A, 3)
    mp = oz.mcts_params(cpuct=2.0, noise_eps=0.25, noise_alpha=1.0, num_iters_per_turn=nsims)
    b = oz.Batch(gid, n_trees, mp)
    b.set_roots(roots, eta)
    t0 = time.perf_counter()
    while True:
        ls, _ = b.advance()
        if len(ls) == 0:
            break
        X, mask = b.vectorize(ls, (dim[2], dim[1], dim[0]))   # GI.vectorize_state (flat index w + W*(h + H*c)) + actions mask, threaded in C
        if net == "resnet":
            # the forward of the tick's batch in cache-sized chunks (a 4096-leaf fp32 activation is 88 MB per layer: the CPU
            # is 5x faster on 256-leaf chunks; the reference itself ships batch_size 64)
            Xt = X.transpose(0, 3, 2, 1)   # [B, W, H, C]
            outs = [netref.forward(blob, dim, A, HP, Xt[i:i + CPU_CHUNK]) for i in range(0, len(ls), CPU_CHUNK)]
            P, V = np.concatenate([o[0] for o in outs]), np.concatenate([o[1] for o in outs])
            Pn, V, _ = netref.forward_normalized(P, V, mask)
        else:
            Pn = mask.astype(np.float32) / mask.sum(1, keepdims=True).astype(np.float32)
            V = np.zeros(len(ls), np.float32)
        b.feed(Pn, V)
    dt = time.perf_counter() - t0
    return b.expansions, dt, b.simulations


def cpu_baseline_legs(threads):
    """BASELINE.md section 2: tree-only and end-to-end figures of the CPU port on 1 and on `threads` host threads (bounded samples)."""
    legs = {}
    for name, (nt, ns, th, net) in {"tree_only_1thread": (512, 200, 1, "uniform"), "tree_only": (4096, 100, threads, "uniform"),
                                    "e2e_1thread": (64, 12, 1, "resnet"), "e2e": (4096, 8, threads, "resnet")}.items():
        ex, dt, sims = cpu_reference_run(nt, ns, th, net=net)
        legs[name] = {"expansions_per_s": ex / dt, "simulations_per_s": sims / dt, "cores": th, "seconds": dt,
                      "sample": "%d trees x %d sims, %s" % (nt, ns, "uniform oracle (tree work only)" if net == "uniform" else "torch-CPU fp32 7-block ResNet, all pending leaves of a tick in chunks of %d" % CPU_CHUNK)}
    return legs


CPU_CHUNK = 256
REF_TREES, REF_SIMS = 4096, 12   # reference arm: the product's pool size, the first REF_SIMS of the 600 simulations


def run_reference(args, rank, world):
    if rank != 0:
        return
    threads = args.cpu_threads or min(os.cpu_count() or 1, 16)
    n_trees, nsims = REF_TREES, REF_SIMS
    for _ in range(max(1, min(args.warmup, 1))):
        cpu_reference_run(256, 4, threads)
    ex, dt = 0, 0.0
    for k in range(args.steps):
        e, d, _ = cpu_reference_run(n_trees, nsims, threads, seed_offset=1000 * k)
        ex += e
        dt += d
    v = ex / dt
    sample = ("%d trees x the first %d of %d sims per step (config[1] pool size and leaf-batch shape: every tick evaluates the pending "
              "leaves of all %d trees, forward in chunks of 256); CPU MCTS (C port of src/mcts.jl, %d host threads over trees) + torch-CPU fp32 "
              "7-block ResNet (%d threads)" % (n_trees, nsims, NSIMS, n_trees, threads, threads))
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "expansions/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            # the SAME config object as the product arm's line (BASELINE config[1]); what the CPU arm actually runs of it per step
            # (a bounded sample: the first REF_SIMS simulations) is stated in cpu_baseline.sample
            "config": product_config(n_trees, NSIMS, BLOCKS, None, max(1, args.gpus)),
            "cpu_baseline": {"value": v, "unit": "expansions/s", "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": "expansions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--trees", type=int, default=TREES_PER_GPU)
    ap.add_argument("--nsims", type=int, default=NSIMS)
    ap.add_argument("--blocks", type=int, default=BLOCKS)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-selfplay", action="store_true", help="skip the full self-play leg (games/s)")
    ap.add_argument("--cpu-threads", type=int, default=0, help="threads of the CPU reference arm (0 = min(cores, 16): torch-CPU conv throughput peaks there on the 128-core box)")
    ap.add_argument("--oracle-net", default=None, choices=[None, "uniform", "synth"], help="tree-only figure: built-in oracle instead of the ResNet")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="write the root statistics of the last timed steps as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return run_reference(args, rank, world)

    import torch
    import _pkg
    az = _pkg.load()
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ctx = az.Context(local)
    comm = az.Comm.from_torch(ctx, dist) if world > 1 else None   # the engine's own NCCL communicator (id exchanged over torch's store)
    gs = az.GameSpec("connect-four")
    S, nsims, A = args.trees, args.nsims, 7
    hp = dict(HP, num_blocks=args.blocks)
    if args.oracle_net:
        net = az.RandomOracle(ctx, gs) if args.oracle_net == "uniform" else az.SynthOracle(ctx, gs)
    else:  # weights: Glorot-uniform, seed 1, fresh BatchNorm statistics (random init of the named architecture)
        net = az.ResNet(ctx, gs, az.ResNetHP(hp["num_blocks"], hp["num_filters"], hp["conv_kernel_size"],
                                             hp["num_policy_head_filters"], hp["num_value_head_filters"]))
        net.load(resnet_blob(gs.state_dim, gs.num_actions, hp, seed=1))
    mp = az.MctsParams(cpuct=2.0, num_iters_per_turn=nsims, dirichlet_noise_eps=0.25, dirichlet_noise_alpha=1.0)
    env = az.MctsEnv(ctx, gs, net, mp, S, capacity_nodes_per_tree=nsims + 8)
    roots = gs.random_positions(SEED_POS, S, 30, first_stream=rank * S)
    eta = make_eta(None, roots, A, 100 + rank)

    def barrier():
        ctx.synchronize()
        if dist is not None:
            torch.cuda.synchronize()
            dist.barrier()

    def step_resident():
        env.reset()
        env.run(nsims)
        return env.last_timing()

    def step_resident_noreset():
        env.run(nsims)
        return env.last_timing()

    def step_e2e():
        env.reset()
        t0 = time.perf_counter()
        NWP = env.explore(roots, nsims, eta)   # H2D roots+eta, 600 sims, D2H N/W/P
        dt = time.perf_counter() - t0
        return dt, env.last_timing()["expansions"], NWP

    env.set_roots(roots, eta)
    for _ in range(args.warmup):
        step_resident()
    # ---- timed: device-resident (CUDA-graph ticks; no per-launch events) ----
    l0 = ctx.num_launches
    barrier()
    with ClockSampler(local) as clk:
        ms, ex, ticks = 0.0, 0, 0
        t_wall = time.perf_counter()
        for _ in range(args.steps):
            t = step_resident()
            ms += t["ms_total"]
            ex += t["expansions"]
            ticks += t["ticks"]
        barrier()
        t_wall = time.perf_counter() - t_wall
    launches = ctx.num_launches - l0
    if args.dump_outputs:
        resident_NWP = env.root_stats()   # the last timed step's trees, before the passes below rebuild them
    # ---- roofline pass: the same steps again with CUDA events around the tower launches (events on the library's own
    #      stream; recording them per launch disables graph replay, hence a separate pass) ----
    prof = None
    if not args.oracle_net:
        net.set_profiling(True)
        p_ms, p_ex = 0.0, 0
        for _ in range(args.steps):
            t = step_resident()
            p_ms += t["ms_total"]
            p_ex += t["expansions"]
        prof = net.get_profile()
        prof.update(step_ms=p_ms, expansions=p_ex)
        net.set_profiling(False)
    # ---- tree-kernel pass: CUDA events around az_k_select and az_k_expand_backup of every tick (graph replay off) ----
    env.set_profiling(True)
    tp_nodes, tp_sims, tp_ex = 0, 0, 0
    for _ in range(args.steps):
        env.reset()
        c0 = env.counters()
        t = step_resident_noreset()
        c1 = env.counters()
        tp_nodes += int((c1[1] - c0[1]).sum())
        tp_sims += int((c1[0] - c0[0]).sum())
        tp_ex += t["expansions"]
    tprof = env.get_profile()
    tprof.update(nodes=tp_nodes, sims=tp_sims, expansions=tp_ex)
    env.set_profiling(False)
    # ---- timed: end to end through host buffers ----
    barrier()
    e_dt, e_ex = 0.0, 0
    for _ in range(args.steps):
        d, e, e2e_NWP = step_e2e()
        e_dt += d
        e_ex += e
    barrier()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dict(zip(("N", "W", "P", "e2e_N", "e2e_W", "e2e_P"), resident_NWP + e2e_NWP)), rank, world)
    sims = args.steps * S * nsims
    # ---- full self-play (games/s): simulate() with the shipped Connect-Four MctsParams, one game per slot ----
    sp_out = None
    if not args.no_selfplay and not args.oracle_net:
        env.close()
        env = None
        import importlib.util
        spec_d = importlib.util.spec_from_file_location("az_distributed", os.path.join(ROOT, "alphazero.jl_b200", "distributed.py"))
        azd = importlib.util.module_from_spec(spec_d)
        spec_d.loader.exec_module(azd)
        total_games = 2 * S * world   # two games per worker slot, 4096 games in flight per GPU at any time
        count, first = azd.split_games(total_games, world, rank)
        spp = az.SelfPlayParams(
            az.MctsParams(cpuct=2.0, num_iters_per_turn=nsims, temperature=az.PLSchedule([0, 20, 30], [1.0, 1.0, 0.3]),
                          dirichlet_noise_eps=0.25, dirichlet_noise_alpha=1.0),
            az.SimParams(num_games=count, num_workers=S, batch_size=S, reset_every=2))
        barrier()
        t0 = time.perf_counter()
        sp_h = az.SelfPlay(ctx, gs, net, spp, seed=1234)
        sp_h.start(count, first)
        sp_h.wait()
        out = sp_h.fetch()                                                        # includes the D2H fetch of all samples
        t_play = time.perf_counter() - t0
        # iteration-end exchange (src/simulations.jl:282-289) inside the engine: this rank's device-resident samples ->
        # az_samples_allgather (one count all-gather + one padded NCCL all-gather of packed rows, nothing staged on the host)
        rp = {}
        tr0 = time.perf_counter()
        smp = az.Samples.from_selfplay(sp_h)
        rp["export_ms"] = 1e3 * (time.perf_counter() - tr0)
        t1 = time.perf_counter()
        gathered, gather_ms, counts = smp, 0.0, [len(smp)]
        if comm is not None:
            gathered, counts = comm.allgather_samples(smp)
            gather_ms = comm.last_ms
        barrier()
        t_gather = time.perf_counter() - t1
        gather2_ms, gather2_wall = 0.0, 0.0
        if comm is not None:      # the same exchange again (NCCL's buffers for this size exist now): the steady-state figure of later iterations
            tg2 = time.perf_counter()
            g2, _ = comm.allgather_samples(smp)
            gather2_ms = comm.last_ms
            gather2_wall = time.perf_counter() - tg2
            g2.close()
        # replay-buffer side (SURVEY 8f rank 2) on this rank's samples, device resident: augment -> merge -> convert
        tr0 = time.perf_counter()
        aug = smp.augment_with_symmetries()
        rp["augment_ms"] = 1e3 * (time.perf_counter() - tr0); tr0 = time.perf_counter()
        mrg = aug.merge_by_state()
        rp["merge_ms"] = 1e3 * (time.perf_counter() - tr0); tr0 = time.perf_counter()
        cvbuf = mrg.convert_buffers()          # caller-allocated, already touched host arrays (a replay buffer that exists)
        tr0 = time.perf_counter()
        cv = mrg.convert(az.LOG_WEIGHT, out=cvbuf)
        rp["convert_to_host_ms"] = 1e3 * (time.perf_counter() - tr0)
        rp["convert_to_host_MB"] = sum(v.nbytes for v in cvbuf.values()) / 1e6
        rp.update(samples=len(smp), augmented=len(aug), merged=len(mrg), bytes_per_sample=24 + 8 * 7 + 8 + 8 + 4,
                  note="host wall clock per call incl. cudaMalloc of outputs and stream sync; rank 0's share")
        total_gathered = len(gathered)
        for x in (aug, mrg) + ((gathered,) if gathered is not smp else ()) + (smp,):
            x.close()
        del cv
        sp_h.close()
        sp_out = dict(t=t_play + t_gather, t_gather=t_gather, gather_device_ms=gather_ms, gather2_device_ms=gather2_ms, gather2_wall_s=gather2_wall, games=count, samples=int(out["samples"]),
                      expansions=float(out["expansions"]), total_samples=total_gathered, mean_moves=float(out["moves"].mean()),
                      mean_edepth=float(out["edepth"].mean()))
    # ---- arena (SURVEY 8f rank 1): pit_networks of two 7-block nets with the shipped Connect-Four ArenaParams
    # (games/connect-four/params.jl:32-45: 600 sims, cpuct 2, eps 0.05, tau 0.2, flip_probability 0.5, alternate_colors,
    # reset_every 2), one game per worker; every rank plays its own share, no collective ----
    ar_out = None
    if not args.no_selfplay and not args.oracle_net:
        net_b = az.ResNet(ctx, gs, az.ResNetHP(hp["num_blocks"], hp["num_filters"], hp["conv_kernel_size"],
                                               hp["num_policy_head_filters"], hp["num_value_head_filters"]))
        net_b.load(resnet_blob(gs.state_dim, gs.num_actions, hp, seed=2))
        AW = max(2, S // 2)
        app = az.SelfPlayParams(
            az.MctsParams(cpuct=2.0, num_iters_per_turn=nsims, temperature=az.ConstSchedule(0.2), dirichlet_noise_eps=0.05,
                          dirichlet_noise_alpha=1.0),
            az.SimParams(num_games=AW, num_workers=AW, batch_size=AW, reset_every=2, flip_probability=0.5, alternate_colors=True))
        barrier()
        t0 = time.perf_counter()
        ao = az.simulate(ctx, gs, net, app, seed=4321, first_game_index=rank * AW, baseline=net_b, gamma=1.0)
        barrier()
        ar_out = dict(t=time.perf_counter() - t0, games=AW, expansions=float(ao["expansions"]), avgr=float(ao["game_rewards"].mean()),
                      redundancy=float(ao["redundancy"]), mean_moves=float(ao["moves"].mean()))
        net_b.close()
    # ---- reduce over ranks: time = max, work = sum ----
    if dist is not None:
        if ar_out is not None:
            ta = torch.tensor([ar_out["t"]], device="cuda", dtype=torch.float64)
            dist.all_reduce(ta, op=dist.ReduceOp.MAX)
            wa = torch.tensor([ar_out["games"], ar_out["expansions"]], device="cuda", dtype=torch.float64)
            dist.all_reduce(wa, op=dist.ReduceOp.SUM)
            ar_out["t"] = ta.item()
            ar_out["games"], ar_out["expansions"] = wa.tolist()
        t = torch.tensor([ms, e_dt], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        w = torch.tensor([ex, e_ex, sims, launches], device="cuda", dtype=torch.float64)
        dist.all_reduce(w, op=dist.ReduceOp.SUM)
        ms, e_dt = t.tolist()
        ex, e_ex, sims, launches = w.tolist()
        if sp_out is not None:
            tt = torch.tensor([sp_out["t"], sp_out["t_gather"]], device="cuda", dtype=torch.float64)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            ww = torch.tensor([sp_out["games"], sp_out["samples"], sp_out["expansions"]], device="cuda", dtype=torch.float64)
            dist.all_reduce(ww, op=dist.ReduceOp.SUM)
            sp_out["t"], sp_out["t_gather"] = tt.tolist()
            sp_out["games"], sp_out["samples"], sp_out["expansions"] = ww.tolist()
    if rank == 0:
        value = ex / (ms / 1e3)
        line = {"metric": METRIC, "value": value, "unit": "expansions/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f16" if not args.oracle_net else "f64", "data": "synthetic",
                "config": product_config(S, nsims, args.blocks, args.oracle_net, world),
                "simulations_per_s": sims / (ms / 1e3), "expansions_per_simulation": ex / sims, "ticks_per_step": ticks / args.steps,
                "e2e": {"value": e_ex / e_dt, "unit": "expansions/s",
                        "h2d_bytes_per_step": int(S * 24 + eta.nbytes),
                        "d2h_bytes_per_step": int(S * A * (8 + 8 + 4))},
                "gpu_launches": int(launches), "clocks": clk.summary(), "host_wall_s_resident": t_wall}
        if sp_out is not None:
            line["selfplay"] = {"games_per_s": sp_out["games"] / sp_out["t"], "samples_per_s": sp_out["samples"] / sp_out["t"],
                                "expansions_per_s": sp_out["expansions"] / sp_out["t"], "seconds": sp_out["t"],
                                "allgather_seconds": sp_out["t_gather"], "allgather_device_ms": sp_out["gather_device_ms"], "allgather_device_ms_repeat": sp_out["gather2_device_ms"], "allgather_seconds_repeat": sp_out["gather2_wall_s"],
                                "allgather": "az_samples_allgather: NCCL, packed 104 B rows, device resident (no host staging)", "games": int(sp_out["games"]), "samples": int(sp_out["samples"]),
                                "gathered_samples_on_rank0": sp_out["total_samples"], "mean_moves_per_game": sp_out["mean_moves"],
                                "mean_exploration_depth": sp_out["mean_edepth"],
                                "config": "simulate(): %d games per GPU on 4096 concurrent worker slots (two per slot), 600 sims/move, cpuct 2, eps 0.25, tau PL([0,20,30],[1,1,.3]), reset_every 2; wall clock incl. sample D2H + all-gather" % (2 * S)}
        if sp_out is not None:
            line["replay"] = rp
        if ar_out is not None:
            line["arena"] = {"games_per_s": ar_out["games"] / ar_out["t"], "expansions_per_s": ar_out["expansions"] / ar_out["t"],
                             "seconds": ar_out["t"], "games": int(ar_out["games"]), "mean_moves_per_game": ar_out["mean_moves"],
                             "avg_reward_rank0": ar_out["avgr"], "redundancy_rank0": ar_out["redundancy"],
                             "config": "pit_networks(): two random-init 7-block ResNets, %d games per GPU on %d workers (two trees + two oracles per worker), 600 sims/move, cpuct 2, eps 0.05, tau 0.2, flip_probability 0.5, alternate_colors, reset_every 2" % (max(2, S // 2), max(2, S // 2))}
        if prof and prof["evals"]:
            peak, how = peaks()
            nconv = 2 * args.blocks
            achieved = prof["expansions"] * CONV_MFLOP_PER_LEAF * nconv / 1e6 / (prof["tower_ms"] / 1e3)   # rank 0's own pass
            line["roofline"] = {"bound": "tensor", "kernel": "az_k_tower_yrow" if prof["tower_launches"] == prof["evals"] else "az_k_conv_yrow", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                                "frac": achieved / peak, "traffic": NCU_TRAFFIC_BYTES, "peak_source": how,
                                "avg_launch_us": 1e3 * prof["tower_ms"] / max(1, prof["tower_launches"]),
                                "tower_launches": prof["tower_launches"], "avg_layer_us": 1e3 * prof["tower_ms"] / max(1, prof["evals"] * nconv),
                                "algorithmic_flop_per_launch": "12.39 MFLOP x leaves of the tick x conv layers per launch (SURVEY 8d: 2*42*128*1152 per leaf per conv layer; the persistent tower kernel runs all %d layers in one launch)" % nconv,
                                "how": "CUDA events around the tower (%d conv layers; one persistent launch or one launch per layer) of every tick on the library stream, in a profiled pass of the same %d steps right after the timed region (graph replay off); step time in that pass %.1f ms"
                                       % (nconv, args.steps, prof["step_ms"] / args.steps),
                                "network_share_of_step": prof["total_ms"] / prof["step_ms"],
                                "tower_share_of_step": prof["tower_ms"] / prof["step_ms"]}
        if tprof["ticks"]:
            hbm = hbm_peak()
            # SURVEY 8(d): select reads one 128 B line per traversed node, backup rewrites 24 B per traversed node, expand
            # probes 16 B and writes a 128 B line + Vest (148 B) per new node
            sel_bytes = 128.0 * tprof["nodes"]
            bk_bytes = 24.0 * tprof["nodes"] + 148.0 * tprof["expansions"]
            tree_ms = tprof["select_ms"] + tprof["expand_ms"]
            ach = (sel_bytes + bk_bytes) / 1e9 / (tree_ms / 1e3)
            line["roofline_tree"] = {
                "bound": "hbm", "kernels": "az_k_select + az_k_expand_backup", "achieved": ach, "peak": hbm[0], "unit": "GB/s",
                "frac": ach / hbm[0], "peak_source": hbm[1],
                "traffic": NCU_TREE_TRAFFIC_BYTES,
                "select_us_per_tick": 1e3 * tprof["select_ms"] / tprof["ticks"], "expand_backup_us_per_tick": 1e3 * tprof["expand_ms"] / tprof["ticks"],
                "select_GBps": sel_bytes / 1e9 / (tprof["select_ms"] / 1e3), "expand_backup_GBps": bk_bytes / 1e9 / (tprof["expand_ms"] / 1e3),
                "mean_depth": tprof["nodes"] / max(1, tprof["sims"]), "algorithmic_bytes_per_sim": (sel_bytes + bk_bytes) / max(1, tprof["sims"]),
                "share_of_step": tree_ms / sum_ms(tprof),
                "note": "latency-bound pointer chase: one simulation in flight per tree (reference semantics, no virtual loss), so memory-level "
                        "parallelism = 4096 dependent chains; the kernels move ~5 MB per launch and cannot approach the HBM roofline at this pool size "
                        "(north_star's 60 % target is not met; see DESIGN.md section 3 and profiles/r02*_tree_ncu_summary.txt)"}
        if not args.no_cpu_baseline and not args.oracle_net:
            threads = args.cpu_threads or min(os.cpu_count() or 1, 16)
            legs = cpu_baseline_legs(threads)
            line["cpu_baseline"] = {"value": legs["e2e"]["expansions_per_s"], "unit": "expansions/s", "cores": threads, "kind": "port",
                                    "sample": legs["e2e"]["sample"] + " (first 8 of the 600 simulations of config[1]); CPU MCTS = C port of src/mcts.jl",
                                    "legs": legs}
        print(json.dumps(line))
    if env is not None:
        env.close()
    net.close()
    if comm is not None:
        comm.close()
    ctx.close()
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
