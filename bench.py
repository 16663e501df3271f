#!/usr/bin/env python
"""bench.py -- headline benchmark: MCTS simulations/sec (NPS), crazyhouse start position, Batch_Size 64.

One "step" = one complete search (`go`) of --sims simulations with a fresh tree: root evaluation, then mini-batch
iterations of select -> RISE conv stack (tcgen05) -> scatter / backup, all device-resident.  NPS is computed exactly like
the reference: (root.visitSum - root.freeVisits) / elapsed (engine/src/evalinfo.cpp:73-85, node.cpp:1303-1306).

  --threads 2 (default): the reference's UCI default `Threads 2` (uci/optionsuci.cpp:182) -- two logical search threads
           per tree in the fixed schedule of oracle/mcts.h: one thread selects its next mini-batch while the other's
           is at the network.  Deterministic, bit-exact against the oracle's and the compiled reference's two threads
           in the same schedule (tests/test_ref_mcts.py, tests/test_search_gpu.py).
  --threads 1: the single-threaded parity mode; reported in the same line as `threads1` when the headline runs 2.
  value  : device-resident NPS -- CUDA events on the search stream around each go (root board already uploaded)
  e2e    : the same searches through the public host API (BoardState -> MCTSAgent.evaluate_board_state -> EvalInfo),
           wall clock, host<->device copies inside
  roofline: conv stack (the dominant kernels): algorithmic FLOPs of the leaves a search EVALUATES / the device time of
           its network forwards (CUDA events around every forward, taken live on extra searches right after the timed
           ones) vs the measured sustained bf16 tensor peak of MEASURED_PEAKS.json
  predict_seam: the drop-in NeuralNetAPI::predict seam alone -- host buffers through ara_net_predict (H2D planes,
           forward, D2H value + full policy), evaluations per second, like the reference's `inference` command
           (uci/crazyara.cpp:156-181)
  cpu_baseline / --impl reference: the reference's OWN search code (node.cpp, searchthread.cpp, MCTSAgent ... compiled
           unchanged into oracle/_ref/libref_mcts.so, kind "reference"; the oracle port oracle/mcts.c when that library
           is absent, kind "port") with the fp32 torch CPU network on the host cores, on the SAME workload (same
           simulations, batch size, threads).
  --config 2|3: BASELINE.json's other single-GPU search configurations (cfg 2: crazyhouse RISEv2 Batch_Size 8, 800
           simulations; cfg 3: chess RISEv3.3 Batch_Size 64, 1600 simulations) instead of the headline workload.
  --config 4|5: the self-play configurations (cfg 4: chess960, RISEv3.3, 8 concurrent games per GPU; cfg 5: King of the
           Hill + Three-check mixed, RISEv2 63 channels, Batch_Size 128 rows per forward): FINISHED games per hour.
  --dump-outputs DIR: after the timed steps, the last step's search result (root moves, visits, Q, priors, MCTS policy,
           principal variation, root scalars) as DIR/<name>.npy, for comparing two builds output for output.
Multi-GPU: replicas only (games/searches never interact; no collective on the data path): every rank runs the same
workload on its own GPU, value = sum of nodes / max over ranks of the time ("weak" scaling).
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "MCTS simulations/sec (NPS) crazyhouse startpos batch=64"
UNIT = "nodes/s"


def net_flops_per_position(arch):
    """2*MAC per evaluated position (BN folded), SURVEY Appendix B."""
    C = arch["channels"]
    f = 2 * 64 * C * arch["in_channels"] * 9
    for k, se, cop in zip(arch["kernels"], arch["se_types"], arch["c_ops"]):
        f += 2 * 64 * (C * cop) * 2 + 2 * 64 * cop * k * k
        if se == "ca_se":
            f += 2 * (C * (C // 2)) * 2
        elif se == "eca_se":
            f += 2 * C * C
    f += 2 * 64 * C * C * 9 + 2 * 64 * C * arch["policy_channels"] * 9
    f += 2 * 64 * C * 8 + (2 * 512 * 4 if arch["wdl"] else 2 * (512 * 256 + 256))
    return f


class ClockSampler(threading.Thread):
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        super().__init__(daemon=True)
        self.device = device
        self.samples = []
        self.stop_flag = False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                                      "-i", str(self.device)], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        sm, mx, reasons = [], 0, set()
        for s in self.samples:
            try:
                sm.append(float(s[1]))
                mx = max(mx, float(s[2]))
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


WORKLOADS = {
    # name: (variant, variant id, mode, net family, in channels, policy channels, input version, batch, sims)
    "M": ("crazyhouse", 1, "crazyhouse", "risev2", 34, 81, 1, 64, 3200),
    "2": ("crazyhouse", 1, "crazyhouse", "risev2", 34, 81, 1, 8, 800),
    "3": ("chess", 0, "chess", "risev33", 52, 76, 3, 64, 1600),
}


def make_arch(family, cin, pch):
    from crazyara_b200 import synthetic
    return synthetic.risev2(cin, pch) if family == "risev2" else synthetic.risev33(cin, pch)


def host_threads():
    try:
        avail = len(os.sched_getaffinity(0))
    except Exception:
        avail = os.cpu_count() or 1
    try:  # cgroup CPU quota (the container may see every host core but only be allowed a few)
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            avail = min(avail, max(1, int(int(q) / int(p))))
    except Exception:
        pass
    # beyond ~16 threads the 8x8-board convolutions of one forward only get slower
    return max(1, min(avail, int(os.environ.get("ARA_CPU_THREADS", "16"))))


def cpu_arm(workload, sims, batch, threads, steps, warmup):
    """Reference arm / cpu_baseline: the reference's own search (compiled, oracle/_ref) or the oracle port, with the fp32
    torch CPU network, on the same workload.  Returns (nps, ms per step, cores, kind, description)."""
    import torch

    from oracle import net as onet
    from oracle import refmcts
    from oracle import search as osr
    from oracle.chess import Position
    variant, vid, mode, family, cin, pch, version = WORKLOADS[workload][:7]
    cores = host_threads()
    torch.set_num_threads(max(1, cores // threads))
    from crazyara_b200 import synthetic
    arch = make_arch(family, cin, pch)           # the same random network the GPU arm runs
    sd = synthetic.random_state_dict(arch, 0)
    st = osr.default_settings(mode, batch_size=batch, simulations=sims, input_version=version, threads=threads)
    use_ref = refmcts.available()
    if use_ref and threads == 2:
        st.reserved = 1  # the reference's own two OS threads (run_mcts_search), not the deterministic schedule

    def net_fn(planes, keys=None):
        out = onet.forward(sd, arch, planes)
        return out["value"], out["prob"]
    channels = cin
    n_labels = pch * 64

    def one():
        pos = Position(variant=variant)
        t0 = time.perf_counter()
        if use_ref:
            r = refmcts.run(pos, None, vid, False, [], st, net_fn=net_fn, channels=channels, n_labels=n_labels)
        else:
            S = osr.Search(st)
            r = S.run(pos, net_fn, threads=threads)
            S.close()
        return r["nodes"], time.perf_counter() - t0

    for _ in range(warmup):
        one()
    nodes, secs = 0, 0.0
    for _ in range(steps):
        n, dt = one()
        nodes += n
        secs += dt
    kind = "reference" if use_ref else "port"
    what = ("the reference's search code compiled unchanged (node.cpp, searchthread.cpp, MCTSAgent: oracle/_ref/libref_mcts.so)"
            if use_ref else "C oracle search (oracle/mcts.c)")
    desc = (f"{steps} searches of {sims} simulations (Batch_Size {batch}, Threads {threads}) of the same workload; {what} + "
            f"fp32 torch CPU network, {cores} host threads")
    return nodes / secs, secs / steps * 1e3, cores, kind, desc


def predict_seam_leg(net, batch, channels, n_labels, seconds=1.5):
    """The drop-in seam alone: NeuralNetAPI::predict with caller-owned host buffers (pinned like neuralnetapiuser.cpp:52-59):
    H2D planes, forward, D2H value + the full policy, synchronous -- evaluations per second."""
    import numpy as np
    import torch
    x = torch.rand(batch, channels, 8, 8).pin_memory().numpy()
    v = torch.zeros(batch).pin_memory().numpy()
    p = torch.zeros(batch, n_labels).pin_memory().numpy()
    for _ in range(5):
        net.predict(x, v, p, None, n=batch)
    t0 = time.perf_counter()
    calls = 0
    while time.perf_counter() - t0 < seconds:
        net.predict(x, v, p, None, n=batch)
        calls += 1
    dt = time.perf_counter() - t0
    assert np.isfinite(v).all()
    return {"evals_per_s": calls * batch / dt, "ms_per_call": dt / calls * 1e3, "batch": batch,
            "h2d_bytes_per_call": int(x.nbytes), "d2h_bytes_per_call": int(v.nbytes + p.nbytes),
            "note": "ara_net_predict: pinned host buffers in, value + full soft-maxed policy out, synchronous"}


def multi_tree_leg(blob, device, trees, batch, sims, flops_pos, reps=3):
    """T independent searches (each Batch_Size `batch`) advanced together on one GPU: the analysis-server / arena shape.
    Every iteration one network forward serves all trees, so the conv stack sees T*batch positions."""
    from crazyara_b200.engine import BoardState, MCTSAgent, default_settings
    from crazyara_b200.nn import NeuralNetAPI
    net = NeuralNetAPI("gpu", device, batch * trees, blob)
    agent = MCTSAgent(net, default_settings("crazyhouse", batch_size=batch, simulations=sims), device, trees)
    openings = ["", "e2e4", "d2d4", "g1f3", "e2e4 e7e5", "d2d4 d7d5", "c2c4", "b1c3"]
    states = []
    for t in range(trees):
        s = BoardState().set("", False, 1)
        if openings[t % len(openings)]:
            s.do_uci(*openings[t % len(openings)].split())
        states.append(s)
    best = None
    for rep in range(reps + 2):
        profiled = rep == reps + 1  # the last repetition carries events between the kernels for the phase split
        agent.set_profile(profiled)
        for t, s in enumerate(states):
            agent.set_position(s, t)
        agent.evaluate_board_state()
        if rep == 0:
            continue
        res = agent.results()
        if profiled:
            prof = agent.profile()
            evals = sum(r["evals"] for r in res)
            best.update({"net_ms": prof["net_ms"], "select_ms": prof["select_ms"], "apply_ms": prof["apply_ms"],
                         "conv_tflops": evals * flops_pos / (prof["net_ms"] * 1e-3) / 1e12})
            continue
        ms = agent.last_go_ms()
        nodes = sum(r["nodes"] for r in res)
        row = {"trees": trees, "batch_per_tree": batch, "simulations": sims, "nps": nodes / (ms * 1e-3), "ms_per_go": ms}
        if best is None or row["nps"] > best["nps"]:
            best = row
    agent.close()
    net.close()
    return best


def selfplay_leg(blob, device, n_games, seconds, mode="crazyhouse", variants=1, is960=False, threads=1, max_plies=160,
                 input_version=1):
    """Self-play games/hour (second half of BASELINE.json's metric): `n_games` concurrent games per GPU with the
    reference's RL search settings (rl_config.py:34-65: 800 nodes +- 5 %, Batch_Size 8, Dirichlet 0.25/0.3, temperature
    0.8 decaying over 15 plies, resignation) -- crazyara_b200.selfplay.Arena."""
    from crazyara_b200.nn import NeuralNetAPI
    from crazyara_b200.selfplay import Arena, rl_settings
    st = rl_settings(mode, threads=threads, input_version=input_version)
    # Threads 1: two groups of games, each with its own agent and network buffers, searched from two host threads, so
    # that one group's tree kernels overlap the other's network forward; Threads 2 does that inside one agent
    groups = 2 if (threads == 1 and n_games % 2 == 0) else 1
    nets = [NeuralNetAPI("gpu", device, n_games // groups * st.batch_size, blob) for _ in range(groups)]
    arena = Arena(nets, st, variant=variants, n_games=n_games, device=device, is960=is960, max_plies=max_plies, seed=1)
    arena.run(max_steps=2)  # warm-up (graph capture, allocations)
    arena.finished.clear()
    arena.nodes, arena.search_ms, arena.resigned = 0, 0.0, 0
    res = arena.run(max_seconds=seconds)
    arena.close()
    for net in nets:
        net.close()
    # random weights do not finish games the way a trained network does: games still running at `max_plies` are
    # adjudicated as draws (the reference has no such limit; stated with the figure); the rate per searched move is
    # reported beside the finished games
    return {"concurrent_games": n_games, "game_groups": groups, "threads": threads, "rows_per_forward": n_games // groups * st.batch_size,
            "settings": f"RL defaults (rl_config.py): nodes 800 +-5 %, Batch_Size 8, Dirichlet eps 0.25 alpha 0.3, temperature 0.8 x 0.92^ply "
                        f"for 15 plies, resignation 90 % of games at q < -0.9; games adjudicated at {max_plies} plies (random weights)",
            "moves_per_s": res["moves_per_s"], "games_per_hour": res["games_per_hour"],
            "games_per_hour_at_100_plies": res["moves_per_s"] * 36.0,
            "games_finished_in_window": res["games"], "games_resigned": res["resigned"], "avg_plies_finished": res["avg_plies"],
            "search_nps": res["nps"], "wall_s": res["wall_s"]}


SELFPLAY_CONFIGS = {
    # BASELINE.json configs[3] / [4]: mode, variants, chess960, net family, in channels, policy channels, input version,
    # concurrent games per GPU
    "4": ("chess", 0, True, "risev33", 52, 76, 3, 8),             # 64 concurrent chess960 games over 8 GPUs
    "5": ("lichess", [2, 3], False, "risev2", 63, 84, 1, 16),      # KOTH + Three-check mixed, 16 x Batch_Size 8 = 128 rows
}


def selfplay_config_main(args, rank, local_rank, world):
    """--config 4 | 5: finished self-play games per hour."""
    mode, variants, is960, family, cin, pch, version, games = SELFPLAY_CONFIGS[args.config]
    names = {"4": "chess960 self-play, 8 concurrent games per GPU, RISEv3.3 52x8x8 -> 76x64",
             "5": "King of the Hill + Three-check mixed self-play (one MODE_LICHESS network for both), 16 concurrent games per "
                  "GPU = 128 rows per forward, RISEv2 63x8x8 -> 84x64"}
    metric = "self-play games/hr (BASELINE cfg %s)" % args.config
    if args.impl == "reference":
        if rank == 0:
            print(json.dumps({"impl": "reference", "metric": metric, "unavailable": "the reference's self-play needs its engine binary "
                              "(Stockfish fork + NN backend absent); the search alone is timed by --config M/2/3 --impl reference"}))
        return
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from crazyara_b200 import synthetic
    from crazyara_b200.weights import export_blob
    arch = make_arch(family, cin, pch)
    tmp = tempfile.mkdtemp(prefix="ara_bench_")
    blob = export_blob(synthetic.random_state_dict(arch, 0), arch, os.path.join(tmp, f"net_{rank}.arab"), input_version=version * 10)
    seconds = args.selfplay_seconds if args.selfplay_seconds > 8.0 else 30.0
    sampler = ClockSampler(local_rank)
    sampler.start()
    if dist is not None:
        dist.barrier()
    leg = selfplay_leg(blob, local_rank, games, seconds, mode=mode, variants=variants, is960=is960, threads=args.threads,
                       max_plies=200, input_version=version)
    sampler.stop_flag = True
    sampler.join(timeout=2)
    tot = [leg["games_per_hour"], leg["moves_per_s"], leg["search_nps"]]
    if dist is not None:
        t = torch.tensor(tot, device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        tot = t.tolist()
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak_tf = peaks.get("bf16_tflops_sustained", 1400.0)
        conv_tf = tot[2] / world * net_flops_per_position(arch) / 1e12  # per GPU: evaluated nodes/s x FLOP per position
        print(json.dumps({
            "metric": metric, "value": tot[0], "unit": "games/h", "n_gpus": world, "steps": 1, "warmup": 1,
            "ms_per_step": leg["wall_s"] * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f16 tensor-core operands, f32 accumulate", "data": "synthetic (seeded random weights)",
            "config": {"workload": names[args.config], "parallelism": f"replicas x{world} (independent games per GPU, no collective)",
                       "window_s": seconds, **{k: leg[k] for k in ("settings", "concurrent_games", "threads", "rows_per_forward")}},
            "e2e": {"value": tot[0], "unit": "games/h", "h2d_bytes_per_step": 280 * games, "d2h_bytes_per_step": 14392 * games,
                    "note": "the arena is end to end by construction: host game loop, per-move host<->device traffic"},
            "moves_per_s": tot[1], "search_nps": tot[2], "per_gpu": leg, "gpu_launches": -1, "clocks": sampler.summary(),
            "roofline": {"bound": "tensor", "achieved": conv_tf, "peak": peak_tf, "unit": "TFLOP/s",
                         "frac": conv_tf / peak_tf if peak_tf else None, "traffic": None,
                         "achieved_from": "searched nodes per second x FLOP per position (per GPU, over the wall time of the arena)"}}))
    if dist is not None:
        dist.destroy_process_group()


def search_leg(agent, net, steps, flush):
    """`steps` timed searches of the headline kind on an existing agent: (nodes, device ms, wall s, last result)"""
    import torch

    from crazyara_b200.engine import BoardState
    nodes, dev_ms, wall_s, last = 0, 0.0, 0.0, None
    for _ in range(steps):
        flush.fill_(1)  # L2 flush between steps (outside the timed region)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = agent.evaluate_board_state(BoardState().set("", False, agent._bench_variant))
        wall_s += time.perf_counter() - t0
        dev_ms += agent.last_go_ms()
        nodes += int(r["nodes"])
        last = r
    return nodes, dev_ms, wall_s, last


# the EvalInfo fields of a search result that --dump-outputs writes, besides the root moves and the principal variation;
# elapsed_ms and nps are timings, not results
RESULT_ARRAYS = ("visits", "q", "prior", "policy")
RESULT_SCALARS = ("root_value", "best_move_q", "visit_sum", "free_visits", "nodes", "best_idx", "node_type", "pv_len",
                  "iterations", "evals", "tree_nodes", "nodes_pre_search", "sum_select_k", "sum_depth", "error")


def dump_outputs(out_dir, result, variant_id):
    """Writes a search result (the dict MCTSAgent.evaluate_board_state returns for the start position) as
    out_dir/<name>.npy: the root's children in the search's order (moves as 16-bit move codes, visits, Q, priors, MCTS
    policy), the principal variation as move codes, and every scalar of the result, so that two builds can be compared
    output for output.  Q and priors stay float32, everything else is float64."""
    import numpy as np

    from crazyara_b200.engine import BoardState
    os.makedirs(out_dir, exist_ok=True)
    state = BoardState().set("", False, variant_id)
    arrays = {"moves": np.array([state.uci_to_action(m) for m in result["moves"]], np.float64)}
    pv = []
    for m in result["pv"]:
        pv.append(state.uci_to_action(m))
        state.do_uci(m)
    arrays["pv"] = np.array(pv, np.float64)
    for name in RESULT_ARRAYS:
        a = np.asarray(result[name])
        arrays[name] = a.astype(np.float32 if a.dtype == np.float32 else np.float64)
    for name in RESULT_SCALARS:
        arrays[name] = np.array([result[name]], np.float32 if name in ("root_value", "best_move_q") else np.float64)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="M", choices=["M", "2", "3", "4", "5"],
                    help="M: the headline workload; 2, 3: BASELINE.json's other search configurations; 4, 5: self-play")
    ap.add_argument("--sims", type=int, default=0, help="simulations per search (default: the configuration's)")
    ap.add_argument("--batch", type=int, default=0, help="Batch_Size (default: the configuration's)")
    ap.add_argument("--threads", type=int, default=2, choices=[1, 2], help="Threads: 2 = the reference's default (two logical "
                    "search threads: one selects while the other's batch is evaluated), 1 = single-threaded parity mode")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the CPU arm (profiling runs)")
    ap.add_argument("--trees", type=int, default=32, help="extra leg: concurrent searches per GPU (0 = skip)")
    ap.add_argument("--selfplay-seconds", type=float, default=8.0, help="extra leg: self-play arena window (0 = skip)")
    ap.add_argument("--selfplay-games", type=int, default=64)
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the search result of the last one "
                    "as DIR/<name>.npy (search configurations M, 2, 3 on the GPU)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.config in ("4", "5")):
        ap.error("--dump-outputs writes the GPU search result: --impl ours with --config M, 2 or 3")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.config in ("4", "5"):
        return selfplay_config_main(args, rank, local_rank, world)
    variant, vid, mode, family, cin, pch, version, d_batch, d_sims = WORKLOADS[args.config]
    batch = args.batch or d_batch
    sims = args.sims or d_sims
    net_name = "RISEv2-mobile" if family == "risev2" else "RISEv3.3"
    workload = (f"{variant} startpos, {net_name} {cin}x8x8 -> {pch}x64 policy map, Batch_Size {batch}, "
                f"Simulations {sims}, Threads {args.threads}, reference UCI defaults (node temperature 1.7, virtual_mix, "
                f"MCTS solver on, no Dirichlet/epsilon), fresh tree per step")
    metric = METRIC if args.config == "M" else f"MCTS simulations/sec (NPS) {variant} startpos batch={batch} (BASELINE cfg {args.config})"

    if args.impl == "reference":
        if rank != 0:
            return
        steps = args.steps
        warm = min(args.warmup, 1)
        nps, ms, cores, kind, sample = cpu_arm(args.config, sims, batch, args.threads, steps, warm)
        print(json.dumps({
            "impl": "reference", "metric": metric, "value": nps, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
            "warmup": warm, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic (seeded random weights, start position)",
            "config": {"workload": workload, "sample": sample},
            "cpu_baseline": {"value": nps, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": nps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        # NCCL prints its version banner on stdout at VERSION level; stdout carries exactly one JSON line
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    from crazyara_b200.engine import MCTSAgent, default_settings
    from crazyara_b200.nn import NeuralNetAPI
    from crazyara_b200.weights import export_blob
    from crazyara_b200 import synthetic  # seeded random weights (no trained weights ship with the reference)

    arch = make_arch(family, cin, pch)
    flops_pos = net_flops_per_position(arch)
    tmp = tempfile.mkdtemp(prefix="ara_bench_")
    blob = export_blob(synthetic.random_state_dict(arch, 0), arch, os.path.join(tmp, f"net_{rank}.arab"), input_version=version * 10)
    net = NeuralNetAPI("gpu", local_rank, batch, blob)
    settings = default_settings(mode, batch_size=batch, simulations=sims, threads=args.threads, input_version=version)
    agent = MCTSAgent(net, settings, local_rank, 1)
    agent._bench_variant = vid
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")  # > 126 MB L2

    search_leg(agent, net, args.warmup, flush)
    launches0 = agent.launch_count() + net.launch_count()
    sampler = ClockSampler(local_rank)
    sampler.start()
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    nodes, dev_ms, wall_s, last = search_leg(agent, net, args.steps, flush)
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    sampler.stop_flag = True
    sampler.join(timeout=2)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last, vid)
    launches = agent.launch_count() + net.launch_count() - launches0
    # phase split: CUDA events between the kernels of every iteration, which the timed searches above do without
    # (an iteration is a graph launch there) -- measured on extra searches
    agent.set_profile(True)
    n_prof = 3
    net_ms = sel_ms = app_ms = 0.0
    forwards = evals = 0
    for _ in range(n_prof):
        _, _, _, r = search_leg(agent, net, 1, flush)
        prof = agent.profile()
        net_ms += prof["net_ms"] / n_prof
        sel_ms += prof["select_ms"] / n_prof
        app_ms += prof["apply_ms"] / n_prof
        forwards += prof["net_forwards"] / n_prof
        evals += int(r["evals"]) / n_prof
    agent.set_profile(False)

    from crazyara_b200.multi import aggregate_counters
    total_nodes, max_dev_ms, max_wall, launches = aggregate_counters(nodes, dev_ms, wall_s, launches, dist, "cuda")

    # secondary legs (outside the timed region of the headline number)
    extra = {}
    if args.threads == 2:  # the single-threaded parity mode beside it
        agent.close()
        st1 = default_settings(mode, batch_size=batch, simulations=sims, threads=1, input_version=version)
        agent = MCTSAgent(net, st1, local_rank, 1)
        agent._bench_variant = vid
        search_leg(agent, net, 2, flush)
        n1, d1, w1, _ = search_leg(agent, net, max(3, args.steps // 3), flush)
        extra["threads1"] = {"nps": n1 / (d1 * 1e-3), "e2e_nps": n1 / w1, "note": "Threads 1: the deterministic parity mode "
                             "(visit counts bit-exact against the single-threaded reference)"}
    extra["predict_seam"] = predict_seam_leg(net, batch, cin, pch * 64)
    agent.close()
    net.close()
    if args.config == "M":
        if args.trees > 0:
            extra["multi_tree"] = multi_tree_leg(blob, local_rank, args.trees, batch, sims, flops_pos)
        if args.selfplay_seconds > 0:
            extra["selfplay"] = selfplay_leg(blob, local_rank, args.selfplay_games, args.selfplay_seconds)
    if dist is not None:  # whole-job figures: sums over ranks (independent replicas)
        sums = torch.tensor([extra.get("multi_tree", {}).get("nps", 0.0), extra.get("selfplay", {}).get("moves_per_s", 0.0),
                             extra.get("selfplay", {}).get("games_per_hour", 0.0)], device="cuda", dtype=torch.float64)
        dist.all_reduce(sums, op=dist.ReduceOp.SUM)
        if "multi_tree" in extra:
            extra["multi_tree"]["nps_all_gpus"] = sums[0].item()
        if "selfplay" in extra:
            extra["selfplay"]["moves_per_s_all_gpus"] = sums[1].item()
            extra["selfplay"]["games_per_hour_all_gpus"] = sums[2].item()

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak_tf = peaks.get("bf16_tflops_sustained", 1400.0)
        peak_src = "measured (MEASURED_PEAKS.json bf16_tflops_sustained)" if peaks else "fallback 1.4 PFLOP/s sustained"
        # achieved = the FLOPs of the leaves the search evaluated (not of the padded rows of its forwards) / forward time
        conv_tflops = evals * flops_pos / (net_ms * 1e-3) / 1e12 if net_ms > 0 else 0.0
        traffic = None  # DRAM bytes per launch of the dominant tensor kernel, from the committed `ncu --set full` capture
        for prof_file in ("r02_ncu_trunk_pair.json", "r02_ncu_trunk.json", "r01_ncu_rise_trunk_kernel.json"):
            try:
                k = json.load(open(os.path.join(ROOT, "profiles", prof_file)))["kernels"][0]
                scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
                traffic = (k["dram__bytes_read.sum"] * scale[k["dram__bytes_read.sum unit"]] +
                           k["dram__bytes_write.sum"] * scale[k["dram__bytes_write.sum unit"]])
                break
            except Exception:
                pass
        value = total_nodes / (max_dev_ms * 1e-3)
        e2e_value = total_nodes / max_wall
        out = {
            "metric": metric, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": max_dev_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f16 tensor-core operands, f32 accumulate (reference default Precision float16); f32/f64 search arithmetic",
            "data": f"synthetic (seeded random {net_name} weights; {variant} start position)",
            "config": {"workload": workload, "parallelism": f"replicas x{world} (one search per GPU, no collective)",
                       "l2_flush_between_steps": True, "nodes_per_step": nodes / args.steps, "threads": args.threads,
                       "tree_stream_ms_per_step" if args.threads == 2 else "select_ms_per_step": sel_ms,
                       "net_ms_per_step": net_ms, "apply_ms_per_step": app_ms, "net_forwards_per_step": forwards,
                       "best_move": last.get("best_move"), "evals_per_step": evals},
            "e2e": {"value": e2e_value, "unit": UNIT,
                    "h2d_bytes_per_step": 128 + 136 + 16, "d2h_bytes_per_step": 14392 + 4 * (2 + int(last["iterations"]) // 2)},
            "gpu_launches": int(launches),
            "clocks": sampler.summary(),
            "roofline": {"bound": "tensor", "achieved": conv_tflops, "peak": peak_tf, "unit": "TFLOP/s",
                         "frac": conv_tflops / peak_tf if peak_tf else None, "traffic": traffic,
                         "traffic_note": "rise_trunk_c_kernel, one launch of 64 positions, dram__bytes_read+write "
                                         "(profiles/r02_ncu_trunk_pair.json; cold L2: the weights + the input tile)",
                         "kernel": f"{net_name} conv stack per forward of {batch} positions: rise_trunk_c_kernel (all bottleneck "
                                   "blocks on CTA pairs, tcgen05 SS MMAs with the channels in M, one launch) + stem/policy "
                                   "conv_gemm_kernel + head kernels",
                         "achieved_from": "evaluated leaves x FLOP per position / device time of the forwards",
                         "flop_per_position": flops_pos, "peak_source": peak_src},
        }
        try:
            # the other big kernel, against ITS roofline (SURVEY 8d): select reads 32 B of header + 13 B per open child
            # (Q, n, P, vl) at every tree level -- a dependent pointer chase, so far below the HBM peak by nature
            if args.threads == 1:
                sel_bytes = 32.0 * float(last.get("sum_depth", 0)) + 13.0 * float(last.get("sum_select_k", 0))
                hbm_peak = float(peaks.get("hbm_gbs", 6500.0))
                sel_gbs = sel_bytes / (sel_ms * 1e-3) / 1e9 if sel_ms > 0 else 0.0
                out["roofline_select"] = {"bound": "hbm", "achieved": sel_gbs, "peak": hbm_peak, "unit": "GB/s",
                                          "frac": sel_gbs / hbm_peak if hbm_peak else None,
                                          "algorithmic_bytes_per_search": sel_bytes,
                                          "note": "select_kernel: one warp per tree, one dependent L2/HBM round trip per tree "
                                                  "level; latency-bound (profiles/r01_ncu_select_kernel.json)"}
        except Exception:
            pass
        if world == 1 and not args.no_cpu_baseline:
            nps, ms, cores, kind, sample = cpu_arm(args.config, sims, batch, args.threads, 2, 0)
            out["cpu_baseline"] = {"value": nps, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample}
        for k in ("threads1", "predict_seam"):
            if k in extra:
                out[k] = extra[k]
        if "multi_tree" in extra:
            mt = extra["multi_tree"]
            mt["conv_frac_of_peak"] = mt["conv_tflops"] / peak_tf if peak_tf else None
            out["multi_tree"] = mt
        if "selfplay" in extra:
            out["selfplay"] = extra["selfplay"]
        print(json.dumps(out))
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
