#!/usr/bin/env python
"""bench.py -- env-steps/sec across the ES population (BASELINE.json metric) on N B200s of one node.

Workload (BASELINE.json configs[1], SURVEY.md 8d config 2): Frostbite-shaped ES generation, population 1000
(n = 500 antithetic pairs), LargeModel conv policy (P = 4,052,658, 18 actions), 256 resident env slots per GPU (--slots), synthetic
uint8 84x84x4 observations, fixed episode length T (default 1000 env steps), population sharded over the ranks.
One "step" = one GENERATION: rollouts of this rank's shard of the population for T ticks each, then the update
(all_gather returns -> centred ranks -> ES gradient over the local noise indices -> all_reduce(g) -> Adam).

  value   device-resident: observations / rewards already in HBM when the timed region starts; ticks launched kernel by
          kernel, kernels and consecutive ticks chained by programmatic dependent launch (DNE_BENCH_GRAPH=1: CUDA graphs).
  e2e     the same generation through the public API es_distributed.es.run_master with a HOST environment: every
          tick copies that tick's observations host->device from pinned memory and the actions device->host.
  --impl reference   the reference worker/master loop restated on the CPU (oracle/cpu_worker.py) on all host cores.

Timing: >= 3 warm-up steps; device timing with CUDA events bracketed by barrier + synchronize, max over ranks.
Every tick streams >= 1 GB of noise slices (>> 126 MB L2) so no input survives in L2 between timed iterations
(config.l2: "inputs larger than L2").
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "deep-neuroevolution_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np   # noqa: E402

NET = "LargeModel"
POP = 1000
SLOTS = 256            # BASELINE.json configs[1]: 256 parallel envs per GPU (the run uses min(SLOTS, 2 * local pairs))
SIGMA, L2, LR = 0.005, 0.005, 0.01          # configurations/frostbite_es.json


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference", "cpu-sample", "gpu-ref-proxy"])
    ap.add_argument("--workload", default="es", choices=["es", "mlp", "ga", "nsr"],
                    help="es = BASELINE.json configs[1] (the contract's default line); mlp / ga / nsr = configs[4] / [2] / [3] "
                         "(bench_workloads.py), same JSON contract")
    ap.add_argument("--episode-len", type=int, default=int(os.environ.get("DNE_BENCH_T", 1000)))
    ap.add_argument("--pop", type=int, default=POP)
    ap.add_argument("--slots", type=int, default=SLOTS)
    ap.add_argument("--noise-count", type=int, default=int(os.environ.get("DNE_NOISE_COUNT", 250_000_000)))
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-sample-steps", type=int, default=40, help="env steps per episode in the CPU sample")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed generation computed as DIR/<name>.npy "
                         "(es workload, b200 impl): the inputs are seeded, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and (args.impl != "b200" or args.workload != "es"):
        ap.error("--dump-outputs is implemented for --impl b200 --workload es")
    return args


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback"


# ---------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        time.sleep(0.05)
        sm = [float(r[1]) for r in self.rows if len(r) >= 8 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 8 and r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 8 for i in range(4) if r[4 + i].lower().startswith("active")})
        def num(x):
            try:
                return float(x)
            except ValueError:
                return None
        pw = [num(r[3]) for r in self.rows if len(r) >= 8 and num(r[3]) is not None]
        lim = []
        try:                                                      # one separate query: an unknown field must not cost the clock samples
            out = subprocess.run(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=enforced.power.limit",
                                  "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=10).stdout
            lim = [v for v in (num(x.strip()) for x in out.splitlines()) if v is not None]
        except Exception:
            pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm), "power_w": float(np.median(pw)) if pw else None,
                "power_limit_w": max(lim) if lim else None}


# ---------------------------------------------------------------------------------------------------------------
def exp_dict(args):
    """The experiment the e2e leg drives through es_distributed.es.run_master -- configurations/frostbite_es.json
    with the headline population / policy (BASELINE.json configs[1])."""
    return {
        "config": {"calc_obstat_prob": 0.0, "episodes_per_batch": args.pop, "eval_prob": 0.0, "l2coeff": L2,
                   "noise_stdev": SIGMA, "snapshot_freq": 0, "timesteps_per_batch": 1,
                   "return_proc_mode": "centered_rank", "episode_cutoff_mode": args.episode_len},
        "env_id": "FrostbiteNoFrameskip-v4", "synthetic_episode_len": args.episode_len,
        "optimizer": {"args": {"stepsize": LR}, "type": "adam"},
        "policy": {"args": {}, "type": "LargeModelPolicy"},
    }


def run_b200(args):
    import torch
    import torch.distributed as dist
    from dne import _ffi as F, nets, shard
    from dne.engine import ESUpdate, SlotForward, make_context
    from dne.noise import SharedNoiseTable
    import ctypes as C

    rank, world, local = shard.init_from_env("nccl")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    peaks, peak_src = load_peaks()
    L = F.lib()
    if os.environ.get("DNE_GEMV_CTAS"):
        F.check(L.dne_set_option(b"gemv_ctas_per_sm", int(os.environ["DNE_GEMV_CTAS"])))
    for kv in filter(None, os.environ.get("DNE_OPTS", "").split(",")):       # dev A/B switches: "name=value,name=value"
        k, v = kv.split("=")
        F.check(L.dne_set_option(k.encode(), int(v)))

    t0 = time.time()
    noise = SharedNoiseTable(count=args.noise_count, device=dev)
    ctx = make_context(local, noise)
    t_noise = time.time() - t0
    net = nets.make_net(NET)
    P = net.num_params
    T, n_pairs = args.episode_len, args.pop // 2
    rs = np.random.RandomState(0)
    theta0 = (rs.randn(P) * 0.05).astype(np.float32)           # random-init weights of the named architecture

    # ------------------------------------------------------------------ value: device-resident generation
    lo, hi = shard.shard_bounds(n_pairs, rank, world)
    upd = ESUpdate(ctx, theta0, "adam", stepsize=LR)
    # Slot tables.  Default = BASELINE configs[1]: 256 resident env slots per GPU in ONE table on one stream (four waves
    # of 128 pairs per generation at pop 1000): every kernel runs alone, so the per-launch GEMV timing in `roofline` and
    # the ncu launch list describe the same schedule.  `--slots 1024` gives every antithetic pair a resident slot pair
    # (one wave per generation) split over 4 tables on 4 streams, whose conv chains overlap each other's HBM-bound
    # GEMV: r01 624K vs 527-540K env-steps/s (profiles/r01_bench_n1_1000slots.json; tools/sweep_overlap.py).
    # DNE_BENCH_STREAMS overrides NS; DNE_BENCH_PHASED=1 adds the phase-event hand-off (dne_set_phase_events).
    pairs_local = hi - lo
    slots = max(2, min(args.slots, 2 * pairs_local))
    NS = int(os.environ.get("DNE_BENCH_STREAMS", "4" if slots >= 768 else ("2" if slots >= 384 else "1")))
    part = 2 * (-(-(slots // 2) // NS))                          # whole antithetic pairs per table
    slots = part * NS
    sfs = [SlotForward(ctx, net, part) for _ in range(NS)]
    streams = [torch.cuda.Stream(device=dev) for _ in range(NS)]
    PHASED = os.environ.get("DNE_BENCH_PHASED", "1" if NS > 2 else "0") == "1"
    PHASE_MODE = int(os.environ.get("DNE_PHASE_MODE", "1"))
    phase_ev = [torch.cuda.Event() for _ in range(max(NS, 2))]
    for e in phase_ev:
        e.record()                                               # materialise the handles
    R = 4                                                        # observation pool blocks, rotated every tick
    gen = torch.Generator(device=dev)
    gen.manual_seed(rank)                                        # same arguments -> same observations and rewards
    pool = torch.randint(0, 256, (R, slots, 84, 84, 4), dtype=torch.uint8, device=dev, generator=gen)
    rew_pool = (torch.rand(64, slots, device=dev, generator=gen) < 0.05).float() * 10.0
    ret_acc = torch.zeros(slots, device=dev)
    idx_stream = np.random.RandomState(1)
    tally = {"launches": 0, "pairs": 0}
    net_ref = C.byref(net.desc)
    for sf in sfs:                                                # materialise the optional slot-table tensors once
        sf.set_slots(np.zeros(part, np.int64), np.zeros(part, np.float32), active=np.ones(part, np.uint8))
    fwd_args = [(F.ptr(sf.noise_idx), F.ptr(sf.scale), F.ptr(sf.active), F.ptr(sf.actions), F.ptr(sf.logits),
                 F.ptr(sf.ws), sf.ws.numel()) for sf in sfs]
    part_active = [False] * NS
    obs_ptr = [[F.ptr(pool[r][h * part:(h + 1) * part]) for h in range(NS)] for r in range(R)]
    stream_ptr = [C.c_void_p(s.cuda_stream) for s in streams]
    ev_ptr = [C.c_void_p(e.cuda_event) for e in phase_ev]

    KERNELS_PER_TICK = 6          # conv1-3, theta GEMM, noise GEMV, combine+head (LargeModel, default options)
    # Tick launch.  Default: kernel by kernel on one stream, the six kernels AND consecutive ticks chained by programmatic
    # dependent launch (DESIGN 3.1; dne_set_option("chain_ticks", 1): with device-resident observations the stream's previous
    # kernel of a tick's first convolution is the previous tick's head) -- interleaved A/B (tools/ab_tick.py): 2-5 us per tick
    # faster than one CUDA graph per tick, whose launch boundary is a full dependency.  DNE_BENCH_GRAPH=1 replays graphs.
    USE_GRAPH = os.environ.get("DNE_BENCH_GRAPH", "0") == "1"
    CHAIN = (not USE_GRAPH) and os.environ.get("DNE_BENCH_CHAIN", "1") == "1"
    if NS >= 2 and PHASED:
        USE_GRAPH = False        # the phase-event hand-off between slot tables (cross-stream events) is not captured
    if NS >= 2 and PHASED:
        CHAIN = False
    PROF_EVERY = 16              # every 16th tick carries the CUDA-event records around the GEMV (they break the PDL chain there)
    graphs = {}
    prof_state = {"on": False}

    BREAKDOWN = os.environ.get("DNE_BENCH_BREAKDOWN", "0") == "1"     # diagnostic: adds synchronisations, not a bench value
    bd = []

    def mark(tag, sync=True):
        if BREAKDOWN:
            if sync:
                torch.cuda.synchronize()
            bd.append((tag, time.perf_counter()))

    rollout_ev = []              # (start, end) CUDA events around the rollout part of every generation (this rank's own work)
    last = {}                    # the latest generation's results (device tensors; read back only by --dump-outputs)

    def generation_value():
        mark("start")
        ev_a, ev_b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev_a.record()
        idx_all = np.array([noise.sample_index(idx_stream, P) for _ in range(n_pairs)], dtype=np.int64)
        my = idx_all[lo:hi]
        returns = torch.zeros(len(my), 2, device=dev)
        pairs_per_wave = slots // 2
        cur = torch.cuda.current_stream()
        for w0 in range(0, len(my), pairs_per_wave):
            wave = my[w0:w0 + pairs_per_wave]
            npw = len(wave)
            per = -(-npw // NS)                                   # pairs per stream partition
            parts = [wave[h * per:(h + 1) * per] for h in range(NS)]
            last["active_slots"] = [2 * len(p) for p in parts]
            for h in range(NS):
                k = len(parts[h])
                act = np.zeros(part, dtype=np.uint8)
                act[:2 * k] = 1
                ii = np.zeros(part, dtype=np.int64)
                ii[:2 * k] = np.repeat(parts[h], 2)
                sc = np.tile([SIGMA, -SIGMA], part // 2).astype(np.float32)
                sfs[h].set_slots(ii, sc, active=act)
                part_active[h] = 2 * k < part
            ret_acc.zero_()
            for s in streams:
                s.wait_stream(cur)
            # hot loop: raw C-ABI calls with pre-built ctypes arguments (no per-tick tensor slicing / stream context
            # managers: at 4 slot tables the Python overhead of those was the bottleneck)
            live = [h for h in range(NS) if len(parts[h]) > 0]
            tally["launches"] += T * len(live)
            tally["pairs"] += T * sum(len(parts[h]) for h in live)
            fwd = L.dne_perturb_forward_conv
            set_ev = L.dne_set_phase_events
            theta_p = F.ptr(upd.theta)
            for h in live:           # once per theta (the Adam step of the previous generation dropped the prepared entry)
                with torch.cuda.stream(streams[h]):
                    sfs[h].prepare(upd.theta, part)
            def tick(h, r):
                a = fwd_args[h]
                rc = fwd(ctx.handle, net_ref, theta_p, a[0], a[1], None, a[2] if part_active[h] else None, part, 1,
                         obs_ptr[r][h], None, a[3], a[4], a[5], a[6], stream_ptr[h])
                if rc:
                    F.check(rc)
            mark("wave_setup")
            for t in range(T):
                r = t % R
                for h in live:
                    if NS >= 2 and PHASED:
                        set_ev(ctx.handle, ev_ptr[(h - 1) % NS], ev_ptr[h], PHASE_MODE)
                    if USE_GRAPH and (t % PROF_EVERY) != 0:
                        # the tick's kernel sequence replayed as one CUDA graph (captured once per table / observation
                        # block / active-mask variant): no per-kernel launch gaps.  Every PROF_EVERY-th tick is launched
                        # kernel by kernel so that the GEMV of the timed region is still timed with CUDA events.
                        key = (h, r, part_active[h])
                        g = graphs.get(key)
                        if g is None:
                            L.dne_profile_enable(ctx.handle, 0, 0)
                            torch.cuda.synchronize()
                            g = torch.cuda.CUDAGraph()
                            with torch.cuda.graph(g, stream=streams[h]):
                                tick(h, r)
                            graphs[key] = g
                        with torch.cuda.stream(streams[h]):
                            g.replay()
                        tally["graph_kernels"] = tally.get("graph_kernels", 0) + KERNELS_PER_TICK
                    else:
                        if prof_state["on"] and (t % PROF_EVERY) == 0:
                            L.dne_profile_enable(ctx.handle, 2, 0)          # resume (keeps the samples taken so far)
                            tick(h, r)
                            L.dne_profile_enable(ctx.handle, 0, 0)          # pause: the other ticks carry no event records
                        else:
                            tick(h, r)
                ret_acc.add_(rew_pool[t % 64])                     # one bookkeeping op per tick, main stream
            mark("ticks_enqueued", sync=False)
            for s in streams:
                cur.wait_stream(s)
            mark("ticks_done")
            r = torch.cat([ret_acc[h * part:h * part + 2 * len(parts[h])] for h in range(NS)]).view(-1, 2)
            returns[w0:w0 + npw] = r
        ev_b.record()
        rollout_ev.append((ev_a, ev_b))
        allret = shard.all_gather_rows(returns, n_pairs)
        proc, _ = upd.centered_ranks(allret)
        g = upd.gradient(proc[lo:hi].contiguous(), torch.from_numpy(my).to(dev), denom=2 * n_pairs)
        shard.all_reduce_sum_(g)
        upd.step(L2)
        last.update(returns=allret, centered_ranks=proc, gradient=g)
        mark("update")
        if BREAKDOWN:
            t0 = bd[0][1]
            print(f"[breakdown r{rank}] " + "  ".join(f"{tag}=+{(t - t0) * 1e3:.2f}ms" for tag, t in bd[1:]), file=sys.stderr, flush=True)
        bd.clear()

    def timed(fn, steps, warmup, profile=False):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        shard.barrier()
        torch.cuda.synchronize()
        if profile:
            F.check(L.dne_profile_enable(ctx.handle, 1, 16384))
            prof_state["on"] = True
            F.check(L.dne_profile_enable(ctx.handle, 0, 0))                 # paused; resumed around every 16th tick
        L.dne_launch_count(1)
        tally["graph_kernels"] = 0
        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        shard.barrier()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        clocks = sampler.stop() if rank == 0 else None
        launches = L.dne_launch_count(0) + tally.get("graph_kernels", 0)
        prof = None
        if profile:
            n, tot = C.c_int(), C.c_double()
            prof_state["on"] = False
            F.check(L.dne_profile_enable(ctx.handle, 0, 0))
            F.check(L.dne_profile_read(ctx.handle, C.byref(n), C.byref(tot)))
            prof = (n.value, tot.value)
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), clocks, launches, prof

    if CHAIN:
        F.check(L.dne_set_option(b"chain_ticks", 1))
    try:
        ms_val, clocks, launches, prof = timed(generation_value, args.steps, args.warmup, profile=True)
    finally:
        F.check(L.dne_set_option(b"chain_ticks", 0))
    if args.dump_outputs and rank == 0:
        # rank 0's results of the last timed generation: the updated parameters, the update's inputs, and the final tick's
        # logits / actions on the slots the last wave used (before parity_check reuses the slot tables)
        n_act = last["active_slots"]
        dump_outputs(args.dump_outputs, {
            "theta": upd.theta, "gradient": last["gradient"], "returns": last["returns"],
            "centered_ranks": last["centered_ranks"],
            "logits": torch.cat([sfs[h].logits[:n_act[h]] for h in range(NS)]),
            "actions": torch.cat([sfs[h].actions[:n_act[h]] for h in range(NS)])})
    # this rank's own rollout time per generation (before the all_gather that synchronises the ranks): rank skew shows here
    my_roll = sum(a.elapsed_time(b) for a, b in rollout_ev[-args.steps:]) / args.steps
    roll_t = torch.tensor([my_roll], dtype=torch.float64, device=dev)
    roll_all = [torch.zeros_like(roll_t) for _ in range(world)]
    if world > 1:
        dist.all_gather(roll_all, roll_t)
    else:
        roll_all = [roll_t]
    rank_rollout_ms = [round(float(t.item()), 3) for t in roll_all]
    env_steps = args.steps * args.pop * T
    value = env_steps / (ms_val / 1e3)

    # roofline of the dominant kernel: dense_noise_gemv on the fc layer (97.8% of the weight bytes)
    fc = net.layers[3]
    n_timed, tot_ms = prof
    # algorithmic bytes one launch must read: one noise slice per PAIR (pair-shared) for the fc weights.  The
    # SURVEY 8d per-env-step figure (4*P + obs + action, every member reading its own slice) is reported beside it.
    pairs_per_launch = tally["pairs"] / max(tally["launches"], 1)      # average over every forward of the run
    alg_bytes = pairs_per_launch * 4.0 * fc.cin * fc.cout
    survey_bytes = 2 * pairs_per_launch * (4.0 * P + 84 * 84 * 4 + 4)
    avg_ms = tot_ms / max(n_timed, 1)
    achieved = alg_bytes / (avg_ms * 1e-3) / 1e9 if n_timed else None
    traffic = None
    try:      # DRAM bytes of the same kernel from the committed ncu --set full capture, scaled to this run's pairs/launch
        with open(os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")) as f:
            tj = json.load(f)["gemv_bulk_kernel"]
        traffic = tj["dram_bytes_per_launch"] * pairs_per_launch / tj["pairs_per_launch"]
    except Exception:
        pass
    roofline = {"bound": "hbm",
                "kernel": "gemv_bulk_kernel<2> (fc 7744x512 noise GEMV: cp.async.bulk ring, slice shared by the +/- pair)",
                "achieved": achieved, "peak": peaks["hbm_gbs"], "peak_source": peak_src, "unit": "GB/s",
                "frac": (achieved / peaks["hbm_gbs"]) if achieved else None,
                "traffic": traffic, "launches_timed": n_timed, "avg_launch_ms": avg_ms,
                "algorithmic_bytes_per_launch": alg_bytes, "pairs_per_launch": pairs_per_launch,
                "survey_bytes_per_launch": survey_bytes,
                "schedule": f"{NS} slot table(s) on {NS} stream(s)" + ("; the timed GEMV launches overlap the other table's "
                            "conv / tensor-core kernels, so avg_launch_ms includes that contention" if NS > 1 else ""),
                "whole_run_frac": (args.steps * (hi - lo) * T * 4.0 * fc.cin * fc.cout / (ms_val * 1e-3) / 1e9 / peaks["hbm_gbs"]),
                "frac_survey_bytes": (survey_bytes / (avg_ms * 1e-3) / 1e9 / peaks["hbm_gbs"]) if n_timed else None,
                "note": "algorithmic bytes = one fc noise slice per antithetic PAIR (read once for both members); "
                        "survey_bytes = SURVEY 8d figure (4P + obs + action per env-step, every member its own slice). "
                        "~5% of the slice bytes hit in L2 (random 16 MB slices of a 1 GB table overlap), hence frac > 1."}

    # ------------------------------------------------------------------ output check of the benchmarked kernels
    parity = parity_check(L, ctx, net, sfs[0], upd.theta, obs_ptr[0][0], pool[0][:part], part)

    # ------------------------------------------------------------------ e2e: public API, host environment
    e2e = None
    if not args.no_e2e:
        from es_distributed import es as ES
        from dne.envs import SyntheticAtariEnv
        from es_distributed import tabular_logger
        tabular_logger.set_quiet(True)          # stdout carries exactly one JSON line
        ES.set_default_noise(noise)
        ES._STATE["ctx"] = ctx
        slots_e2e = -(-slots // 4) * 4                       # RolloutRunner: multiple of group (2) x pipeline halves (2)
        env = SyntheticAtariEnv(slots_e2e, episode_len=T, seed=rank)
        marks = {0: time.perf_counter()}        # iterations count from 1: with --warmup 0 the window opens here

        io = {"h2d": 0, "d2h": 0}

        def on_it(it, stats, extra):
            if it > args.warmup:
                io["h2d"] += extra["forward_launches"] * extra["slots_per_launch"] * 84 * 84 * 4
                io["d2h"] += extra["forward_launches"] * extra["slots_per_launch"] * 4
            if it == args.warmup or it == args.warmup + args.steps:
                torch.cuda.synchronize()
                shard.barrier()
                torch.cuda.synchronize()
                marks[it] = time.perf_counter()
        ES.run_master(None, None, exp_dict(args), max_iterations=args.warmup + args.steps, n_slots=slots_e2e,
                      env=env, noise=noise, seed=0, on_iteration=on_it)
        dt = marks[args.warmup + args.steps] - marks[args.warmup]
        tt = torch.tensor([dt], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dt = float(tt.item())
        e2e = {"value": env_steps / dt, "unit": "env-steps/s", "ms_per_step": dt * 1e3 / args.steps,
               "h2d_bytes_per_step": int(io["h2d"] / args.steps), "d2h_bytes_per_step": int(io["d2h"] / args.steps),
               "bytes_scope": "rank 0's copies per generation (every rank copies the same amount +-1 pair)",
               "api": "es_distributed.es.run_master(exp) + dne.envs.SyntheticAtariEnv (host, pinned)"}

    # ------------------------------------------------------------------ CPU baseline (rank 0, N == 1 only)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline(args, noise_host=None)

    if rank == 0:
        line = {
            "metric": "env-steps/sec across ES population (whole box)", "value": value, "unit": "env-steps/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_val / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"frostbite_es_pop{args.pop}_LargeModel_T{T}",
                       "population": args.pop, "noise_pairs": n_pairs, "policy": "LargeModel (P=4052658, 18 actions)",
                       "env_slots_per_gpu": slots, "slot_tables": NS, "episode_len": T, "noise_table": args.noise_count,
                       "tick_launch": "CUDA graph replay (6 kernels; every 16th tick kernel by kernel for the CUDA-event GEMV timing)"
                                      if USE_GRAPH else ("kernel by kernel, kernels and consecutive ticks chained by programmatic dependent "
                                                         "launch (every 16th tick carries the CUDA-event GEMV timing)" if CHAIN else "kernel by kernel"),
                       "sharding": f"population over {world} rank(s); all_gather(returns)+all_reduce(g)",
                       "l2": "inputs larger than L2 (>=1 GB of noise slices streamed per tick)",
                       "step": "one generation (rollouts + update)"},
            "generation_wall_clock_s": ms_val / args.steps / 1e3,
            "parity_checked": bool(parity and parity["checked"]), "parity": parity,
            "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu,
            "noise_table_build_s": t_noise,
            "rank_rollout_ms": rank_rollout_ms,     # per rank: device time of its rollouts per generation (ms_per_step = slowest rank + exchange + update)
        }
        _emit(line)
    if world > 1:
        dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------------------------
DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, tensors):
    """Write each tensor as out_dir/<name>.npy: float64 stays float64, everything else becomes float32 (integer actions are
    exact in float32)."""
    arrays = {}
    for name, t in tensors.items():
        a = t.detach().cpu().numpy()
        arrays[name] = a if a.dtype == np.float64 else a.astype(np.float32)
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ---------------------------------------------------------------------------------------------------------------
def parity_check(L, ctx, net, sf, theta, obs_p, obs, n_slots):
    """After the timed region: one tick of the benchmarked slot table (whatever indices / active mask the last wave
    left in it) through the benchmarked kernels (tcgen05 convolutions + TMA bulk-copy GEMV) and through the plain fp32
    SIMT kernels (dne_set_option conv_tc = 0, gemv_bulk = 0; same C ABI, no oracle involved): logits within twice the
    forward bound of tests/test_gpu_parity.py on every active slot, identical actions wherever the top-2 gap decides."""
    import ctypes as C
    import torch
    from dne import _ffi as F

    def one(fast):
        F.check(L.dne_set_option(b"conv_tc", 2 if fast else 0))
        F.check(L.dne_set_option(b"gemv_bulk", fast))
        sf.logits.fill_(0)
        sf.actions.fill_(-1)
        F.check(L.dne_perturb_forward_conv(ctx.handle, C.byref(net.desc), F.ptr(theta), F.ptr(sf.noise_idx), F.ptr(sf.scale),
                                           None, F.ptr(sf.active), n_slots, 1, obs_p, None, F.ptr(sf.actions),
                                           F.ptr(sf.logits), F.ptr(sf.ws), sf.ws.numel(), F.stream_ptr()))
        torch.cuda.synchronize()
        return sf.logits.clone(), sf.actions.clone()
    try:
        lf, af = one(1)
        ls, as_ = one(0)
    finally:
        L.dne_set_option(b"conv_tc", 2)
        L.dne_set_option(b"gemv_bulk", 1)
    act = sf.active.bool() if sf.active is not None else torch.ones(n_slots, dtype=torch.bool, device=lf.device)
    lf, ls, af, as_ = lf[act], ls[act], af[act], as_[act]
    bound = 4e-5 * torch.clamp(ls.abs().max(dim=1).values, min=1.0)
    err = (lf - ls).abs().max(dim=1).values
    srt = ls.sort(dim=1).values
    decided = (srt[:, -1] - srt[:, -2]) > 2 * bound
    ok = bool((err <= bound).all()) and bool(torch.equal(af[decided], as_[decided])) and bool(torch.isfinite(lf).all())
    if not ok:
        raise RuntimeError(f"bench parity check failed: max |dlogit| {float(err.max()):.3e} (bound {float(bound.min()):.3e})")
    return {"checked": True, "slots": int(act.sum()), "max_abs_dlogit": float(err.max()), "bound": float(bound.min()),
            "decided_frac": float(decided.float().mean()),
            "against": "fp32 SIMT kernels of the same library (conv_tc=0, gemv_bulk=0) on the benchmarked slot table"}


# ---------------------------------------------------------------------------------------------------------------
def cpu_baseline(args, noise_host):
    """Run the bounded CPU sample in a FRESH process (forking 100+ workers out of a process that holds a CUDA context
    and pinned pools is slow and would distort the sample)."""
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "cpu-sample", "--pop", str(args.pop),
           "--episode-len", str(args.episode_len), "--cpu-sample-steps", str(args.cpu_sample_steps),
           "--noise-count", str(args.noise_count)]
    try:
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=300,
                           env={k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")})
        return json.loads(r.stdout.strip().splitlines()[-1])
    except Exception as e:          # never lose the GPU numbers to a baseline hiccup
        return {"value": None, "unit": "env-steps/s", "cores": None, "kind": "port", "sample": f"failed: {e!r}"}


def cpu_sample(args, noise_host=None):
    """Reference worker loop + master update on the host cores, bounded sample (oracle/cpu_worker.py)."""
    from oracle import oracle as O
    from oracle import cpu_worker as W
    cores = W.host_cores()
    net = O.make_net(NET)
    P = net.num_params
    count = max(P + 1_000_000, min(args.noise_count, 30_000_000))   # bounded table for the sample (same slices' statistics)
    if noise_host is None:
        noise_host = O.noise_table(count)
    rs = np.random.RandomState(0)
    theta = (rs.randn(P) * 0.05).astype(np.float32)
    n_pairs = cores                                                  # one pair per worker process
    idx = rs.randint(0, len(noise_host) - P + 1, size=n_pairs).astype(np.int64)
    Ts = args.cpu_sample_steps
    # three samples, median per-env-step time (workers pinned one per core: oracle/cpu_worker.py): a single sample of a
    # DRAM-bound loop on a shared host swung 5x between two driver boxes in r01
    runs = [W.measure_workers(NET, noise_host, theta, list(idx), Ts, SIGMA, cores, seed=r) for r in range(3)]
    runs.sort(key=lambda r: r[3])
    steps, wall, t_setup, t_step = runs[1]
    gen_s, upd_full, n_upd = _cpu_generation_seconds(args, W, noise_host, theta, rs, cores, t_setup, t_step)
    fc_bytes = 4.0 * 7744 * 512                                    # the fc weights every env step streams on the CPU too
    return {"value": args.pop * args.episode_len / gen_s, "unit": "env-steps/s", "cores": cores, "kind": "port",
            "sample": f"median of 3 samples, each {n_pairs} antithetic pairs x {Ts} env steps on {cores} forked 1-thread workers "
                      f"pinned one per core ({steps} steps in {wall:.1f}s wall; {t_step * 1e3:.2f} ms/env-step, {t_setup * 1e3:.1f} ms set-up per "
                      f"episode, extrapolated to T={args.episode_len}) + master update on {n_upd} slices scaled to {args.pop // 2}",
            "ms_per_env_step_per_core": t_step * 1e3, "ms_per_env_step_per_core_samples": [r[3] * 1e3 for r in runs],
            "setup_ms_per_episode": t_setup * 1e3, "host_dram_GBs_implied": cores * fc_bytes / t_step / 1e9,
            "master_update_s_per_generation": upd_full, "generation_wall_clock_s": gen_s}


def _cpu_generation_seconds(args, W, noise_host, theta, rs, cores, t_setup, t_step):
    """Extrapolate the bounded sample to one full generation: pop episodes of T steps spread over `cores` workers
    (set-up once per episode) + the single-process master update (es.py:273-301) measured on 50 slices."""
    P = theta.size
    n_upd = 50
    uidx = rs.randint(0, len(noise_host) - P + 1, size=n_upd).astype(np.int64)
    ret = rs.permutation(2 * n_upd).astype(np.float32).reshape(n_upd, 2)
    upd_s, _ = W.measure_master_update(noise_host, theta, uidx, ret)
    upd_full = upd_s * (args.pop // 2) / n_upd
    rollout_s = args.pop * (t_setup + args.episode_len * t_step) / cores
    return rollout_s + upd_full, upd_full, n_upd


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path (restated: oracle/cpu_worker.py), all host
    cores, same metric / config; each step is a bounded sample of the workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle as O
    from oracle import cpu_worker as W
    cores = W.host_cores()
    net = O.make_net(NET)
    P = net.num_params
    noise_host = O.noise_table(max(P + 1_000_000, min(args.noise_count, 30_000_000)))
    rs = np.random.RandomState(0)
    theta = (rs.randn(P) * 0.05).astype(np.float32)
    Ts = args.cpu_sample_steps
    n_upd = 50
    vals, times = [], []
    for it in range(args.warmup + args.steps):
        idx = rs.randint(0, len(noise_host) - P + 1, size=cores).astype(np.int64)
        steps, wall, t_setup, t_step = W.measure_workers(NET, noise_host, theta, list(idx), Ts, SIGMA, cores, seed=it)
        gen_s, _, _ = _cpu_generation_seconds(args, W, noise_host, theta, rs, cores, t_setup, t_step)
        if it >= args.warmup:
            vals.append(args.pop * args.episode_len / gen_s)
            times.append(wall)
    v = float(np.mean(vals))
    sample = (f"per step: {cores} antithetic pairs x {Ts} env steps on {cores} forked 1-thread workers + master update "
              f"on {n_upd} slices scaled to {args.pop // 2}; generation time extrapolated to pop {args.pop} x T {args.episode_len}")
    _emit({
        "impl": "reference", "metric": "env-steps/sec across ES population (whole box)", "value": v,
        "unit": "env-steps/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": float(np.mean(times)) * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"frostbite_es_pop{args.pop}_LargeModel_T{args.episode_len}",
                   "population": args.pop, "policy": "LargeModel (P=4052658, 18 actions)", "episode_len": args.episode_len},
        "cpu_baseline": {"value": v, "unit": "env-steps/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "reference TF/redis workers cannot run (tensorflow, gym, ALE, redis absent): CPU restatement of "
                "es.py:411-426 + policies.py:399-409 and es.py:273-301 (oracle/cpu_worker.py)"})


def _emit(obj):
    """The ONE JSON line of the contract, written to the process's original stdout."""
    os.write(_REAL_STDOUT, (json.dumps(obj) + "\n").encode())


if __name__ == "__main__":
    # stdout carries exactly one JSON line: everything else that libraries print to fd 1 (NCCL's version banner,
    # loggers) is routed to stderr for the whole run.
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    a = parse()
    if a.impl == "cpu-sample":
        _emit(cpu_sample(a))
    elif a.impl == "reference":
        run_reference(a)
    elif a.impl == "gpu-ref-proxy":
        import bench_workloads
        bench_workloads.run_gpu_ref_proxy(a, _emit, ClockSampler)
    elif a.workload != "es":
        import bench_workloads
        bench_workloads.run(a, _emit, ClockSampler, load_peaks)
    else:
        run_b200(a)
