#!/usr/bin/env python
"""bench.py — node state-transitions/s of ApplyState on B200 (BASELINE.json metric).

A "step" is one ApplyState pass over one synthetic cluster snapshot. Workload at N=1: BASELINE config C3
(10 M nodes, MaxParallelUpgrades=100, MaxUnavailable=25%). At N>1 every rank holds one 10 M-node contiguous
shard of an N x 10 M-node cluster (config C5 at N=8): weak scaling, one exchange of the constraint counters
per step.

  value      device-resident inputs, CUDA-event time of K steps, max over ranks, whole-job nodes/s
  e2e        the same step through the host-pointer C ABI, pinned host arrays in, H2D + kernels + D2H inside the
             timed region: ust_apply_state_packed (uint16 revisions / int8 DaemonSet indices on the host side,
             8 B/node up; --e2e-format wide = ust_apply_state, 13 B/node up)
  e2e_delta  (N=1, informative) ust_apply_state_delta: the snapshot stays resident, 1 % of the nodes are
             re-encoded and uploaded per step, everything is evaluated, all outputs come back
  roofline   dominant kernel (ust_stream_kernel): 16 algorithmic bytes per node / average step duration
             (CUDA events), against the measured HBM copy bandwidth of MEASURED_PEAKS.json
  by_config  (N=1) the other BASELINE configurations and the paths the headline does not take, each timed the same
             way and each verified against the SoA oracle on the timed buffers:
               C2      1 M nodes, no limits
               C3_cut  C3's data under MaxParallelUpgrades=0 / MaxUnavailable=30 %: the slot budget cuts in the
                       middle of the array. first_call_us: every call under a policy the previous call did not
                       have (no speculation hint); steady_us: same policy, every buffer set perturbed (0.1 % of
                       the state bytes differ from set to set), so the hint is stale but close
               C4      10 M nodes + ~300 M workload pods in CSR lists, pod deletion and drain enabled
               small   100 k and 10 k nodes (what a reconcile of a real cluster sees): us per call
  N>1        parity_checked: after the timed region the shards' outputs are gathered on rank 0 and compared with the
             SoA oracle on the unsharded cluster, for the timed policy and for one whose budget cuts mid-cluster;
             exchange_us = step time minus the step time of the same shard on a handle without a communicator
  cpu_baseline / --impl reference   the oracle's reference-shaped restatement of the Go loop (1 thread —
             the reference's ApplyState is strictly sequential), bounded sample of the same workload;
             cpu_baseline.soa_scalar_1core: the same decisions over the SoA encoding (the generous CPU baseline)

--dump-outputs DIR writes what the last timed step returned to its caller as float32 / float64 .npy files, so that
two builds can be compared output for output (the inputs are a pure function of the arguments):
  node_index   which nodes the other arrays hold: all of them, or a fixed seeded sample of DUMP_NODES sorted indices
  next_state   next_state of those nodes
  actions      action bits of those nodes
  outcome      actuator outcome of those nodes (--pods only)
  counters     every ust_counters field except `reserved`, in declaration order (hist[16] first)
At N>1 each rank writes its own shard's files with a _rank<r> suffix and a proportionally smaller sample.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "k8s-operator-libs_b200"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

BYTES_PER_NODE = 16  # state 1 + flags 4 + pod_rev 4 + ds_idx 4 read, next_state 1 + actions 2 written (DESIGN.md §4)
SHARD_NODES = 10_000_000
CPU_SAMPLE_NODES = 1_000_000
L2_BYTES = 126 * 1024 * 1024
DUMP_NODES = 1 << 21  # --dump-outputs: 8 + 4 + 4 (+ 4) bytes per sampled node, at most 40 MB in all


def ncu_traffic():
    """(dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, name of the committed ncu
    capture it comes from). This run does not measure it (a number taken under ncu is never a bench value)."""
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_ncu_traffic.json")))
    if not files:
        return None, None
    try:
        with open(files[-1]) as f:
            d = json.load(f)
        return d["dram_bytes_read"] + d["dram_bytes_write"], "profiles/" + os.path.basename(files[-1]) + " (" + d.get("kernel", "?") + ")"
    except Exception:
        return None, None


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            for k, nm in enumerate(names):
                if len(r) > 4 + k and r[4 + k].lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def cpu_reference_rate(policy, soa, reps, variant=0):
    """variant 0: reference-shaped oracle (ApplyState only, objects built untimed); variant 1: the same decisions over
    the struct-of-arrays encoding, scalar loop (BASELINE.md §2 `cpu_soa`: the generous CPU baseline). One host thread. nodes/s."""
    import helpers
    n = int(soa["state"].shape[0])
    sec = helpers.oracle().ust_oracle_time_apply_state(
        C.c_int(variant), C.byref(policy), C.c_int64(n), soa["state"].ctypes.data_as(C.c_void_p),
        soa["flags"].ctypes.data_as(C.c_void_p), soa["pod_rev"].ctypes.data_as(C.c_void_p),
        soa["ds_idx"].ctypes.data_as(C.c_void_p), C.c_int32(int(soa["ds_rev"].shape[0])),
        soa["ds_rev"].ctypes.data_as(C.c_void_p), None, C.c_int(reps))
    return n / sec, sec


def run_reference(args, rank, world):
    """--impl reference: the reference's own (sequential, CPU) ApplyState, represented by the oracle's
    reference-shaped restatement — Go is not installed here or on the GPU box (DESIGN.md §3)."""
    if rank != 0:
        return
    from ust import synth
    cfg = synth.CONFIGS["C3" if world == 1 else "C5"]
    pol = synth.config_policy("C3")
    soa = synth.make_nodes(CPU_SAMPLE_NODES, cfg["seed"])
    cpu_reference_rate(pol, soa, max(1, min(args.warmup, 1)))
    t0 = time.time()
    rate, sec = cpu_reference_rate(pol, soa, max(1, args.steps))
    sample = f"first {CPU_SAMPLE_NODES} nodes of the workload, {max(1, args.steps)} ApplyState passes, median"
    line = {
        "impl": "reference", "metric": "node state-transitions/sec", "value": rate, "unit": "nodes/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8/i32", "data": "synthetic",
        "config": {"workload": workload_name(world), "sample_nodes": CPU_SAMPLE_NODES},
        "cpu_baseline": {"value": rate, "unit": "nodes/s", "cores": 1, "kind": "port", "sample": sample},
        "e2e": {"value": rate, "unit": "nodes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "wall_s": time.time() - t0,
    }
    print(json.dumps(line), flush=True)


def workload_name(world):
    if world == 1:
        return "C3: 10M-node synthetic cluster, MaxParallelUpgrades=100, MaxUnavailable=25%, 1xB200"
    return (f"C5-style: {world}x10M-node contiguous shards ({world * 10}M nodes), MaxParallelUpgrades=100, "
            f"MaxUnavailable=25%, one exchange of the constraint counters per ApplyState")


class DeviceBench:
    """Device-resident timing of ust_apply_state_device over rotating buffer sets (the same protocol for every
    configuration): warm-up, then `steps` back-to-back calls queued behind a GPU-side spin, bracketed by CUDA events
    on the launching stream."""

    def __init__(self, torch, dist, ustlib, abi, dev, world):
        self.torch, self.dist, self.ustlib, self.abi, self.dev, self.world = torch, dist, ustlib, abi, dev, world
        self.counters = torch.zeros(C.sizeof(abi.Counters) // 8, dtype=torch.int64, device=dev)
        self.fn = ustlib.load().ust_apply_state_device
        self._align = torch.zeros(1, device=dev)

    def on(self, h):
        """Time calls of handle `h`: they run on the handle's own stream (stream argument NULL), and so do the CUDA events
        and the launch-queue blocker - torch is made to treat that stream as current. (Events recorded on any other stream
        would not bracket the kernels: round-1 lesson.)"""
        ext = self.torch.cuda.ExternalStream(h.stream(), device=self.dev)
        self.torch.cuda.set_stream(ext)
        self._ext = ext

    def upload(self, soa, sets, outcome=False):
        torch = self.torch
        n = int(soa["state"].shape[0])
        bufs = []
        for _ in range(sets):
            d = {k: torch.from_numpy(v).to(self.dev) for k, v in soa.items()}
            d["next"] = torch.empty(n, dtype=torch.uint8, device=self.dev)
            d["actions"] = torch.empty(n, dtype=torch.int16, device=self.dev)
            d["outcome"] = torch.empty(n, dtype=torch.uint8, device=self.dev) if outcome else None
            bufs.append(d)
        return bufs

    def bind(self, h, pol, bufs, pods_struct=None):
        """pre-bound ctypes arguments per buffer set: the launch loop must not be the bottleneck (a step is ~30 us)"""
        n = int(bufs[0]["state"].shape[0])
        n_ds = int(bufs[0]["ds_rev"].shape[0])
        pol_p = C.c_void_p(C.addressof(pol))
        cnt_p = C.c_void_p(self.counters.data_ptr())
        st_p = None   # the handle's own stream
        bound = []
        for b in bufs:
            bound.append((h._h, pol_p, C.c_int64(n), C.c_void_p(b["state"].data_ptr()), C.c_void_p(b["flags"].data_ptr()),
                          C.c_void_p(b["pod_rev"].data_ptr()), C.c_void_p(b["ds_idx"].data_ptr()), C.c_int32(n_ds),
                          C.c_void_p(b["ds_rev"].data_ptr()), C.byref(pods_struct) if pods_struct is not None else None,
                          C.c_void_p(b["next"].data_ptr()), C.c_void_p(b["actions"].data_ptr()),
                          C.c_void_p(b["outcome"].data_ptr()) if b["outcome"] is not None else None, cnt_p, st_p))
        return bound

    def call(self, h, args):
        rc = self.fn(*args)
        if rc:
            raise self.ustlib.UstError(rc, h.last_error())

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def blocker(self):
        # ~1.5 ms of GPU spinning: the host queues the timed launches behind it, so the CUDA events bracket
        # back-to-back GPU execution rather than the Python launch rate
        self.torch.cuda._sleep(3_000_000)

    def time_steps(self, h, seq, steps, warmup):
        """seq(i) -> bound argument tuple of step i. Returns total milliseconds of `steps` steps (this rank)."""
        torch = self.torch
        torch.cuda.synchronize()   # uploads were queued on torch's stream, the calls go to the handle's
        self.on(h)
        for i in range(warmup):
            self.call(h, seq(i))
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.blocker()
        if self.world > 1:
            # line the ranks' streams up ON THE DEVICE before the clock starts: the host barrier above leaves the ranks
            # hundreds of microseconds apart (8 Python processes), and with coupled ranks every rank's timed region
            # would include the wait for the last one to begin (measured: +17 us/step over 50 steps at N=8)
            self.dist.all_reduce(self._align)
        e0.record()
        for i in range(steps):
            self.call(h, seq(warmup + i))
        e1.record()
        self.barrier()
        torch.cuda.set_stream(torch.cuda.default_stream(self.dev))   # the handle (and its stream) may be closed next
        self._ext = None
        return e0.elapsed_time(e1)

    def counters_struct(self):
        return self.abi.Counters.from_buffer_copy(self.counters.cpu().numpy().tobytes())

    def counters_dict(self):
        return self.counters_struct().as_dict()

    def redone_tiles(self):
        return int(self.counters_struct().reserved[0])


def same_as_oracle(helpers, pol, soa, buf, pods=None):
    """next_state / actions (/ actuator_outcome) of one timed buffer set against the SoA oracle, bit for bit."""
    ref = helpers.oracle_apply(pol, soa, pods, variant=1)
    ok = np.array_equal(buf["next"].cpu().numpy(), ref[1]) and np.array_equal(buf["actions"].cpu().numpy().view(np.uint16), ref[2])
    if buf.get("outcome") is not None and ref[3] is not None:
        ok = ok and np.array_equal(buf["outcome"].cpu().numpy(), ref[3])
    return bool(ok)


def dump_outputs(out_dir, buf, cnt, rank, world):
    """--dump-outputs: the outputs of one timed buffer set and the counters of the last call (module docstring)."""
    n = int(buf["next"].shape[0])
    m = min(n, DUMP_NODES // world)
    idx = np.arange(n) if m == n else np.sort(np.random.default_rng(0).choice(n, size=m, replace=False))
    arrays = {"node_index": idx.astype(np.float64),
              "next_state": buf["next"].cpu().numpy()[idx].astype(np.float32),
              "actions": buf["actions"].cpu().numpy().view(np.uint16)[idx].astype(np.float32),
              "counters": np.array(cnt["hist"] + [v for k, v in cnt.items() if k != "hist"], dtype=np.float64)}
    if buf.get("outcome") is not None:
        arrays["outcome"] = buf["outcome"].cpu().numpy()[idx].astype(np.float32)
    os.makedirs(out_dir, exist_ok=True)
    suffix = f"_rank{rank}" if world > 1 else ""
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + suffix + ".npy"), a)


def print_stamps(ustlib, h):
    g = min(int(os.environ["UST_STAMPS"]), 148)
    st = (C.c_uint64 * (4 * g + 16))()
    ustlib.load().ust_debug_stamps(h._h, st, g)
    a = np.array(st, dtype=np.int64)
    v = a[4 * g:]
    a = a[:4 * g].reshape(g, 4)
    a = a[a[:, 0] > a[:, 0].max() - 1_000_000]   # CTAs of the last launch only (a small snapshot uses fewer)
    t0 = a[:, 0].min()
    rel = (a - t0) / 1e3
    v = (v - t0) / 1e3
    print("stamps us: entry[min,max]=%.1f,%.1f first_tile[min,med,max]=%.1f,%.1f,%.1f stream_end[min,med,max]=%.1f,%.1f,%.1f "
          "exit[max]=%.1f | verify kernel CTA 0: woken %.1f vector %.1f decided %.1f redo done %.1f | decide: begin %.2f derived %.2f written %.2f synced %.2f | verify kernel entry: CTA 0 %.1f last CTA %.1f" % (
              rel[:, 0].min(), rel[:, 0].max(), rel[:, 1].min(), np.median(rel[:, 1]), rel[:, 1].max(),
              rel[:, 2].min(), np.median(rel[:, 2]), rel[:, 2].max(), rel[:, 3].max(), v[0], v[1], v[2], v[3], v[4], v[5], v[6], v[7], v[8], v[9]), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ust", choices=["ust", "reference"])
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--nodes", type=int, default=SHARD_NODES, help="nodes per GPU (default: the BASELINE workload)")
    ap.add_argument("--sets", type=int, default=16, help="rotating input/output buffer sets (L2 defeat)")
    ap.add_argument("--exchange", default="fused", choices=["fused", "nccl"], help="N>1: counter exchange mechanism")
    ap.add_argument("--maxpar", type=int, default=None, help="tuning: override MaxParallelUpgrades")
    ap.add_argument("--maxunav", default=None, help="tuning: override MaxUnavailable ('nil', int or 'NN%%')")
    ap.add_argument("--quick", action="store_true", help="tuning: device-resident timing of one configuration only")
    ap.add_argument("--e2e-format", default="packed", choices=["wide", "packed"],
                    help="host format of the e2e leg: wide = ust_apply_state (int32 pod_rev / ds_idx), packed = "
                         "ust_apply_state_packed (uint16 / int8: 8 instead of 13 bytes per node over PCIe)")
    ap.add_argument("--pods", action="store_true", help="tuning (with --quick): the C4 workload as the timed configuration")
    ap.add_argument("--no-by-config", action="store_true", help="skip the by_config legs (C2, C3_cut, C4, small)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step to DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs --impl ust: the reference run returns no outputs")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    import helpers
    from ust import abi, lib as ustlib, synth

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: libust.so has no CPU path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    warmup = max(args.warmup, 3)
    n = args.nodes
    cfg = synth.CONFIGS["C3" if world == 1 else "C5"]
    pol = synth.config_policy("C3")
    if args.maxpar is not None or args.maxunav is not None:
        mu = {"nil": None}.get(args.maxunav, args.maxunav) if args.maxunav is not None else "25%"
        if isinstance(mu, str) and mu.isdigit():
            mu = int(mu)
        pol = abi.make_policy(max_parallel_upgrades=args.maxpar if args.maxpar is not None else 100, max_unavailable=mu)
    if args.pods:
        if not args.quick:
            raise SystemExit("--pods selects C4 as the timed configuration of a --quick run; the full run reports C4 under by_config")
        cfg = synth.CONFIGS["C4"]
        pol = synth.config_policy("C4")
    soa = synth.make_nodes(n, cfg["seed"], start=rank * n)
    n_ds = int(soa["ds_rev"].shape[0])

    h = ustlib.Handle(local_rank)
    exchange = "none"
    if world > 1:
        uid = [ustlib.get_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        h.comm_init(rank, world, uid[0])
        exchange = "ncclAllReduce of 42 int64 lanes between the streaming and the verification kernel"
        if args.exchange == "fused":
            # every rank must end up in the same mode: agree on whether all of them mapped their peers
            ok = torch.ones(1, device=dev)
            try:
                h.comm_set_mode(1)
            except ustlib.UstError:
                ok.zero_()
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            if ok.item() > 0:
                exchange = "in-kernel NVLink mailbox exchange (CUDA IPC peer memory) inside the verification kernel"
            else:
                h.comm_set_mode(0)

    B = DeviceBench(torch, dist, ustlib, abi, dev, world)
    # Rotating buffer sets: a step never finds more than 126 MB / (SETS x 160 MB) of its inputs in L2.
    # (Two sets are NOT enough: the streaming loads are evict-first, so L2 keeps a fixed ~126 MB subset of
    # the 320 MB alive and half of every step would be L2 hits — measured in round 1, profiles/README.md.)
    SETS = max(2, args.sets)
    pods_dev = pods_struct = pods = None
    if args.pods:
        pods = synth.make_pods_blocked(n, cfg["seed"], start=rank * n)
        pods_dev = {k: torch.from_numpy(v).to(dev) for k, v in pods.items()}
        pods_struct = abi.Pods(pods_dev["pod_off"].data_ptr(), pods_dev["pod_flags"].data_ptr(), int(pods["pod_flags"].shape[0]))
        SETS = min(SETS, 4)
    bufs = B.upload(soa, SETS, outcome=args.pods)
    bound = B.bind(h, pol, bufs, pods_struct)

    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = h.launch_count()
    t_wall0 = time.time()
    total_ms = B.time_steps(h, lambda i: bound[i % SETS], args.steps, warmup)
    t_wall = time.time() - t_wall0
    launches = h.launch_count() - launches0
    clocks = sampler.stop()
    launches_per_step = launches / float(args.steps + warmup)

    tmax = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    total_ms = float(tmax.item())
    value = world * n * args.steps / (total_ms * 1e-3)
    cnt = B.counters_dict()
    assert cnt["error_code"] == 0
    verified = None
    last = (warmup + args.steps - 1) % SETS   # the buffer set of the last timed step
    if world == 1:
        verified = same_as_oracle(helpers, pol, soa, bufs[last], pods)
        assert verified, "timed outputs differ from the oracle"
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, bufs[last], cnt, rank, world)

    line = None
    if rank == 0:
        peak, peak_src = peaks()
        kern_ms = total_ms / args.steps
        achieved = BYTES_PER_NODE * n / (kern_ms * 1e-3) / 1e9
        traffic, traffic_src = ncu_traffic() if (world == 1 and n == SHARD_NODES and not args.pods) else (None, None)
        line = {
            "metric": "node state-transitions/sec", "value": value, "unit": "nodes/s", "n_gpus": world,
            "steps": args.steps, "warmup": warmup, "ms_per_step": kern_ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8/i32", "data": "synthetic",
            "config": {"workload": workload_name(world), "nodes_per_gpu": n, "bytes_per_node": BYTES_PER_NODE,
                       "l2": f"inputs larger than L2: {SETS} rotating buffer sets of {BYTES_PER_NODE * n / 1e6:.0f} MB each "
                             f"({SETS * BYTES_PER_NODE * n / 1e9:.2f} GB vs 126 MB L2, at most {100 * 126e6 / (SETS * BYTES_PER_NODE * n):.0f}% of a step can hit)",
                       "exchange": exchange},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                         "kernel": "ust_stream_kernel", "kernel_ms": kern_ms, "frac_of_8TBs": achieved / 8000.0,
                         "note": "kernel_ms = the step (streaming kernel + the verification kernel that follows it under "
                                 "programmatic dependent launch) averaged over the timed region"},
            "clocks": clocks, "gpu_launches": int(round(launches_per_step * args.steps)), "wall_s_timed_region": t_wall,
            "counters": {k: cnt[k] for k in ("total_managed", "in_progress", "unavailable", "max_unavailable", "upgrades_available")},
            "verified_vs_oracle": verified,
        }

    if args.quick:
        if rank == 0:
            fnr = ustlib.load().ust_debug_relaxed_calls
            fnr.restype = C.c_longlong
            fnr.argtypes = [C.c_void_p]
            print("counters:", {k: cnt[k] for k in ("candidates", "upgrades_available", "max_unavailable")},
                  "redone tiles:", B.redone_tiles(), "overlapped calls:", fnr(h._h), "of", h.launch_count() // 2, flush=True)
        if rank == 0 and os.environ.get("UST_STAMPS"):
            print_stamps(ustlib, h)
        if rank == 0:
            print(json.dumps({k: line[k] for k in ("value", "ms_per_step", "roofline", "clocks")}), flush=True)
        h.close()
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- N > 1: parity of the sharded run against the unsharded oracle, and what the exchange costs ----------------
    if world > 1:
        def gathered(policy):
            B.call(h, B.bind(h, policy, bufs[:1])[0])
            B.barrier()
            nx = [torch.empty(n, dtype=torch.uint8, device=dev) for _ in range(world)] if rank == 0 else None
            ac = [torch.empty(2 * n, dtype=torch.uint8, device=dev) for _ in range(world)] if rank == 0 else None   # NCCL has no int16
            dist.gather(bufs[0]["next"], nx, dst=0)
            dist.gather(bufs[0]["actions"].view(torch.uint8), ac, dst=0)
            if rank != 0:
                return None
            return (np.concatenate([t.cpu().numpy() for t in nx]), np.concatenate([t.cpu().numpy() for t in ac]).view(np.uint16),
                    B.counters_dict())
        cut_pol = abi.make_policy(max_parallel_upgrades=0, max_unavailable="45%")   # the budget runs out on a later rank
        got = [gathered(pol), gathered(cut_pol)]
        # the exchange: the same shard on a handle without a communicator
        h_local = ustlib.Handle(local_rank)
        bound_l = B.bind(h_local, pol, bufs)
        loc_ms = B.time_steps(h_local, lambda i: bound_l[i % SETS], args.steps, warmup)
        tl = torch.tensor([loc_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(tl, op=dist.ReduceOp.MAX)
        h_local.close()
        if rank == 0:
            whole = synth.make_nodes(world * n, cfg["seed"])
            mism = 0
            for policy, g in zip((pol, cut_pol), got):
                ref = helpers.oracle_apply(policy, whole, variant=1)
                mism += int(np.sum(g[0] != ref[1])) + int(np.sum(g[1] != ref[2])) + (0 if g[2] == ref[4] else 1)
            gr = (got[1][0] == 2) & ((whole["state"] & 15) == 1) & ((whole["state"] & abi.UST_HOT_UNSCHEDULABLE) == 0)
            line["parity_checked"] = True
            line["mismatches"] = mism
            line["parity"] = {"policies": ["timed policy (C3/C5)", "MaxParallelUpgrades=0, MaxUnavailable=45% (the budget runs out mid-cluster: ranks before the cut fully granted, the cut rank partly, ranks behind it not at all)"],
                              "nodes": world * n, "slots_granted_cut_policy": int(gr.sum()),
                              "ranks_with_grants": int(len(set((np.nonzero(gr)[0] // n).tolist()))),
                              "against": "SoA oracle on the unsharded cluster (next_state, actions, every counter)"}
            line["exchange_us"] = (total_ms - float(tl.item())) / args.steps * 1e3
            line["local_ms_per_step"] = float(tl.item()) / args.steps
            assert mism == 0, f"sharded outputs differ from the unsharded oracle in {mism} places"
            del whole
        B.barrier()

    # ---- e2e: host-pointer C ABI with pinned host buffers, H2D + kernels + D2H inside the timed region ----
    host = {k: ustlib.pinned_array(v.shape, v.dtype) for k, v in soa.items()}
    for k in soa:
        host[k][...] = soa[k]
    out = (ustlib.pinned_array(n, np.uint8), ustlib.pinned_array(n, np.uint16), None)
    packed = args.e2e_format == "packed"
    if packed:
        assert soa["pod_rev"].min() >= 0 and soa["pod_rev"].max() < 65536 and soa["ds_idx"].min() >= -128 and n_ds <= 127
        pk = (ustlib.pinned_array(n, np.uint16), ustlib.pinned_array(n, np.int8))
        pk[0][...] = soa["pod_rev"]
        pk[1][...] = soa["ds_idx"]

    def e2e_step():
        if packed:
            h.apply_state_packed(pol, host, want_outcome=False, out=out, check=True, packed=pk)
        else:
            h.apply_state(pol, host, want_outcome=False, out=out, check=True)

    for _ in range(2):
        e2e_step()
    B.barrier()
    t0 = time.time()
    for _ in range(args.e2e_steps):
        e2e_step()
    B.barrier()
    e2e_s = time.time() - t0
    te = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = world * n * args.e2e_steps / float(te.item())
    if world == 1:
        assert np.array_equal(out[0], bufs[(warmup + args.steps - 1) % SETS]["next"].cpu().numpy()), "e2e result differs from the device-resident result"

    # ---- the same through the delta entry point: the snapshot stays resident, 1 % of the nodes are re-encoded and
    # re-uploaded per step (a reconcile that watches resourceVersions), the whole snapshot is evaluated, all outputs
    # come back. Informative only - `e2e` above (full upload every step) is the headline.
    delta = None
    if world == 1:
        rng = np.random.default_rng(7)
        m = max(1, n // 100)
        steps_d = max(3, args.e2e_steps)

        def pinned(a):
            # what an encoder writes into: page-locked memory (ust_host_alloc), like the arrays of the full-upload leg
            p_ = ustlib.pinned_array(a.shape[0], a.dtype)
            p_[:] = a
            return p_

        deltas = []
        for _ in range(steps_d + 1):
            idx = rng.choice(n, size=m, replace=False).astype(np.int64)
            src = rng.integers(0, n, size=m)
            deltas.append((pinned(idx), {k: pinned(soa[k][src]) for k in ("state", "flags", "pod_rev", "ds_idx")}))
        h.apply_state_delta(pol, n, deltas[0][0], deltas[0][1], soa["ds_rev"], want_outcome=False, out=out)
        torch.cuda.synchronize()
        t0 = time.time()
        for idx, ch in deltas[1:]:
            rc = h.apply_state_delta(pol, n, idx, ch, soa["ds_rev"], want_outcome=False, out=out)[0]
            assert rc == 0, h.last_error()
        torch.cuda.synchronize()
        d_s = time.time() - t0
        delta = {"value": n * steps_d / d_s, "unit": "nodes/s", "ms_per_step": d_s / steps_d * 1e3, "changed_nodes_per_step": m,
                 "h2d_bytes_per_step": 21 * m + 4 * n_ds, "d2h_bytes_per_step": 3 * n + C.sizeof(abi.Counters), "steps": steps_d}
        # ... and with sparse outputs (ust_apply_state_delta_sparse): only the outputs that differ from the previous
        # call's come back. The caller's full arrays, patched with them, are checked against the dense result.
        cap = n // 8
        sp = (ustlib.pinned_array(cap + 1, np.int64), ustlib.pinned_array(cap + 1, np.uint8), ustlib.pinned_array(cap + 1, np.uint16))
        full_next, full_act = out[0].copy(), out[1].copy()
        cur = {k: soa[k].copy() for k in ("state", "flags", "pod_rev", "ds_idx")}
        for idx, ch in deltas:   # the dense leg applied these in order: replay them on the host copy
            for k in cur:
                cur[k][idx] = ch[k]
        more = []
        for _ in range(steps_d + 1):
            idx = rng.choice(n, size=m, replace=False).astype(np.int64)
            src = rng.integers(0, n, size=m)
            more.append((pinned(idx), {k: pinned(soa[k][src]) for k in ("state", "flags", "pod_rev", "ds_idx")}))
        n_outs = []
        t_sparse = 0.0
        for j, (idx, ch) in enumerate(more):
            torch.cuda.synchronize()
            t0 = time.time()
            rc, n_out, oi, on, oa, _ = h.apply_state_delta_sparse(pol, idx, ch, soa["ds_rev"], cap, out=sp)
            dt = time.time() - t0
            assert rc == 0 and n_out <= cap, (rc, n_out, h.last_error())
            full_next[oi[:n_out]] = on[:n_out]
            full_act[oi[:n_out]] = oa[:n_out]
            for k in cur:
                cur[k][idx] = ch[k]
            if j > 0:      # the first call warms the buffers up
                t_sparse += dt
                n_outs.append(n_out)
        ref = helpers.oracle_apply(pol, dict(cur, ds_rev=soa["ds_rev"]), variant=1)
        sparse_ok = bool(np.array_equal(full_next, ref[1]) and np.array_equal(full_act, ref[2]))
        assert sparse_ok, "sparse delta outputs, patched into the previous outputs, differ from the oracle"
        delta["sparse_outputs"] = {"ms_per_step": t_sparse / steps_d * 1e3, "value": n * steps_d / t_sparse, "unit": "nodes/s",
                                   "changed_outputs_per_step": float(np.mean(n_outs)), "h2d_bytes_per_step": 21 * m + 4 * n_ds,
                                   "d2h_bytes_per_step": int(11 * np.mean(n_outs)) + 8 + C.sizeof(abi.Counters),
                                   "entry_point": "ust_apply_state_delta_sparse", "verified_vs_oracle": sparse_ok}

    # ---- by_config (N = 1): the other configurations, same timing protocol, each verified on the timed buffers ------
    by_config = None
    if world == 1 and not args.no_by_config and n == SHARD_NODES:
        peak, _ = peaks()
        by_config = {"C3": {"ms": line["ms_per_step"], "frac": line["roofline"]["frac"], "bytes_per_node": BYTES_PER_NODE,
                            "verified_vs_oracle": verified, "redone_tiles_per_call": 0}}
        # the same steps in strict order (UST_OVERLAP=0: every call waits for the previous call's verification kernel, as
        # calls that share buffers always do): the time of ONE call, where the headline is the rate of a pipeline of them
        os.environ["UST_OVERLAP"] = "0"
        h_serial = ustlib.Handle(local_rank)
        del os.environ["UST_OVERLAP"]
        bound_s = B.bind(h_serial, pol, bufs)
        ms_serial = B.time_steps(h_serial, lambda i: bound_s[i % SETS], args.steps, warmup)
        by_config["C3"]["serial_ms"] = ms_serial / args.steps
        by_config["C3"]["serial_frac"] = BYTES_PER_NODE * n / (ms_serial / args.steps * 1e-3) / 1e9 / peak
        by_config["C3"]["note"] = ("ms: back-to-back calls on separate buffer sets overlap (a call's streaming kernel starts while the "
                                   "previous call is being decided); serial_ms: strict order, one call at a time")
        h_serial.close()
        del bound_s

        def frac_of(nbytes, ms):
            return nbytes / (ms * 1e-3) / 1e9 / peak

        # C3_cut: the budget cuts mid-array. Buffer sets perturbed: 0.1 % of the state bytes differ from set to set.
        rng = np.random.default_rng(11)
        variants = []
        for k in range(SETS):
            st = soa["state"].copy()
            idx = rng.choice(n, size=n // 1000, replace=False)
            st[idx] = soa["state"][rng.integers(0, n, size=idx.shape[0])]
            variants.append(st)
            bufs[k]["state"].copy_(torch.from_numpy(st))
        torch.cuda.synchronize()
        pol_a = abi.make_policy(max_parallel_upgrades=0, max_unavailable="30%")
        pol_b = abi.make_policy(max_parallel_upgrades=0, max_unavailable="31%")
        pol_c = abi.make_policy(max_parallel_upgrades=0, max_unavailable="32%")
        pols3 = (pol_a, pol_b, pol_c)
        bound3 = tuple(B.bind(h, p_, bufs) for p_ in pols3)
        bound_a = bound3[0]
        steps_c = max(10, args.steps // 2)
        # first call: three policies in turn, so no call finds a hint made under its own signature (a call looks at
        # the hint of the previous call or, when it overlaps that call, of the one before)
        ms_first = B.time_steps(h, lambda i: bound3[i % 3][i % SETS], steps_c, warmup)
        i_last = warmup + steps_c - 1
        redone_first = B.redone_tiles()
        v_first = same_as_oracle(helpers, pols3[i_last % 3], dict(soa, state=variants[i_last % SETS]), bufs[i_last % SETS])
        ms_steady = B.time_steps(h, lambda i: bound_a[i % SETS], args.steps, warmup)
        i_last = warmup + args.steps - 1
        redone_steady = B.redone_tiles()
        v_steady = same_as_oracle(helpers, pol_a, dict(soa, state=variants[i_last % SETS]), bufs[i_last % SETS])
        by_config["C3_cut"] = {
            "policy": "MaxParallelUpgrades=0, MaxUnavailable=30% on C3's data: the slot budget cuts mid-array",
            "first_call_us": ms_first / steps_c * 1e3, "steady_us": ms_steady / args.steps * 1e3,
            "frac_first": frac_of(BYTES_PER_NODE * n, ms_first / steps_c), "frac_steady": frac_of(BYTES_PER_NODE * n, ms_steady / args.steps),
            "redone_tiles_first_call": redone_first, "redone_tiles_steady": redone_steady,
            "perturbation": "every buffer set differs from the base snapshot in 0.1 % of its state bytes (stale-but-close hint)",
            "verified_vs_oracle": bool(v_first and v_steady)}
        del bound_a, bound3, variants

        # C2 and the small snapshots: what a reconcile of a real cluster sees
        small = {}
        for name, nn, sets in (("C2", 1_000_000, 32), ("100k", 100_000, 64), ("10k", 10_000, 64)):
            c = synth.CONFIGS["C2"]
            s2 = synth.make_nodes(nn, c["seed"])
            p2 = synth.config_policy("C2")
            b2 = B.upload(s2, sets)
            bd2 = B.bind(h, p2, b2)
            steps2 = max(args.steps, 100)
            ms2 = B.time_steps(h, lambda i: bd2[i % sets], steps2, warmup)
            v2 = same_as_oracle(helpers, p2, s2, b2[(warmup + steps2 - 1) % sets])
            entry = {"nodes": nn, "us_per_call": ms2 / steps2 * 1e3, "ms": ms2 / steps2, "frac": frac_of(BYTES_PER_NODE * nn, ms2 / steps2),
                     "bytes_per_node": BYTES_PER_NODE, "buffer_sets": sets, "verified_vs_oracle": v2}
            if name == "C2":
                by_config["C2"] = entry
            else:
                small[name] = entry
            del b2, bd2
        by_config["small"] = small

        # C4: pod lists. Bytes the configuration moves: the five node streams + outputs, the hot byte and the summary byte
        # of the pod pass, and the CSR offsets + lists of the nodes whose actuator looks at its pods.
        del bufs, bound
        torch.cuda.empty_cache()
        c4 = synth.CONFIGS["C4"]
        s4 = synth.make_nodes(n, c4["seed"])
        pods4 = synth.make_pods_blocked(n, c4["seed"])
        p4 = synth.config_policy("C4")
        pd = {k: torch.from_numpy(v).to(dev) for k, v in pods4.items()}
        ps4 = abi.Pods(pd["pod_off"].data_ptr(), pd["pod_flags"].data_ptr(), int(pods4["pod_flags"].shape[0]))
        sets4 = 4
        b4 = B.upload(s4, sets4, outcome=True)
        bd4 = B.bind(h, p4, b4, ps4)
        steps4 = max(10, args.steps // 2)
        launches0 = h.launch_count()
        ms4 = B.time_steps(h, lambda i: bd4[i % sets4], steps4, warmup)
        l4 = (h.launch_count() - launches0) / float(steps4 + warmup)
        v4 = same_as_oracle(helpers, p4, s4, b4[(warmup + steps4 - 1) % sets4], pods4)
        code = s4["state"] & 15
        need = (code >= 3) & (code <= 5)
        lens = np.diff(pods4["pod_off"].astype(np.int64))
        moved = (14 + 4 + 2) * n + int(np.sum(2 * lens[need] + 8))  # streaming pass 14 read + 4 written, pod pass 1 + 1
        by_config["C4"] = {"nodes": n, "pods": int(pods4["pod_flags"].shape[0]), "ms": ms4 / steps4, "us_per_call": ms4 / steps4 * 1e3,
                           "bytes_moved_per_call": moved, "bytes_per_node_moved": moved / n, "frac": frac_of(moved, ms4 / steps4),
                           "frac_of_81B_budget": frac_of(81 * n, ms4 / steps4), "launches_per_call": l4,
                           "nodes_whose_lists_are_read": int(need.sum()), "verified_vs_oracle": v4}
        del b4, bd4, pd

    if rank == 0:
        if delta is not None:
            line["e2e_delta"] = delta
        if by_config is not None:
            line["by_config"] = by_config
        line["e2e"] = {"value": e2e_value, "unit": "nodes/s", "h2d_bytes_per_step": (8 if packed else 13) * n + 4 * n_ds,
                       "entry_point": "ust_apply_state_packed" if packed else "ust_apply_state",
                       "d2h_bytes_per_step": 3 * n + C.sizeof(abi.Counters), "steps": args.e2e_steps,
                       "ms_per_step": float(te.item()) / args.e2e_steps * 1e3}
        # ---- CPU baseline beside it: bounded sample, 1 thread (the reference loop is sequential) ----
        m = min(CPU_SAMPLE_NODES, n)
        sample = {k: (v[:m].copy() if k != "ds_rev" else v) for k, v in soa.items()}
        rate, sec = cpu_reference_rate(pol, sample, 3)
        rate_soa, _ = cpu_reference_rate(pol, sample, 3, variant=1)
        line["cpu_baseline"] = {"value": rate, "unit": "nodes/s", "cores": 1, "kind": "port", "soa_scalar_1core": rate_soa,
                                "sample": f"first {m} nodes of the workload, ApplyState only, median of 3 passes "
                                          f"({sec:.2f} s each), reference-shaped oracle (Go unavailable)"}
        print(json.dumps(line), flush=True)
    h.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
