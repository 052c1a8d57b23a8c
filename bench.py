#!/usr/bin/env python
"""bench.py - throughput of the DFQ calibration hot path on B200.

One "step" = one pass of the hot path (BN fold -> cross-layer equalization to convergence -> bias correction) over
one synthetic stack of independent Conv[512,512,3,3]+BN+ReLU -> Conv[512,512,3,3]+BN blocks (BASELINE.json
configs[4], the configuration the metric's HBM-roofline half is quoted on; it is the largest single-GPU
configuration: 4096 layer pairs = 38.65 GB of fp32 weights).  Output: ONE JSON line (see README / DESIGN.md).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--layers L] [--impl b200|reference] [--dump-outputs DIR]

  value      whole-job Conv/BN layer-pairs per second with the stack resident in HBM (device-timed, CUDA events)
  e2e        the same metric through the public API with HOST buffers: pinned host -> device, calibrate, device -> host
  roofline   the dominant kernel (k_cle_engine): algorithmic bytes (8 B per weight per sweep) / its event-timed
             duration, against MEASURED_PEAKS.json
  cpu_baseline  the oracle (oracle/) timed on the host cores on a bounded sample of the same workload

`--impl reference` times the reference's CPU implementation of the path (its algorithm restated in oracle/, since
the reference is Python and is not present on the GPU box) on the same workload shape.
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

METRIC = "conv_bn_layer_pairs_equalized_and_corrected_per_second"
UNIT = "layers/s"
C, K = 512, 3
N_PER_LAYER = C * C * K * K


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=10)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--layers", type=int, default=4096, help="Conv/BN pairs in the synthetic stack per GPU")
    p.add_argument("--e2e-layers", type=int, default=512, help="pairs moved host->device->host per e2e step")
    p.add_argument("--e2e-chunk", type=int, default=16, help="pairs per pipelined chunk of the e2e arm (measured: 32 pairs / 4 slots 4.93 k pairs/s, 16 / 6 5.05 k)")
    p.add_argument("--e2e-slots", type=int, default=6, help="arena slots of the e2e pipeline")
    p.add_argument("--cpu-layers", type=int, default=0, help="pairs in the CPU-baseline sample (0 = auto)")
    p.add_argument("--impl", default="b200", choices=["b200", "reference"])
    p.add_argument("--quantize", action="store_true", help="also fake-quantize weights/biases (8 bit) inside the step")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--no-mbv2", action="store_true")
    p.add_argument("--no-parity-check", action="store_true")
    p.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                   help="which curve is the line's headline `value` (the other one is reported next to it): weak = --layers "
                        "pairs PER GPU, strong = --layers pairs IN TOTAL split over the GPUs (SURVEY 8(d) config 5)")
    p.add_argument("--no-strong", action="store_true", help="skip the strong-scaling measurement")
    p.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed as DIR/<name>.npy (rank 0)")
    return p.parse_args()


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled while the timed region runs (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self._halt = index, [], threading.Event()

    def run(self):
        while not self._halt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self._halt.wait(0.2)

    def stop(self):
        self._halt.set()
        self.join(timeout=6)
        sm = sorted(float(r[1]) for r in self.rows if len(r) > 2 and r[1].replace(".", "").isdigit())
        reasons = []
        for name, col in (("hw_slowdown", 4), ("hw_thermal_slowdown", 5), ("sw_thermal_slowdown", 6), ("sw_power_cap", 7)):
            if any(len(r) > col and r[col].lower().startswith("active") for r in self.rows):
                reasons.append(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None,
                "sm_max_mhz": float(self.rows[0][2]) if self.rows and self.rows[0][2].replace(".", "").isdigit() else None,
                "samples": len(self.rows), "reasons": reasons}


# dram__bytes_read.sum + dram__bytes_write.sum of the equalization kernel (k_cle_stack) from the committed `ncu --set full`
# capture (profiles/r2_cle_stack_v2.md: 19.346 GB read + 19.292 GB written at 1024 pairs, 2 sweeps; algorithmic 38.655 GB).  The
# kernel's traffic is linear in the number of pairs (every block is identical), so the figure is scaled to the benched size;
# None for other sweep counts.  (k_cle_engine, round 1: 38.809 GB, profiles/r1_ncu_full_1024layers.md.)
NCU_TRAFFIC_1024_PAIRS_2_SWEEPS = 38.638e9
NCU_TRAFFIC_SOURCE = "ncu --set full capture of k_cle_stack at 1024 pairs (profiles/r2_cle_stack_v2.md), scaled linearly to the benched pairs"


def ncu_traffic(layers, sweeps):
    return NCU_TRAFFIC_1024_PAIRS_2_SWEEPS * layers / 1024.0 if sweeps == 2 else None


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


# ----------------------------------------------------------------------------------------------------------
# CPU arm: the oracle on the same workload shape
# ----------------------------------------------------------------------------------------------------------
def cpu_pipeline(n_pairs, seed=1234, eager=False):
    """Time one calibration step (fold -> equalize to convergence -> correct) of `n_pairs` layer pairs on the host.
    Returns (seconds, sweeps)."""
    import numpy as np
    import torch
    from oracle import dfq_oracle as O
    if eager:
        from oracle import eager_port as E
    n_blocks = max(1, n_pairs // 2)
    g = torch.Generator().manual_seed(seed)
    std = (2.0 / (K * K * C)) ** 0.5
    blocks = []
    for _ in range(n_blocks):
        ws = []
        for _ in range(2):
            w = torch.randn(C, C, K, K, generator=g) * std
            w = w * (10 ** torch.empty(C).uniform_(-1, 1, generator=g)).view(-1, 1, 1, 1)
            bn = [torch.empty(C).uniform_(0.5, 1.5, generator=g), torch.randn(C, generator=g) * 0.2,
                  torch.randn(C, generator=g) * 0.1, torch.empty(C).uniform_(0.5, 1.5, generator=g)]
            ws.append((w, bn))
        blocks.append(ws)
    t0 = time.perf_counter()
    sweeps = 0
    if eager:
        sweeps = E.calibrate_blocks(blocks)
    else:
        for ws in blocks:                   # every block is its own model: one reference-style call each (own exit rule)
            layers, bns = [], []
            for w, bn in ws:
                w2, b2, fw, fb = O.bn_fold(w.numpy(), None, *[x.numpy() for x in bn], 1e-5)
                layers.append(O.OLayer(w2, b2)); bns.append((fw, fb))
            rel = O.ORelation(0, 1, 0)
            n, _ = O.cross_layer_equalization(layers, bns, [rel])
            sweeps = max(sweeps, n)
            e = O.relu_expectation(*bns[0])
            d = O.bias_delta(layers[1].w, e)
            layers[1].b = layers[1].b + (-d)
            bns[1] = (bns[1][0], bns[1][1] + (-d))
    return time.perf_counter() - t0, sweeps


def bind_to_gpu_numa_node(local_rank):
    """Pin this rank (and therefore its page-locked buffers: first touch) to the NUMA node its GPU hangs off.  Round 1's
    e2e arm scaled 0.67 / 0.49 at 4 / 8 GPUs because every rank allocated its pinned staging memory wherever the launcher
    happened to start it (GPUs 4-7 sit on node 1).  Returns dict(node, cpus) or None when the topology is not exposed."""
    try:
        import torch
        p = torch.cuda.get_device_properties(local_rank)
        if hasattr(p, "pci_bus_id") and hasattr(p, "pci_device_id"):
            dev = "%04x:%02x:%02x.0" % (getattr(p, "pci_domain_id", 0), p.pci_bus_id, p.pci_device_id)
        else:
            out = subprocess.run(["nvidia-smi", "-i", str(local_rank), "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                                 capture_output=True, text=True, timeout=10).stdout.strip().lower()
            dev = out[-12:] if len(out) >= 12 else out
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % dev).read())
        if node < 0:
            return None
        cpus = []
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.extend(range(int(a), int(b or a) + 1))
        cpus = sorted(set(cpus) & set(os.sched_getaffinity(0)))
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        policy = None
        try:      # memory too: set_mempolicy(MPOL_PREFERRED, node) - page-locked allocations made by driver threads follow it
            import ctypes
            import platform
            if platform.machine() == "x86_64" and node < 64:
                mask = ctypes.c_ulong(1 << node)
                if ctypes.CDLL(None, use_errno=True).syscall(238, 1, ctypes.byref(mask), 65) == 0:
                    policy = "preferred"
        except Exception:
            pass
        return {"node": node, "cpus": len(cpus), "mempolicy": policy}
    except Exception:
        return None


DUMP_CAP = 10 * 2 ** 20 // 4       # floats per dumped array: the six arrays stay under 64 MB together


def dump_outputs(out_dir, stack, res):
    """Write what one calibration step of `stack` computed, as a caller of the path receives it, to out_dir/<name>.npy:
    the calibrated weights, corrected biases, folded BN vectors (fake_weight / fake_bias) and scale vectors S of every
    layer, and the sweeps each block took.  An array longer than DUMP_CAP floats is replaced by the same seeded sample of
    its elements (sorted indices into the concatenation over the layers) on every run, so two builds compare element for
    element.  The weights of the default stack (38.65 GB) are always sampled."""
    import numpy as np
    import torch
    sess, C, N = stack.sess, stack.C, stack.N

    def sample_index(n):
        if n <= DUMP_CAP:
            return torch.arange(n)
        g = torch.Generator().manual_seed(0)
        return torch.randint(n, (DUMP_CAP,), generator=g).sort().values

    def gather(offs, n_each):
        """Elements of the arena windows [off, off + n_each) for off in offs, concatenated (and sampled)."""
        idx = sample_index(len(offs) * n_each)
        flat = torch.tensor(offs, dtype=torch.int64)[idx // n_each] + idx % n_each
        return sess.arena.index_select(0, flat.to(sess.device))

    layers = [sess.layer(li) for li in stack.layers]
    arrays = {"weights": gather([l["w_off"] for l in layers], N),
              "bias": gather([l["bias_off"] for l in layers], C),
              "bn_fake_weight": gather([v["fake_w"] for v in stack.vec], C),
              "bn_fake_bias": gather([v["fake_b"] for v in stack.vec], C),
              "scales": gather(list(stack.cle_plan["s_offs"]), C),
              "sweeps": torch.from_numpy(np.asarray(res.group_sweeps, dtype=np.float64))}
    arrays = {k: v.cpu().numpy() for k, v in arrays.items()}
    assert sum(a.nbytes for a in arrays.values()) <= 64 * 2 ** 20
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def one_socket_cores():
    """One logical CPU per physical core of the socket this process starts on (sysfs topology), or None."""
    try:
        allowed = sorted(os.sched_getaffinity(0))
        seen, pick, pkg0 = set(), [], None
        for c in allowed:
            base = "/sys/devices/system/cpu/cpu%d/topology/" % c
            pkg = int(open(base + "physical_package_id").read())
            core = int(open(base + "core_id").read())
            if pkg0 is None:
                pkg0 = pkg
            if pkg == pkg0 and (pkg, core) not in seen:
                seen.add((pkg, core)); pick.append(c)
        return pick or None
    except Exception:
        return None


def run_reference(args, rank, world):
    """The reference's CPU execution of the path (oracle/eager_port.py: dfq.py's per-channel eager loop, deepcopy per sweep,
    seven-pass fake quantization) on the box's host cores.  SURVEY 8(d): a 64-pair subsample of the stack; threads = the
    physical cores of ONE socket with the process pinned to them (the ops are tiny - 4608-element rows - so more threads
    only add OpenMP spin noise: round 1 saw 1.35 ... 15 pairs/s on the same box type with all 128 logical CPUs); value =
    median step.  The reference itself is Python and absent on the GPU box: kind "port"."""
    import torch
    if rank != 0:
        return
    cores = one_socket_cores()
    if cores:
        try:
            os.sched_setaffinity(0, cores)
        except Exception:
            pass
    n_thr = len(cores) if cores else max(1, (os.cpu_count() or 2) // 2)
    torch.set_num_threads(n_thr)
    pairs = args.cpu_layers or 64
    for _ in range(min(args.warmup, 1)):
        cpu_pipeline(4, eager=True)
    times = []
    budget = time.perf_counter() + 150.0           # keep the whole arm within a few minutes on a slow box
    for _ in range(max(3, min(args.steps, 5))):
        dt, sweeps = cpu_pipeline(pairs, eager=True)
        times.append(dt)
        if time.perf_counter() > budget and len(times) >= 3:
            break
    times.sort()
    dt = times[len(times) // 2]
    val = pairs / dt
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": len(times),
            "warmup": min(args.warmup, 1), "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "synthetic stack Conv[512,512,3,3]+BN pairs (BASELINE configs[4])", "layers_per_step": pairs,
                       "sweeps": sweeps, "step_seconds": [round(t, 3) for t in times],
                       "spread": round((times[-1] - times[0]) / dt, 3)},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": n_thr, "kind": "port",
                             "sample": "%d layer pairs per step (SURVEY 8(d) subsample of the 4096-pair stack), median of %d steps, "
                                       "PyTorch-eager per-channel port of dfq.py (oracle/eager_port.py), %d threads pinned to the "
                                       "physical cores of one socket" % (pairs, len(times), n_thr)},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------------------
# BASELINE configs[1]: MobileNetV2 (random init) equalize + correct on one GPU - latency, not bandwidth
# ----------------------------------------------------------------------------------------------------------
def mobilenetv2_latency(dev, reps=5):
    """52 Conv/BN pairs + classifier of the reference's MobileNetV2 graph (tests/golden/topology_mobilenetv2.json), seeded
    random weights on the HOST.  Returns dict(plan_ms, e2e_ms, device_ms, sweeps): e2e = pinned H2D + fold + equalize to
    convergence + bias correction + D2H + in-place write-back through dfq_b200.calibrate.GraphCalibration; device = the
    same three launches with the model resident (CUDA events)."""
    import torch
    import torch.nn as nn
    from dfq_b200 import workload
    from dfq_b200.calibrate import GraphCalibration
    path = os.path.join(ROOT, "tests", "golden", "topology_mobilenetv2.json")
    if not os.path.exists(path):
        return None
    topo = workload.load_topology(path)
    graph, bottoms, modules = workload.build_graph(topo, seed=0)
    targ = [nn.Conv2d, nn.Linear]
    backup = [{k: v.clone() for k, v in m.state_dict().items()} for m in modules]
    eps0 = [getattr(m, "eps", None) for m in modules]

    def restore():
        """Undo a calibration in place (parameters stay the same objects the plan is bound to).  Single-threaded: the tensor
        library's OpenMP workers keep spinning on every allowed CPU for a while after a parallel copy, and this harness step
        ends right where the timed region begins (the rank is bound to one NUMA node's CPUs)."""
        nt = torch.get_num_threads()
        torch.set_num_threads(1)
        try:
            _restore()
        finally:
            torch.set_num_threads(nt)

    def _restore():
        with torch.no_grad():
            for m, sd, e in zip(modules, backup, eps0):
                if isinstance(m, (nn.Conv2d, nn.Linear)):
                    m.weight.copy_(sd["weight"])
                    if m.bias is not None:
                        m.bias.copy_(sd["bias"]) if "bias" in sd else m.bias.zero_()
                elif isinstance(m, nn.BatchNorm2d):
                    for k in ("weight", "bias", "running_mean", "running_var"):
                        getattr(m, k).copy_(sd[k])
                    m.eps = e
    pairs = sum(1 for m in modules if isinstance(m, nn.BatchNorm2d))
    t0 = time.perf_counter()
    cal = GraphCalibration(graph, bottoms, targ, device=dev)
    plan_ms = (time.perf_counter() - t0) * 1e3
    e2e, devms, sweeps, parts = [], [], 0, []
    for i in range(reps + 2):
        restore()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        cal.upload()
        t1 = time.perf_counter()
        cal.run_device(equalize=True, correction=True)
        t2 = time.perf_counter()
        cal.download()
        torch.cuda.synchronize()
        t3 = time.perf_counter()
        res = cal.last_cle
        if i >= 2:
            e2e.append((t3 - t0) * 1e3)
            parts.append(((t1 - t0) * 1e3, (t2 - t1) * 1e3, (t3 - t2) * 1e3))
        sweeps = res.n_sweeps
    restore()
    cal.upload()
    pristine = cal.sess.arena.clone()
    for i in range(reps + 2):
        cal.sess.arena.copy_(pristine)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        cal.run_device(equalize=True, correction=True)
        b.record()
        torch.cuda.synchronize()
        if i >= 2:
            devms.append(a.elapsed_time(b))
    return {"pairs": pairs, "relations": len(cal.relations), "sweeps": sweeps, "plan_ms": plan_ms,
            "e2e_ms": sorted(e2e)[len(e2e) // 2], "device_ms": sorted(devms)[len(devms) // 2],
            "e2e_parts_ms": {"stage_and_h2d_enqueue": sorted(p[0] for p in parts)[len(parts) // 2],
                             "launches_until_results_known": sorted(p[1] for p in parts)[len(parts) // 2],
                             "d2h_and_write_back": sorted(p[2] for p in parts)[len(parts) // 2]},
            "pairs_per_s_e2e": pairs / (sorted(e2e)[len(e2e) // 2] * 1e-3),
            "what": "BN fold + equalization to convergence + bias correction of MobileNetV2 (random init, seed 0); e2e = "
                    "host parameters -> pinned H2D -> 3 launches -> D2H -> in place"}


# ----------------------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------------------
def run_b200(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from dfq_b200.engine import Session
    from dfq_b200.workload import DeviceStack

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa = bind_to_gpu_numa_node(local_rank)          # before any page-locked allocation
    free, total = torch.cuda.mem_get_info()
    layers = args.layers - (args.layers % 2)
    bytes_per_layer = 4 * (N_PER_LAYER + 8 * C)
    while layers > 2 and 2.1 * layers * bytes_per_layer > 0.92 * free:
        layers //= 2
    n_blocks = layers // 2

    sess = Session(dev)
    stack = DeviceStack(sess, n_blocks, C, K, seed=1234 + rank, quantize=args.quantize)
    stack.generate()
    pristine = stack.state().clone()
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    class Exchange:
        """The path's one exchange (SURVEY 8(e) "Collective"): ONE all-gather of a flat buffer holding, for this rank's
        shard, the accumulated scale vectors S of every relation, the corrected biases and the BN vectors (fake_weight /
        fake_bias) of every layer - after it every rank holds the [C]-sized results of the whole job; weights stay put."""

        def __init__(self, st):
            self.views = [st.scale_state(), st.channel_state()]
            self.n = sum(v.numel() for v in self.views)
            self.send = torch.empty(self.n, dtype=torch.float32, device=dev)
            self.recv = torch.empty(world * self.n, dtype=torch.float32, device=dev)

        def run(self):
            o = 0
            for v in self.views:
                self.send[o:o + v.numel()].copy_(v); o += v.numel()
            dist.all_gather_into_tensor(self.recv, self.send)

    def make_step(st, se, saved, xch):
        def step(timers=None):
            st.state().copy_(saved)                          # untimed: restores (and evicts L2 when the stack is >> 126 MB)
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
            ev[0].record()
            se.run_bn_fold(st.fold_plan)
            ev[1].record()
            res = se.run_cle_plan(st.cle_plan, cols_ready=st.fold_plan["scanned"])
            ev[2].record()
            se.run_bias_correct_plan(st.bc_plan, 8, col_hints=se.cle_col_hints(st.cle_plan, res))
            if st.quant_plan is not None:
                se.run_quantize(st.quant_plan)
            ev[3].record()
            if xch is not None:
                xch.run()
            ev[4].record()
            torch.cuda.synchronize()
            if timers is not None:
                timers.append([ev[i].elapsed_time(ev[i + 1]) for i in range(4)])
            return res
        return step

    def measure(step_fn):
        for _ in range(max(args.warmup, 3)):
            r = step_fn()
        barrier()
        tm = []
        for _ in range(args.steps):
            r = step_fn(tm)
        barrier()
        return r, tm

    exchange = Exchange(stack) if world > 1 else None
    step = make_step(stack, sess, pristine, exchange)
    for _ in range(max(args.warmup, 3)):
        res = step()
    barrier()
    sampler = ClockSampler(local_rank); sampler.start()
    timers = []
    for _ in range(args.steps):
        res = step(timers)
    barrier()
    clocks = sampler.stop()
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, stack, res)

    # ---- parity of what was just timed: first and last block of this rank's stack vs the oracle (checker only) ---------
    parity = None
    if rank == 0 and not args.no_parity_check:
        from oracle import stack_check
        after = stack.state()
        checks = [stack_check.compare_block(stack.block_arrays(pristine, b), stack.block_arrays(after, b))
                  for b in sorted({0, n_blocks - 1})]
        parity = {"blocks_checked": sorted({0, n_blocks - 1}), "of_blocks": n_blocks,
                  "weights_bit_exact": all(c["weights_bit_exact"] and c["vectors_bit_exact"] for c in checks),
                  "bias_max_normwise_error": max(c["bias_normwise"] for c in checks),
                  "sweeps_equal_oracle": all(c["sweeps"] == int(res.group_sweeps[b]) for c, b in zip(checks, sorted({0, n_blocks - 1}))),
                  "oracle": "oracle/stack_check.py on the pristine bits of the timed stack, after the last timed step"}
        # ... and a size-independent property over EVERY block of the stack (torch reductions on the device): after the
        # equalization the range of row c of the first conv equals the range of input column c of the second conv
        # (s = sqrt(r2/r1) makes both sqrt(r1*r2), dfq.py:58), and nothing is non-finite
        w = after[:2 * n_blocks * N_PER_LAYER].view(n_blocks, 2, C, C, K * K)
        dev_max = 0.0
        for lo in range(0, n_blocks, 256):
            a, b2 = w[lo:lo + 256, 0], w[lo:lo + 256, 1]
            r1 = a.amax(dim=(2, 3)) - a.amin(dim=(2, 3))
            r2 = b2.amax(dim=(1, 3)) - b2.amin(dim=(1, 3))
            dev_max = max(dev_max, float(((r1 - r2).abs() / r1).max()))
        parity["all_blocks_range_mismatch"] = dev_max
        parity["all_finite"] = bool(torch.isfinite(after).all())
        parity["ok"] = bool(parity["weights_bit_exact"] and parity["bias_max_normwise_error"] < 1e-5 and parity["sweeps_equal_oracle"]
                            and dev_max < 1e-5 and parity["all_finite"])

    t = torch.tensor([sum(sum(r) for r in timers) / len(timers),
                      sum(r[1] for r in timers) / len(timers)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step, ms_cle = float(t[0]), float(t[1])
    value = world * layers / (ms_step * 1e-3)
    phases = [sum(r[i] for r in timers) / len(timers) for i in range(4)]

    # ---- strong scaling: the SAME total stack (--layers pairs) split over the ranks -------------------------------------
    strong = None
    if world > 1 and not args.no_strong:
        s_blocks = max(1, (args.layers // 2) // world)
        s_sess = Session(dev)
        s_stack = DeviceStack(s_sess, s_blocks, C, K, seed=4321 + rank, quantize=args.quantize)
        s_stack.generate()
        s_saved = s_stack.state().clone()
        s_x = Exchange(s_stack)
        s_res, s_tm = measure(make_step(s_stack, s_sess, s_saved, s_x))
        ts = torch.tensor([sum(sum(r) for r in s_tm) / len(s_tm)] + [sum(r[i] for r in s_tm) / len(s_tm) for i in range(4)],
                          dtype=torch.float64, device=dev)
        dist.all_reduce(ts, op=dist.ReduceOp.MAX)
        strong = {"value": world * 2 * s_blocks / (float(ts[0]) * 1e-3), "unit": UNIT, "ms_per_step": float(ts[0]),
                  "layers_total": world * 2 * s_blocks, "layers_per_gpu": 2 * s_blocks, "sweeps": s_res.n_sweeps,
                  "phases_ms_max_over_ranks": {"bn_fold": float(ts[1]), "equalize": float(ts[2]), "bias_correct": float(ts[3]),
                                               "exchange": float(ts[4])},
                  "exchange_bytes_per_rank": 4 * s_x.n,
                  "l2": "%.1f GB of weights per GPU >> 126 MB L2; restored from a pristine copy (untimed) before every step"
                        % (4e-9 * N_PER_LAYER * 2 * s_blocks),
                  "what": "fixed total of %d pairs split over %d GPUs; speed-up over the 1-GPU weak line at the same total is "
                          "strong-scaling efficiency x N" % (world * 2 * s_blocks, world)}
        del s_stack, s_sess, s_saved, s_x
        torch.cuda.empty_cache()

    # ---- roofline of the dominant kernel ----------------------------------------------------------------------
    peak, peak_src = measured_peaks()
    cle_bytes = 8.0 * N_PER_LAYER * layers * res.n_sweeps          # SURVEY 8(d): 8 B per weight per sweep
    achieved = cle_bytes / (ms_cle * 1e-3) / 1e9
    roofline = {"bound": "hbm", "kernel": "k_cle_stack (equalization of the two-layer chains; k_cle_engine when DFQ_CLE_STACK=0)", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": ncu_traffic(layers, res.n_sweeps), "traffic_source": NCU_TRAFFIC_SOURCE, "peak_source": peak_src + " (MEASURED_PEAKS.json hbm_gbs, burst copy)",
                "algorithmic_bytes_per_launch": cle_bytes, "ms_per_launch": ms_cle,
                "whole_step": {"algorithmic_bytes": (26.0 + (12.0 if args.quantize else 0)) * N_PER_LAYER * layers,
                               "GB/s": (26.0 + (12.0 if args.quantize else 0)) * N_PER_LAYER * layers / (ms_step * 1e-3) / 1e9}}

    # ---- end to end with host buffers -----------------------------------------------------------------------------
    e2e = None
    if not args.no_e2e:
        from dfq_b200.workload import HostStackCalibrator
        chunk_blocks = max(1, args.e2e_chunk // 2)                # 16 layer pairs = 151 MB per chunk
        # 2 x 4.8 GB of page-locked memory per rank at 512 pairs, allocated on the rank's own NUMA node (bind_to_gpu_numa_node)
        e2e_pairs = args.e2e_layers
        del pristine
        torch.cuda.empty_cache()
        hc = HostStackCalibrator(dev, chunk_blocks, C, K, quantize=args.quantize, n_slots=args.e2e_slots)
        # the box's page-locked budget is shared by all ranks: every rank tries the full sample and all ranks settle on the
        # size the most constrained one got (halving on failure), so the ranks keep doing equal work
        while True:
            n_chunks = max(2, min(e2e_pairs, layers) // (2 * chunk_blocks))
            n_state = hc.chunk_floats * n_chunks
            try:
                host_in = torch.empty(n_state, dtype=torch.float32, pin_memory=True)
                host_out = torch.empty(n_state, dtype=torch.float32, pin_memory=True)
                ok = 1
            except RuntimeError:
                host_in = host_out = None
                ok = 0
            flag = torch.tensor([ok], dtype=torch.int32, device=dev)
            if world > 1:
                dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            if int(flag.item()) == 1 or n_chunks <= 2:
                break
            host_in = host_out = None
            e2e_pairs //= 2
        e_layers = n_chunks * 2 * chunk_blocks
        for st_ in hc.slots:
            st_.generate()
        for i in range(n_chunks):                                 # synthetic host image (chunks repeat two seeds)
            host_in[i * hc.chunk_floats:(i + 1) * hc.chunk_floats].copy_(hc.slots[i % len(hc.slots)].state())
        torch.cuda.synchronize()

        def e2e_step():
            hc.run(host_in, host_out)

        for _ in range(2):
            e2e_step()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            e2e_step()
        e1.record()
        barrier()
        # the same chunks through the same streams WITHOUT the kernels: what the box's PCIe + host memory give this traffic
        # pattern with all ranks copying at once (the ceiling of the e2e arm)
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        hc.run(host_in, host_out, copy_only=True)
        barrier()
        c0.record()
        for _ in range(2):
            hc.run(host_in, host_out, copy_only=True)
        c1.record()
        barrier()
        mine = torch.tensor([e0.elapsed_time(e1) / args.steps, c0.elapsed_time(c1) / 2], dtype=torch.float64, device=dev)
        per_rank = [torch.zeros_like(mine) for _ in range(world)] if world > 1 else [mine]
        if world > 1:
            dist.all_gather(per_rank, mine)
        tt = torch.stack(per_rank).max(dim=0).values
        e2e = {"value": world * e_layers / (float(tt[0]) * 1e-3), "unit": UNIT, "h2d_bytes_per_step": 4 * n_state,
               "d2h_bytes_per_step": 4 * n_state, "layers_per_step": e_layers, "ms_per_step": float(tt[0]),
               "pcie_GBps_each_way": 4e-9 * n_state / (float(tt[0]) * 1e-3),
               "pcie_GBps_each_way_per_rank": [round(4e-9 * n_state / (float(t[0]) * 1e-3), 2) for t in per_rank],
               "copy_only": {"ms_per_step": float(tt[1]), "GBps_each_way": 4e-9 * n_state / (float(tt[1]) * 1e-3),
                             "GBps_each_way_per_rank": [round(4e-9 * n_state / (float(t[1]) * 1e-3), 2) for t in per_rank],
                             "what": "the same chunks through the same three streams with no kernel launched, all ranks "
                                     "copying at once: the transfer ceiling of this box for the e2e arm"},
               "api": "dfq_b200.workload.HostStackCalibrator.run(pinned_in, pinned_out): %d-pair chunks, H2D / kernels / "
                      "D2H pipelined on three streams over %d arena slots" % (2 * chunk_blocks, args.e2e_slots)}
        del hc, host_in, host_out

    launches_per_step = stack.launches_per_step
    if rank != 0:
        return
    mbv2 = None
    if world == 1 and not args.no_mbv2:
        try:
            del stack, sess
            torch.cuda.empty_cache()
            mbv2 = mobilenetv2_latency(dev)
        except Exception as e:   # noqa: BLE001 - an auxiliary number must not sink the benchmark line
            mbv2 = {"error": repr(e)}
    cpu = None
    if not args.no_cpu_baseline and world == 1:
        pairs = args.cpu_layers or 48          # ~5 s of single-core numpy on the GPU box (plus the input generation)
        import torch as _t
        _t.set_num_threads(os.cpu_count() or 1)
        dt, sw = cpu_pipeline(pairs)
        cpu = {"value": pairs / dt, "unit": UNIT, "cores": 1, "kind": "port",
               "sample": "%d layer pairs, vectorised numpy oracle (oracle/dfq_oracle.py), %d sweeps, %.1f s" % (pairs, sw, dt)}
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": "synthetic stack of %d Conv[512,512,3,3]+BN pairs per GPU (BASELINE configs[4]): "
                                   "BN fold + equalization to convergence + bias correction%s" % (layers, " + 8-bit fake-quant" if args.quantize else ""),
                       "layers_per_gpu": layers, "weights_bytes_per_gpu": 4 * N_PER_LAYER * layers, "sweeps": res.n_sweeps,
                       "parallelism": "independent blocks sharded over %d rank(s); one all-gather of the scale vectors" % world,
                       "l2": "working set %.1f GB >> 126 MB L2; state restored from a pristine copy (untimed) before every step" % (4e-9 * N_PER_LAYER * layers)},
            "phases_ms": {"bn_fold": phases[0], "equalize": phases[1], "bias_correct": phases[2], "exchange": phases[3]},
            "exchange": None if exchange is None else {"bytes_per_rank": 4 * exchange.n,
                                                       "carries": "S of every relation + corrected biases + BN vectors (fake_weight, fake_bias) of every layer, one all_gather_into_tensor"},
            "strong": strong, "numa": numa,
            "clocks": clocks, "e2e": e2e, "gpu_launches": launches_per_step * args.steps,
            "roofline": roofline, "cpu_baseline": cpu, "mobilenetv2": mbv2, "parity_check": parity}
    if args.scaling == "strong" and strong is not None:
        line["weak"] = {"value": line["value"], "ms_per_step": line["ms_per_step"], "layers_per_gpu": layers}
        line["value"], line["ms_per_step"], line["scaling"] = strong["value"], strong["ms_per_step"], "strong"
        line["config"]["workload"] = "synthetic stack of %d Conv[512,512,3,3]+BN pairs IN TOTAL split over %d GPUs (BASELINE configs[4])" % (strong["layers_total"], world)
    print(json.dumps(line))


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    import torch
    import torch.distributed as dist
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_b200(args, rank, world, local_rank)
    finally:
        if world > 1:
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
