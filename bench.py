#!/usr/bin/env python
"""Benchmark of the message-passing hot path (BASELINE.json metric: edges/sec per GNN layer; % of HBM roofline).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--agg sum|max] [--workload graph2class|varmisuse]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json configs[1]): Graph2Class synthetic batch -- 80 graphs x 2,560 nodes = 204,800 nodes, 8 raw
edge types -> T = 17, E = 1,105,920 layer-level edges, hidden 128, 8 GatedMessagePassingLayers, fp32.
One "step" = one minibatch through the layer loop: edge-plan build + 8 layers.  `value` = E * L / step_time
(edges/s per GNN layer), inputs resident in HBM.  `e2e` = the same metric through the public module API with HOST
(pinned) inputs: H2D of states + int64 edge lists and D2H of the output states inside the timed region.
Multi-GPU: graph-granular sharding -- every rank owns its own batch of graphs (block-diagonal => no halo, no
data-path collective), weak scaling; value = (all ranks' edges) * L / max-over-ranks time.
`--impl reference`: the reference's CPU path (torch-CPU oracle port: same ATen ops as the reference classes + the
restated torch_scatter) on all host threads, rank 0 only.
`--dump-outputs DIR`: after the timed steps, rank 0 writes the output node states of the last timed step of the headline loop
to DIR/node_states.npy (float32; a fixed, seeded sample of DUMP_MAX_ROWS rows when there are more).  The inputs and
parameters are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

HIDDEN = 128
NUM_LAYERS = 8
L2_BYTES = 126e6
DUMP_MAX_ROWS = 65536          # 32 MiB of fp32 states at HIDDEN = 128


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def measured_tensor_peak():
    """(TFLOP/s, which).  The per-kernel numbers come from a timed region of ~0.1 s at full clocks (see `clocks` in the line), so the
    BURST cuBLAS bf16 figure is the honest denominator here -- the sustained one was measured at a 1372 MHz power-capped median
    (VERDICT r1: "burst is the right one here")."""
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["bf16_tflops"]), "MEASURED_PEAKS.json bf16_tflops (burst cuBLAS bf16; the timed region is ~0.1 s at full clocks)"
    return 1590.0, "fallback 1.59 PFLOP/s burst (B200_PROFILING.md)"


def tcgen05_peaks():
    """This repo's own tensor-pipe ceiling: back-to-back tcgen05.mma issue rate (csrc/tc_peak.cu, tools/tc_peak.py; committed as
    profiles/r02_tcgen05_peaks.json).  {"f16": TFLOP/s, "tf32": TFLOP/s} at N = 256 with the A operand in tensor memory, or {}."""
    path = os.path.join(ROOT, "profiles", "r02_tcgen05_peaks.json")
    try:
        with open(path) as f:
            res = json.load(f)["results"]
        pick = lambda kind: max(r["tflops"] for r in res if r["kind"] == kind and r["N"] == 256)  # noqa: E731
        return {"f16": pick("f16"), "tf32": pick("tf32"), "source": "profiles/r02_tcgen05_peaks.json (own tcgen05.mma issue-rate kernel, M=128 N=256)"}
    except (OSError, ValueError, KeyError):
        return {}


def ncu_traffic(dtype: str):
    """DRAM traffic per launch (dram__bytes_read.sum + dram__bytes_write.sum) of the CURRENT kernels, from the committed ncu
    --set full capture: profiles/ncu_traffic.json, written by tools/ncu_summary.py --traffic from the .ncu-rep of the round.
    Empty when no capture of this dtype's kernels is committed (traffic is then reported as null)."""
    path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    try:
        with open(path) as f:
            d = json.load(f)
        return {k: float(v) for k, v in d.get(dtype, {}).get("kernels", {}).items()}, d.get(dtype, {}).get("source")
    except (OSError, ValueError):
        return {}, None


def usable_cores() -> int:
    """Host cores this process may actually use: min(affinity mask, cgroup CPU quota)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:  # cgroup v2
            quota, period = f.read().split()
        if quota != "max":
            n = min(n, max(1, int(float(quota) / float(period))))
    except (OSError, ValueError):
        try:  # cgroup v1
            with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as f:
                quota = int(f.read())
            with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f:
                period = int(f.read())
            if quota > 0:
                n = min(n, max(1, quota // period))
        except (OSError, ValueError):
            pass
    return max(1, n)


# ------------------------------------------------------------------------------------------------------
# clocks sampling during the timed region
# ------------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock / throttle-reason samples DURING the timed region.  NVML (pynvml) polled every few ms from a thread -- the
    timed region is only ~0.1 s, too short for `nvidia-smi -lms` -- with nvidia-smi as the fallback."""
    FIELDS = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.samples = []          # (sm_mhz, power_w, reasons bitmask or list)
        self.sm_max = None
        self.proc = None
        self.stop = threading.Event()
        self.thread = None
        self.source = None

    def _nvml_handle(self):
        import pynvml

        pynvml.nvmlInit()
        try:
            uuid = str(torch.cuda.get_device_properties(self.gpu).uuid)
            return pynvml, pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid).encode())
        except Exception:
            return pynvml, pynvml.nvmlDeviceGetHandleByIndex(self.gpu)

    def _poll_nvml(self, nv, h):
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        while not self.stop.is_set():
            try:
                self.samples.append((int(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)), nv.nvmlDeviceGetPowerUsage(h) / 1000.0,
                                     int(get_reasons(h))))
            except Exception:
                break
            time.sleep(0.004)

    def __enter__(self):
        try:
            nv, h = self._nvml_handle()
            self.sm_max = int(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            self.source = "nvml"
            self.thread = threading.Thread(target=self._poll_nvml, args=(nv, h), daemon=True)
            self.thread.start()
            return self
        except Exception:
            self.source = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "20"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.source = "nvidia-smi"
            self.thread = threading.Thread(target=self._read_smi, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None
        return self

    def _read_smi(self):
        for line in self.proc.stdout:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) >= 8:
                try:
                    reasons = [n for n, c in (("hw_slowdown", 4), ("hw_thermal_slowdown", 5), ("sw_thermal_slowdown", 6), ("sw_power_cap", 7))
                               if parts[c].lower().startswith("active")]
                    self.samples.append((int(float(parts[1])), float(parts[3]), reasons))
                    self.sm_max = int(float(parts[2]))
                except ValueError:
                    pass

    def __exit__(self, *exc):
        self.stop.set()
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except subprocess.TimeoutExpired:
                self.proc.kill()
        if self.thread is not None:
            self.thread.join(timeout=2)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["clock sampling unavailable"]}
        sm = sorted(s[0] for s in self.samples)
        reasons = set()
        for _, _, r in self.samples:
            if isinstance(r, int):   # NVML bitmask (nvml.h nvmlClocksEventReason*)
                for name, bit in (("sw_power_cap", 0x4), ("hw_slowdown", 0x8), ("sw_thermal_slowdown", 0x20), ("hw_thermal_slowdown", 0x40)):
                    if r & bit:
                        reasons.add(name)
            else:
                reasons.update(r)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": self.sm_max, "reasons": sorted(reasons), "samples": len(sm),
                "power_w_max": max(s[1] for s in self.samples), "source": self.source}


# ------------------------------------------------------------------------------------------------------
# workload
# ------------------------------------------------------------------------------------------------------
def make_batch(workload: str, seed_offset: int = 0, num_graphs=None):
    from ptgnn_b200 import synthetic

    if workload == "graph2class":
        return synthetic.graph2class_batch(num_graphs or 80, seed=1234 + seed_offset)
    if workload == "varmisuse":
        return synthetic.varmisuse_batch(num_graphs or 40, seed=1235 + seed_offset)
    raise ValueError(workload)


def build_model(num_types: int, agg: str, kind: str = "gated"):
    import ptgnn_b200 as P

    torch.manual_seed(0)
    if kind == "mlp":     # the reference's VarMisuse default stack (varmisuse/train.py:43-74) without its residual pseudo-layers
        layers = [P.MlpMessagePassingLayer(HIDDEN, HIDDEN, HIDDEN, num_types, agg) for _ in range(NUM_LAYERS)]
    else:
        layers = [P.GatedMessagePassingLayer(HIDDEN, HIDDEN, num_types, agg) for _ in range(NUM_LAYERS)]
    gnn = P.GraphNeuralNetwork(layers, torch.nn.Identity(), introduce_backwards_edges=True, add_self_edges=True)
    return gnn.eval()


def oracle_layer_specs(gnn):
    specs = []
    p = "_GatedMessagePassingLayer__"
    for layer in gnn.message_passing_layers:
        sd = {k: v.detach().cpu() for k, v in layer.state_dict().items()}
        T = sum(1 for k in sd if k.startswith(p + "edge_message_transformation_layers."))
        specs.append(dict(kind="gated", edge_weights=[sd[f"{p}edge_message_transformation_layers.{t}.weight"] for t in range(T)],
                          gru_w_ih=sd[p + "state_update.weight_ih"], gru_w_hh=sd[p + "state_update.weight_hh"],
                          gru_b_ih=sd[p + "state_update.bias_ih"], gru_b_hh=sd[p + "state_update.bias_hh"]))
    return specs


def cpu_reference_run(batch, gnn, agg: str, steps: int, warmup: int, budget_s: float):
    """Times the reference's CPU path (oracle port) on all host threads.  Each step = the 8-layer loop on a bounded
    sample (a prefix of the batch's graphs chosen so that the whole run fits `budget_s`)."""
    from oracle import ptgnn_oracle as O  # test/bench infrastructure: the CPU baseline, never the product path
    from ptgnn_b200.synthetic import GraphBatch

    usable = usable_cores()
    specs = [dict(s, aggregation_fn=agg) for s in oracle_layer_specs(gnn)]
    nodes_per_graph = batch.num_nodes // batch.num_graphs

    def sub_batch(g):
        n = g * nodes_per_graph
        adj = []
        for s, t in batch.adjacency_lists:
            keep = t < n  # graphs are contiguous node ranges and edges are intra-graph
            adj.append((s[keep], t[keep]))
        return GraphBatch(n, g, adj, batch.node_to_graph_idx[:n])

    def run(b, h):
        adj = O.expand_adjacency(b.adjacency_lists, b.num_nodes, True, True)
        with torch.no_grad():
            return O.gnn_forward(h, adj, specs)[-1]

    gen = torch.Generator().manual_seed(7)
    # calibrate on 4 graphs: pick the fastest thread count the host offers (oversubscribed OpenMP teams are slower
    # than smaller ones on many-core boxes), then size the sample
    cal = sub_batch(min(4, batch.num_graphs))
    h = torch.randn(cal.num_nodes, HIDDEN, generator=gen)
    best = None
    for cand in sorted({usable, min(usable, 64), min(usable, 32), min(usable, 16), min(usable, 8)}, reverse=True):
        torch.set_num_threads(cand)
        run(cal, h)
        t0 = time.perf_counter()
        run(cal, h)
        dt = time.perf_counter() - t0
        if best is None or dt < best[0]:
            best = (dt, cand)
        if time.perf_counter() - t0 > 20.0:  # pathological setting: do not spend the budget calibrating
            continue
    threads = best[1]
    torch.set_num_threads(threads)
    per_graph = best[0] / cal.num_graphs
    graphs = int(max(1, min(batch.num_graphs, budget_s / max(per_graph * (steps + warmup), 1e-9))))
    sample = sub_batch(graphs)
    h = torch.randn(sample.num_nodes, HIDDEN, generator=gen)
    for _ in range(warmup):
        run(sample, h)
    t0 = time.perf_counter()
    for _ in range(steps):
        run(sample, h)
    dt = (time.perf_counter() - t0) / steps
    edges = sample.layer_level_edges()
    return {
        "value": edges * NUM_LAYERS / dt, "ms_per_step": dt * 1e3, "cores": threads, "kind": "port",
        "sample": f"{graphs}/{batch.num_graphs} graphs of the batch ({sample.num_nodes} nodes, {edges} layer-level edges), "
                  f"{NUM_LAYERS} layers, {steps} timed steps, torch {torch.__version__} CPU, {threads} threads "
                  f"(fastest of the thread counts tried; host offers {usable})",
    }


def dump_outputs(out_dir: str, node_states: torch.Tensor) -> None:
    """Writes `node_states` ([N, HIDDEN], any float dtype, on the GPU) as out_dir/node_states.npy in float32: all rows, or the
    same seeded sample of DUMP_MAX_ROWS rows (in ascending row order) on every run when N is larger."""
    import numpy as np

    n = node_states.shape[0]
    if n > DUMP_MAX_ROWS:
        rows = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:DUMP_MAX_ROWS].sort().values
        node_states = node_states.index_select(0, rows.to(node_states.device))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "node_states.npy"), node_states.float().cpu().numpy())


# ------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--agg", default="sum", choices=["sum", "max", "mean", "min"])
    ap.add_argument("--workload", default="graph2class", choices=["graph2class", "varmisuse"])
    ap.add_argument("--layers", default="gated", choices=["gated", "mlp"],
                    help="mlp = MlpMessagePassingLayer stack (the VarMisuse default); extra record, not the headline config")
    ap.add_argument("--dtype", default="f32", choices=["f32", "bf16"],
                    help="node-state dtype; f32 is the headline (reference CPU path precision), bf16 = BASELINE.json configs[3]")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graphs", action="store_true", help="do not measure the CUDA-graph replay variant of the e2e loop")
    ap.add_argument("--no-train", action="store_true", help="skip the forward + backward extra measurement")
    ap.add_argument("--no-row-shard", action="store_true", help="skip the node-range-split (all-gather) extra measurement")
    ap.add_argument("--profile", action="store_true", help="only the HBM-resident loop (for runs under ncu); prints no bench line")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the output node states of the last timed step to DIR/node_states.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.profile):
        ap.error("--dump-outputs applies to the timed GPU loop (--impl ours, without --profile)")
    args.warmup = max(args.warmup, 3)
    if args.layers == "mlp":
        args.no_cpu_baseline = True      # the CPU-port leg is written for the headline (gated) stack

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    metric = "edges/sec per GNN layer"
    config = {
        "workload": f"{args.workload} synthetic batch per GPU: 80x2560=204,800 nodes, 8 raw edge types -> T=17, E=1,105,920 "
                    f"layer-level edges, hidden {HIDDEN}, {NUM_LAYERS} {'Mlp' if args.layers == 'mlp' else 'Gated'}MessagePassingLayers ({args.agg}), {args.dtype}"
                    if args.workload == "graph2class" else
                    f"varmisuse synthetic batch per GPU: 40x2000 nodes, 11 raw types -> T=23, E=480,000, hidden {HIDDEN}, "
                    f"{NUM_LAYERS} {'Mlp' if args.layers == 'mlp' else 'Gated'}MessagePassingLayers ({args.agg}), {args.dtype}",
        "step": "edge-plan build + 8 layers on one minibatch",
        "parallelism": f"graph-sharded x{world} (no data-path collective)",
        "l2": "per-layer working set (states in + packed copy + aggregate + states out: 0.42 GB fp32 / 0.16 GB bf16) > 126 MB L2 and "
              "every layer reads what the previous one wrote; no explicit flush",
    }

    # ---------------------------------------------------------------- reference arm (CPU, rank 0 only)
    if args.impl == "reference":
        if rank != 0:
            return
        batch = make_batch(args.workload)
        gnn = build_model(2 * len(batch.adjacency_lists) + 1, args.agg, args.layers)
        r = cpu_reference_run(batch, gnn, args.agg, args.steps, args.warmup, budget_s=150.0)
        line = {
            "impl": "reference", "metric": metric, "value": r["value"], "unit": "edges/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
            "cpu_baseline": {"value": r["value"], "unit": "edges/s", "cores": r["cores"], "kind": r["kind"], "sample": r["sample"]},
            "e2e": {"value": r["value"], "unit": "edges/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
        }
        print(json.dumps(line))
        return

    # ---------------------------------------------------------------- our arm (GPU)
    assert torch.cuda.is_available(), "bench.py --impl ours needs a GPU (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    import torch.distributed as dist

    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    import ptgnn_b200 as P
    from ptgnn_b200 import _native as N

    batch = make_batch(args.workload, seed_offset=rank)  # every rank owns different graphs (weak scaling)
    T = 2 * len(batch.adjacency_lists) + 1
    gnn = build_model(T, args.agg, args.layers).to(dev)
    E = batch.layer_level_edges()
    n_nodes = batch.num_nodes

    gen = torch.Generator().manual_seed(7 + rank)
    state_dtype = torch.bfloat16 if args.dtype == "bf16" else torch.float32
    esz = 2 if args.dtype == "bf16" else 4
    h_host = torch.randn(n_nodes, HIDDEN, generator=gen).to(state_dtype).pin_memory()
    adj_host = [(s.pin_memory(), t.pin_memory()) for s, t in batch.adjacency_lists]
    out_host = torch.empty(n_nodes, HIDDEN, dtype=state_dtype).pin_memory()
    h_dev = h_host.to(dev)
    adj_dev = [(s.to(dev), t.to(dev)) for s, t in adj_host]
    n2g = batch.node_to_graph_idx.to(dev)
    ident = torch.arange(n_nodes, dtype=torch.int64, device=dev)

    def expanded(adj):
        return list(adj) + [(t, s) for s, t in adj] + [(ident, ident)]

    def step_resident():
        P.clear_plan_cache()  # every step is a new minibatch: the plan is rebuilt inside the timed region
        with torch.no_grad():
            return gnn.gnn(h_dev, expanded(adj_dev), None, n2g, {}, {})

    def step_e2e():
        P.clear_plan_cache()
        with torch.no_grad():
            h = h_host.to(dev, non_blocking=True)
            adj = [(s.to(dev, non_blocking=True), t.to(dev, non_blocking=True)) for s, t in adj_host]
            res = gnn(node_data={"input": h}, adjacency_lists=adj, edge_feature_data=[], node_to_graph_idx=n2g,
                      reference_node_ids={}, reference_node_graph_idx={}, num_graphs=batch.num_graphs)
            out_host.copy_(res.output_node_representations, non_blocking=True)
        return res

    class PipelinedE2E:
        """Same per-step work as step_e2e (H2D of the step's inputs from pinned host memory, plan + 8 layers through the
        public module API, D2H of the result), but software-pipelined across steps on three streams: the H2D of step i+1
        and the D2H of step i-1 overlap the kernels of step i -- what the reference's own background minibatch threads do
        (`ptgnn/baseneuralmodel/abstractneuralmodel.py:348-357`)."""

        def __init__(self, graphed: bool = False, pooled: bool = False):
            self.graphed = graphed           # replay GraphNeuralNetwork.capture() graphs (one per input buffer) instead of eager calls
            self.pooled = pooled             # result read back = per-graph mean of the output states (a Graph2Class-style readout on the
                                             # native scatter kernel) instead of all node states
            self.pool_host = [torch.empty(batch.num_graphs, HIDDEN, dtype=torch.float32).pin_memory() for _ in range(2)]
            self.graphs = [None, None]
            self.h2d, self.d2h = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
            self.h_buf = [torch.empty_like(h_dev) for _ in range(2)]
            self.adj_buf = [[(torch.empty_like(s), torch.empty_like(t)) for s, t in adj_dev] for _ in range(2)]
            self.out_host = [torch.empty(n_nodes, HIDDEN, dtype=state_dtype).pin_memory() for _ in range(2)]
            self.in_ready = [torch.cuda.Event() for _ in range(2)]
            self.compute_done = [torch.cuda.Event() for _ in range(2)]
            self.d2h_done = [torch.cuda.Event() for _ in range(2)]
            self.keep = [None, None]
            self.i = 0
            self.prefetched = [False, False]

        def _prefetch(self, k):
            with torch.cuda.stream(self.h2d):
                self.h2d.wait_event(self.compute_done[k])      # the step that last read buffer k has finished
                self.h_buf[k].copy_(h_host, non_blocking=True)
                for (ds, dt), (hs, ht) in zip(self.adj_buf[k], adj_host):
                    ds.copy_(hs, non_blocking=True)
                    dt.copy_(ht, non_blocking=True)
                self.in_ready[k].record(self.h2d)
            self.prefetched[k] = True

        def step(self):
            k = self.i % 2
            main = torch.cuda.current_stream(dev)
            if not self.prefetched[k]:
                self._prefetch(k)
            main.wait_event(self.in_ready[k])
            if self.graphed:
                if self.graphs[k] is None:      # first use of this buffer pair (inside the warm-up): capture plan + 8 layers
                    self.graphs[k] = gnn.capture(self.h_buf[k], gnn.expand_adjacency(self.adj_buf[k], n_nodes, dev), n2g)
                out = self.graphs[k].replay()
            else:
                P.clear_plan_cache()
                with torch.no_grad():
                    res = gnn(node_data={"input": self.h_buf[k]}, adjacency_lists=list(self.adj_buf[k]), edge_feature_data=[],
                              node_to_graph_idx=n2g, reference_node_ids={}, reference_node_graph_idx={}, num_graphs=batch.num_graphs)
                out = res.output_node_representations
            result, result_host = out, self.out_host[k]
            if self.pooled:
                result, result_host = P.scatter_mean(out.float(), n2g, dim=0, dim_size=batch.num_graphs), self.pool_host[k]
            self.compute_done[k].record(main)
            with torch.cuda.stream(self.d2h):
                self.d2h.wait_event(self.compute_done[k])
                result_host.copy_(result, non_blocking=True)
                self.d2h_done[k].record(self.d2h)
            if self.pooled:
                result.record_stream(self.d2h)
            if not self.graphed:
                out.record_stream(self.d2h)
            self.keep[k] = out
            self.prefetched[k] = False
            self._prefetch(1 - k)                               # inputs of the next step
            self.i += 1

        def finish(self):                                       # the timed region ends when the last result is on the host
            main = torch.cuda.current_stream(dev)
            for ev in self.d2h_done:
                main.wait_event(ev)
            main.wait_stream(self.h2d)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup, finish=None, keep_last=False):
        for _ in range(warmup):
            fn()
        if finish:
            finish()
        barrier()
        launches0 = N.launch_count()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        t_host = time.perf_counter()
        for _ in range(steps - 1):
            fn()
        last = fn()
        if finish:
            finish()
        b.record()
        timed.host_ms = (time.perf_counter() - t_host) * 1e3 / steps   # host enqueue time per step (no device sync)
        timed.last = last if keep_last else None                         # what the last timed step returned
        barrier()
        ms = a.elapsed_time(b)
        t = torch.tensor([ms], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()) / steps, (N.launch_count() - launches0) / steps

    if args.profile:
        for _ in range(args.warmup + args.steps):
            step_resident()
        torch.cuda.synchronize()
        return
    with ClockSampler(local_rank) as clocks:
        ms_step, launches = timed(step_resident, args.steps, args.warmup, keep_last=bool(args.dump_outputs))
    clock_summary = clocks.summary()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, timed.last)
    timed.last = None
    ms_e2e_serial, _ = timed(step_e2e, args.steps, args.warmup)
    pipe = PipelinedE2E()
    ms_e2e_eager, _ = timed(pipe.step, args.steps, args.warmup, finish=pipe.finish)
    host_ms_eager = timed.host_ms
    ms_e2e, host_ms_e2e, e2e_mode = ms_e2e_eager, host_ms_eager, "eager"
    if not args.no_graphs:
        try:
            gpipe = PipelinedE2E(graphed=True)
            ms_g, _ = timed(gpipe.step, args.steps, max(args.warmup, 4), finish=gpipe.finish)
            if ms_g < ms_e2e_eager:
                ms_e2e, host_ms_e2e, e2e_mode = ms_g, timed.host_ms, "cuda-graph"
            graph_info = {"ms_per_step": ms_g, "host_enqueue_ms_per_step": timed.host_ms}
        except Exception as exc:     # capture is an optimisation of the host side only: report, never hide
            graph_info = {"error": repr(exc)[:300]}
    else:
        graph_info = None
    # extra record: the same loop when the result read back is a per-graph readout (41 KB) instead of all node states (105 MB) --
    # what a graph-level model actually returns; shows how much of the multi-GPU e2e figure is the host link
    pooled_info = None
    if not args.no_graphs:
        try:
            ppipe = PipelinedE2E(graphed=True, pooled=True)
            ms_p, _ = timed(ppipe.step, args.steps, max(args.warmup, 4), finish=ppipe.finish)
            pooled_info = {"ms_per_step": ms_p, "value": E * world * NUM_LAYERS / (ms_p * 1e-3), "d2h_bytes_per_step": batch.num_graphs * HIDDEN * 4,
                           "result": "per-graph mean of the output node states (ptgnn_b200.scatter_mean), fp32"}
        except Exception as exc:
            pooled_info = {"error": repr(exc)[:300]}

    total_edges = E * world
    value = total_edges * NUM_LAYERS / (ms_step * 1e-3)
    e2e_value = total_edges * NUM_LAYERS / (ms_e2e * 1e-3)
    h2d = h_host.numel() * esz + sum(s.numel() * 8 + t.numel() * 8 for s, t in adj_host)
    d2h = out_host.numel() * esz

    # ---- per-kernel timing leg (CUDA events on the launch stream, inside the library) -> roofline
    N.kernel_timing(True)
    for _ in range(args.warmup):
        step_resident()
    N.read_kernel_timing()
    ksteps = args.steps
    for _ in range(ksteps):
        step_resident()
    kt = N.read_kernel_timing()
    N.kernel_timing(False)
    peak, peak_src = measured_peaks()
    tensor_peak, tensor_src = measured_tensor_peak()
    D = HIDDEN
    fused = kt.get("reduce", (0.0, 0))[1] == 0          # no stand-alone reduce launches: the fused aggregation kernel ran
    w_bytes = T * D * HIDDEN * (4 if args.dtype == "f32" else 2)          # packed edge weights (hi|lo' fp16 pairs, or bf16)
    if fused:
        alg_bytes = {  # per launch (DESIGN.md section 3): states once (per-graph working set is L2 resident), 5 index bytes per
                       # edge + group offsets, weights, the aggregate written once -- there is no [E, D] tensor any more
            "message": n_nodes * HIDDEN * esz + E * 5 + (n_nodes // 128 + 1) * T * 4 + w_bytes + n_nodes * D * esz,
            "gru": n_nodes * D * esz + 2 * n_nodes * HIDDEN * esz + 6 * HIDDEN * HIDDEN * esz,
            "pack": 2 * n_nodes * HIDDEN * 4,
        }
    else:
        alg_bytes = {
            "message": n_nodes * HIDDEN * esz + E * (D * esz + 8),
            "reduce": E * D * esz + (n_nodes + 1) * 4 + n_nodes * D * esz,
            "gru": n_nodes * D * esz + 2 * n_nodes * HIDDEN * esz + 6 * HIDDEN * HIDDEN * esz,
        }
    k_in = 2 * HIDDEN if args.layers == "mlp" else HIDDEN      # Mlp layers: [h_src ; h_tgt] -> message
    alg_flops = {  # the reference's multiply-adds (x2)
        "message": 2 * E * k_in * D,
        "gru": 2 * n_nodes * (3 * HIDDEN * D + 3 * HIDDEN * HIDDEN),
    }
    # MMAs issued per reference product and their rate relative to the bf16 peak: fused fp32 = 3 kind::f16 products (3xFP16);
    # unfused fp32 message / GRU = 3 kind::tf32 products at half the bf16 rate (3xTF32); bf16 = 1
    gru_ws = fused and os.environ.get("PTGNN_B200_GRU", "") != "tc"        # weights-stationary GRU kernel: 3xFP16 as well
    if args.dtype == "f32":
        exact_div = {"message": 3.0 if fused else 6.0, "gru": 3.0 if gru_ws else 6.0}
    else:
        exact_div = {"message": 1.0, "gru": 1.0}
    own_peaks = tcgen05_peaks()
    kernel_names = {"message": "tc_pipeline_kernel<MsgPolicy> (edge messages)", "reduce": "segment_reduce_stream_kernel",
                    "gru": "tc_pipeline_kernel<GruPolicy> (GRUCell update)", "plan": "edge-plan kernels", "pack": "weight split/pack"}
    if args.dtype == "bf16":
        kernel_names.update(message="tc_pipeline_bf16_kernel<MsgPolicyB>", reduce="segment_reduce_bf16_kernel",
                            gru="tc_pipeline_bf16_kernel<GruPolicyB>")
    if fused:
        kernel_names.update(message="fused_aggregate_kernel (gather -> W_t -> segmented reduce, %s)" % ("3xFP16" if args.dtype == "f32" else "bf16"),
                            gru="gru_ws_kernel (weights-stationary GRUCell, %s)" % ("3xFP16" if args.dtype == "f32" else "bf16") if gru_ws else kernel_names["gru"],
                            pack="pack_states_kernel (fp32 -> fp16 hi|lo' rows) + weight packing", plan="edge-plan + block-plan kernels")
    traffic, traffic_src = ncu_traffic(args.dtype)
    kernels = {}
    for name, (ms, cnt) in kt.items():
        if cnt:
            avg_ms = ms / cnt
            entry = {"kernel": kernel_names.get(name, name), "avg_ms": avg_ms, "launches_per_step": cnt / ksteps,
                     "share_of_step": ms / ksteps / ms_step}
            if name in alg_bytes and not (name == "pack" and args.dtype == "bf16"):
                entry["alg_bytes"] = alg_bytes[name]
                entry["achieved_gbs"] = alg_bytes[name] / (avg_ms * 1e-3) / 1e9
                entry["frac_hbm"] = entry["achieved_gbs"] / peak
                entry["ncu_dram_bytes"] = traffic.get(name)
            if name in alg_flops:
                entry["alg_tflops"] = alg_flops[name] / (avg_ms * 1e-3) / 1e12
                entry["frac_tensor_bf16_peak"] = entry["alg_tflops"] / tensor_peak
            kernels[name] = entry
    # Which roofline bounds a kernel: the larger of its HBM floor (algorithmic bytes / measured copy bandwidth) and its tensor
    # floor (algorithmic flops x MMAs per product / measured bf16 rate).
    for name, entry in kernels.items():
        if "alg_bytes" not in entry:
            continue
        t_hbm = entry["alg_bytes"] / (peak * 1e9)
        ceiling = tensor_peak / exact_div.get(name, 1.0)
        t_tensor = alg_flops[name] / (ceiling * 1e12) if name in alg_flops else 0.0
        entry["floor_ms"] = {"hbm": t_hbm * 1e3, "tensor": t_tensor * 1e3}
        entry["bound"] = "tensor" if t_tensor > t_hbm else "hbm"
        if name in alg_flops:
            entry["tensor_ceiling_tflops"] = ceiling
            entry["frac_tensor_exact_peak"] = entry["alg_tflops"] / ceiling
            if own_peaks:      # the stricter denominator: this GPU's tcgen05 issue rate (kind::f16; kind::tf32 runs at half of it)
                entry["frac_of_tcgen05_issue_rate"] = entry["alg_tflops"] / (own_peaks["f16"] / exact_div.get(name, 1.0))
    # the kernel with the largest share of the step
    dominant = max((k for k in kernels if "alg_bytes" in kernels[k] and k != "pack"),
                   key=lambda k: kernels[k]["avg_ms"] * kernels[k]["launches_per_step"])
    dk = kernels[dominant]
    if dk["bound"] == "tensor":
        roofline = {
            "kernel": dk["kernel"], "bound": "tensor", "achieved": dk["alg_tflops"], "peak": dk["tensor_ceiling_tflops"], "unit": "TFLOP/s",
            "frac": dk["frac_tensor_exact_peak"], "traffic": traffic.get(dominant), "traffic_source": traffic_src,
            "peak_source": tensor_src + " / %g (MMAs issued per fp32-exact product x rate ratio)" % exact_div.get(dominant, 1.0),
            "note": "dominant kernel by time. achieved = the reference's multiply-adds (x2) per launch / CUDA-event launch time; "
                    "kernels[*].floor_ms has both floors and kernels[*].frac_hbm the bandwidth view.",
        }
        if own_peaks:
            roofline["tcgen05_issue_rate"] = {"f16_tflops": own_peaks["f16"], "tf32_tflops": own_peaks["tf32"], "source": own_peaks["source"],
                                              "frac": dk.get("frac_of_tcgen05_issue_rate")}
    else:
        roofline = {
            "kernel": dk["kernel"], "bound": "hbm", "achieved": dk["achieved_gbs"], "peak": peak, "unit": "GB/s",
            "frac": dk["frac_hbm"], "traffic": traffic.get(dominant), "traffic_source": traffic_src, "peak_source": peak_src,
            "note": "dominant kernel by time; algorithmic bytes per launch / CUDA-event launch time (kernels[*].floor_ms has both floors)",
        }
    b_min = 2 * n_nodes * HIDDEN * esz + 8 * E + (T * D * HIDDEN + 6 * HIDDEN * HIDDEN + 6 * HIDDEN) * esz
    layer_ms = ms_step / NUM_LAYERS
    layer_roofline = {"alg_bytes_fully_fused": b_min, "achieved_gbs": b_min / (layer_ms * 1e-3) / 1e9,
                      "frac": b_min / (layer_ms * 1e-3) / 1e9 / peak, "ms_per_layer": layer_ms,
                      "nodes_per_sec_per_layer": n_nodes * world / (layer_ms * 1e-3)}

    # ---- BASELINE.json configs[3] extras (kept out of `value`): (1) the node-range split of ONE connected graph of the same size
    # (N = 204,800, T = 17, E = 1,105,920; strong scaling) with the per-layer NCCL all-gather of the state shards, in this
    # run's dtype; (2) the exposed time of those all-gathers alone.  At world == 1 the all-gather is a no-op.
    row_shard = None
    if args.workload == "graph2class" and not args.no_row_shard:
        from ptgnn_b200 import sharding
        from ptgnn_b200.synthetic import single_random_graph

        g1 = single_random_graph(n_nodes, sum(int(a[0].shape[0]) for a in batch.adjacency_lists), len(batch.adjacency_lists), seed=77)
        full_adj = [(s.to(dev), t.to(dev)) for s, t in g1.adjacency_lists]
        full_adj = list(full_adj) + [(t, s) for s, t in full_adj] + [(ident, ident)]
        shard = sharding.row_shard(n_nodes, full_adj, world, rank)
        loop = sharding.RowShardedLayerLoop(shard)
        own = h_dev[shard.lo:shard.hi].contiguous()
        layer_fns = [lambda o, f, a, L=L: L(o, a, gather_states=f if world > 1 else None) for L in gnn.message_passing_layers]

        def step_rows():
            P.clear_plan_cache()
            with torch.no_grad():
                return loop.run(own, layer_fns)

        def step_allgather_only():
            with torch.no_grad():
                for _ in range(NUM_LAYERS):
                    loop.all_gather_states(own)

        ms_rows, _ = timed(step_rows, args.steps, args.warmup)
        ms_ag, _ = timed(step_allgather_only, args.steps, args.warmup) if world > 1 else (0.0, 0)
        E1 = sum(int(a[0].shape[0]) for a in full_adj)
        row_shard = {"workload": f"one connected random graph, N={n_nodes}, T={len(full_adj)}, E={E1}, node-range split over {world} rank(s), "
                                 f"one all_gather_into_tensor of the [N/P, {HIDDEN}] state shards per layer (NCCL)",
                     "value": E1 * NUM_LAYERS / (ms_rows * 1e-3), "unit": "edges/s", "ms_per_step": ms_rows, "scaling": "strong",
                     "allgather_ms_per_step": ms_ag, "allgather_bytes_per_layer": n_nodes * HIDDEN * esz,
                     "note": "the all-gathers are not overlapped with compute: allgather_ms_per_step is fully exposed"}

    # ---- training step (SURVEY.md section 8 f-1; extra record, kept out of `value`): forward + backward of the same 8-layer stack on
    # the same resident minibatch, loss = mean of the output states, gradients for the states and every parameter
    train = None
    if args.dtype == "f32" and world == 1 and not args.no_train:
        try:
            gnn.train()
            h_train = h_dev.clone().requires_grad_(True)

            def step_train():
                P.clear_plan_cache()
                adj = expanded(adj_dev)
                for p in gnn.parameters():
                    p.grad = None
                h_train.grad = None
                out = gnn.gnn(h_train, adj, None, n2g, {}, {})
                out.mean().backward()

            ms_train, _ = timed(step_train, args.steps, args.warmup)
            train = {"ms_per_step": ms_train, "value": E * NUM_LAYERS / (ms_train * 1e-3), "unit": "edges/s (forward + backward)",
                     "note": "fp32; forward = the fused kernels, backward = native edge-sized kernels on the transposed graph + library GEMMs "
                             "for the parameter gradients (ptgnn_b200/autograd.py)"}
        except Exception as e:  # an extra record must never take the headline line down
            train = {"error": f"{type(e).__name__}: {e}"[:300]}
        finally:
            gnn.eval()

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline and args.dtype == "f32":
        r = cpu_reference_run(batch, gnn, args.agg, steps=3, warmup=1, budget_s=25.0)
        cpu = {"value": r["value"], "unit": "edges/s", "cores": r["cores"], "kind": r["kind"], "sample": r["sample"]}

    if rank == 0:
        line = {
            "metric": metric, "value": value, "unit": "edges/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": args.dtype,
            "data": "synthetic", "config": config, "clocks": clock_summary,
            "e2e": {"value": e2e_value, "unit": "edges/s", "ms_per_step": ms_e2e, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "mode": "pipelined over steps on 3 streams: H2D(i+1) and D2H(i-1) overlap the kernels of step i; every step copies "
                            "its inputs from pinned host memory and its result back; layer loop = " + e2e_mode +
                            (" (GraphNeuralNetwork.capture: plan build + 8 layers replayed as one CUDA graph)" if e2e_mode == "cuda-graph" else ""),
                    "eager_pipelined": {"value": total_edges * NUM_LAYERS / (ms_e2e_eager * 1e-3), "ms_per_step": ms_e2e_eager,
                                        "host_enqueue_ms_per_step": host_ms_eager},
                    "cuda_graph_pipelined": graph_info, "cuda_graph_pipelined_pooled_result": pooled_info,
                    "serial_value": total_edges * NUM_LAYERS / (ms_e2e_serial * 1e-3), "serial_ms_per_step": ms_e2e_serial,
                    "host_enqueue_ms_per_step": host_ms_e2e},
            "gpu_launches": launches * args.steps, "gpu_launches_per_step": launches,
            "roofline": roofline, "layer_roofline": layer_roofline, "kernels": kernels, "cpu_baseline": cpu, "row_shard": row_shard, "train_step": train,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
