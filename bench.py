#!/usr/bin/env python
"""bench.py — headline benchmark of the B200 hot path (BASELINE.json: DLRM & TwoTower fwd samples/s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload all|dlrm|dlrm-sharded|twotower|dcn|dlrm-train] [--batch B] [--dump-outputs DIR]

Headline workload = BASELINE.json configs[1]: mm.DLRMModel, Criteo shape (26 cat, 13 dense, emb 64,
bundled cardinalities = 45.6 M rows / 11.7 GB of tables), batch 65 536, README MLP dims.
A step = one forward pass over one batch of synthetic input.  N>1 (torchrun): one replica per
GPU on disjoint batches, no data-path collective (the forward is replica-local; DESIGN.md (e)),
weak scaling.

Prints ONE JSON line (contract in the task statement): value = device-resident samples/s,
e2e = the same metric through the public host-buffer call (pinned H2D of a PACKED batch — ids at 1/2/3
bytes — + forward + D2H inside the timed region), roofline = dominant kernel vs measured HBM peak (both
the algorithmic-bytes fraction and the DRAM-traffic fraction), cpu_baseline = CPU restatement of the
reference op sequence on this box's host cores (rank 0, N=1 only).
The default `--workload all` adds to the same line:
  "secondary": {"twotower": {...}, "dcn": {...}} — configs[2] (10 M-item catalog, in-batch negatives,
      batch 16 384) and configs[4] (DCN-v2 depth 3 + MLP[256,128], batch 65 536), each with its own value,
      e2e and roofline (the other half of BASELINE.json's metric), replicas under torchrun; plus "dlrm_train":
      one TRAINING step of the headline DLRM (forward + BCE + backward + Adagrad, SURVEY §8(f)-4) as one CUDA graph;
  "sharded": {...} (N > 1 only) — configs[3]: Criteo-TB-shape tables row-sharded over the N GPUs, lookup
      fused into the interaction kernel over NVLink peer memory, checked bit-exact against the unsharded
      model on the same box, with ms/step, NVLink GB/s per GPU and the staged (all-gather + push + barrier)
      protocol timed beside it.
`--impl reference` times the CPU restatement alone on the SAME 65 536-sample step (TensorFlow is not
installable: no network).  `--workload dlrm|twotower|dcn|dlrm-sharded` print a line for that workload only.
`--dump-outputs DIR` writes, after the timed steps, what each timed path computed in its last timed step as
DIR/<name>.npy (float32, rank 0; a fixed, seeded row sample where an output is too large).  Inputs, tables and
weights are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

HBM_FALLBACK_GBS = 6650.0  # B200_PROFILING.md fallback when MEASURED_PEAKS.json is absent


def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return HBM_FALLBACK_GBS, "fallback (B200_PROFILING.md)"


# ---------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi in the background during the timed region)
# ---------------------------------------------------------------------------------------------
class ClockSampler:
    """Polls NVML (SM clock + clock-event reasons) every ~2 ms in a thread for the duration of the
    timed region; the same fields `nvidia-smi --query-gpu=clocks.sm,clocks_event_reasons.*` prints
    (B200_PROFILING.md), without its ~100 ms start-up that would miss a short region."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.sm, self.mask, self.max_mhz = [], 0, None
        self._stop = threading.Event()
        self.t = None
        self.err = None

    def _phys_index(self):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            try:
                return int(vis.split(",")[self.idx])
            except Exception:
                return self.idx
        return self.idx

    def start(self):
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self._phys_index())
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception as e:  # pragma: no cover
            self.err = f"{type(e).__name__}: {e}"
            return
        self.t = threading.Thread(target=self._poll, daemon=True)
        self.t.start()

    def _poll(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                self.mask |= int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
            except Exception as e:  # pragma: no cover
                self.err = f"{type(e).__name__}: {e}"
                return
            time.sleep(0.002)

    def stop(self):
        self._stop.set()
        if self.t is not None:
            self.t.join(timeout=1.0)
        if not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [self.err or "no samples"], "samples": 0}
        reasons = sorted(n for bit, n in self.REASONS.items() if self.mask & bit)
        return {"sm_mhz": float(np.median(self.sm)), "sm_max_mhz": self.max_mhz, "reasons": reasons,
                "samples": len(self.sm)}


# ---------------------------------------------------------------------------------------------
# workloads
# ---------------------------------------------------------------------------------------------
def build_dlrm(mm, datasets, table_seed=4321):
    schema = datasets.criteo_schema()
    model = mm.DLRMModel(schema, embedding_dim=64, bottom_block=mm.MLPBlock([128, 64]),
                         top_block=mm.MLPBlock([128, 64, 32]),
                         embedding_options=mm.EmbeddingOptions(embeddings_initializers={"hash_seed": table_seed}))
    return schema, model


def host_batches(datasets, schema, B, n, seed0=1234):
    out = []
    for i in range(n):
        b = datasets.generate_batch(schema, B, seed=seed0 + i, index_law="uniform", index_dtype=np.int32)
        feats, _ = datasets.split_targets(schema, b)
        out.append(feats)
    return out


def ncu_traffic_bytes(summary: Path):
    """DRAM bytes (read + write) per launch of the dominant kernel, from the committed summary of an
    `ncu --set full` capture (profiles/); None if the file is missing."""
    try:
        rd = wr = None
        for ln in summary.read_text().splitlines():
            parts = ln.split()
            if len(parts) >= 3 and parts[0] == "dram__bytes_read.sum":
                rd = float(parts[1]) * {"Mbyte": 1e6, "Gbyte": 1e9, "Kbyte": 1e3, "byte": 1}[parts[2]]
            if len(parts) >= 3 and parts[0] == "dram__bytes_write.sum":
                wr = float(parts[1]) * {"Mbyte": 1e6, "Gbyte": 1e9, "Kbyte": 1e3, "byte": 1}[parts[2]]
        return None if rd is None or wr is None else rd + wr
    except Exception:
        return None


def dlrm_bytes_per_sample(T=26, D=64, id_bytes_total=104, P=64):
    """SURVEY §8(d): rows read + ids + bottom vector + output row = 8 676 B with int32 ids."""
    F = T + 1
    fused = T * D * 4 + id_bytes_total + D * 4 + (P + F * (F - 1) // 2) * 4
    gather = 2 * T * D * 4 + id_bytes_total  # standalone gather: 13 416 B
    return fused, gather


NCU_FUSED_SUMMARY = "profiles/r02_ncu_fused_operand.txt"  # `ncu --set full` summary of THIS round's dominant kernel

DUMP_LIMIT_BYTES = 64 << 20  # all of --dump-outputs together
DUMP_SAMPLE_BYTES = 16 << 20  # an output larger than this is dumped as a seeded row sample of about this size
DUMP_SEED = 0


def last_output(pf):
    """Device output of the last step submitted to the pipeline `pf`."""
    return pf.output((pf.n - 1) % len(pf.slots))


def sample_rows(t, n=None):
    """A fixed, seeded sample of the rows of the 2-D tensor `t` (of `n` rows, or of about DUMP_SAMPLE_BYTES), in row order."""
    import torch

    if n is None:
        n = DUMP_SAMPLE_BYTES // (4 * max(1, t[0].numel()))
    n = max(1, min(int(n), t.shape[0]))
    idx = np.sort(np.random.default_rng(DUMP_SEED).choice(t.shape[0], size=n, replace=False))
    return t[torch.from_numpy(idx).to(t.device)]


def write_dumps(out_dir, arrays):
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES}-byte limit")
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    for name, a in arrays.items():
        np.save(d / f"{name}.npy", a)


def cpu_baseline_dlrm(model, feats_host, sample_rows, threads):
    """CPU restatement (oracle/oracle_torch.py) on `sample_rows` samples of the same workload, with
    the model's own tables/weights copied to the host."""
    import torch
    from oracle import oracle_torch

    torch.set_num_threads(threads)
    body = model.body
    tables = {n: t.embeddings.cpu() for n, t in body.embeddings.tables.items()}
    f2t = {f: t.table_name for f, t in body.embeddings.feature_to_table.items()}
    layers = lambda mlp: [{"kernel": l.kernel.cpu(), "bias": l.bias.cpu(), "activation": l.activation}
                          for l in mlp.dense_layers]
    bottom, top = layers(body.bottom_block), layers(body.top_block)
    hd = model.prediction.to_call
    head = {"kernel": hd.kernel.cpu(), "bias": hd.bias.cpu(), "activation": hd.activation}
    idx = {n: torch.from_numpy(feats_host[n][:sample_rows]) for n in f2t}
    dense = {n: torch.from_numpy(feats_host[n][:sample_rows]) for n in body.continuous.features}

    def run():
        return oracle_torch.dlrm_forward(idx, dense, tables, f2t, bottom, top, head)

    return run



class Ctx:
    """Process-wide handles shared by the workload functions."""

    def __init__(self, args, mm, datasets, ops, dev, rank, local_rank, world):
        self.args, self.mm, self.datasets, self.ops = args, mm, datasets, ops
        self.dev, self.rank, self.local_rank, self.world = dev, rank, local_rank, world
        self.dumping = bool(args.dump_outputs) and rank == 0
        self.dumps = {}

    def dump(self, name, t):
        """Keep a float32 host copy of an output of a timed path for --dump-outputs (nothing when not dumping)."""
        if self.dumping:
            self.dumps[name] = t.detach().float().cpu().numpy()

    def barrier(self):
        import torch

        if self.world > 1:
            import torch.distributed as dist

            dist.barrier(device_ids=[self.local_rank])
        torch.cuda.synchronize()

    def max_over_ranks(self, *vals):
        import torch

        if self.world == 1:
            return [float(v) for v in vals]
        import torch.distributed as dist

        t = torch.tensor(list(vals), dtype=torch.float64, device=self.dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(x) for x in t.tolist()]

    def sum_over_ranks(self, v):
        import torch

        if self.world == 1:
            return int(v)
        import torch.distributed as dist

        t = torch.tensor([int(v)], dtype=torch.int64, device=self.dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return int(t.item())


def timed_replay(ctx, pf, packed_dev, steps, warmup):
    """K device-resident steps through model.pipeline (graph replays on `depth` streams): CUDA events on the
    submitting stream, barrier + synchronize on both sides, clocks sampled during the region."""
    import torch

    n_bufs = len(packed_dev)
    pf.n = 0
    for i in range(warmup):
        pf.submit_device(packed_dev[i % n_bufs])
    pf.join()
    ctx.barrier()
    sampler = ClockSampler(ctx.local_rank)
    sampler.start()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for i in range(steps):
        pf.submit_device(packed_dev[i % n_bufs])
    pf.join()
    t1.record()
    ctx.barrier()
    clocks = sampler.stop()
    return t0.elapsed_time(t1), clocks


def timed_serial(cf, packed_dev, steps):
    import torch

    n_bufs = len(packed_dev)
    for i in range(3):
        cf.load_device(packed_dev[i % n_bufs])
        cf.replay()
    torch.cuda.synchronize()
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s0.record()
    for i in range(steps):
        cf.load_device(packed_dev[i % n_bufs])
        cf.replay()
    s1.record()
    torch.cuda.synchronize()
    return s0.elapsed_time(s1) / steps


def timed_e2e(ctx, pf, hbs, steps, depth):
    """Public host-buffer call: per step ONE pinned H2D of the packed batch + graph + D2H of the predictions,
    `depth` steps in flight; wall clock from first submit to last result on the host."""
    import torch

    n_bufs = len(hbs)

    def loop(n):
        tickets, res = [], None
        for i in range(n):
            tickets.append(pf.submit(hbs[i % n_bufs]))
            if len(tickets) == depth:
                res = pf.result(tickets.pop(0))
        while tickets:
            res = pf.result(tickets.pop(0))
        return res

    pf.n = 0
    loop(depth + 1)
    ctx.barrier()
    pf.n = 0
    w0 = time.perf_counter()
    res = loop(steps)
    torch.cuda.synchronize()
    ms = (time.perf_counter() - w0) * 1e3
    ctx.barrier()
    return ms, res


def event_times(fn, n, warmup=3):
    """Mean duration of `fn(i)` launched back to back, one CUDA-event pair per launch."""
    import torch

    for i in range(warmup):
        fn(i)
    torch.cuda.synchronize()
    evs = []
    for i in range(n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn(i)
        e1.record()
        evs.append((e0, e1))
    torch.cuda.synchronize()
    return float(np.mean([a.elapsed_time(b) for a, b in evs]))


# ---------------------------------------------------------------------------------------------
# headline: DLRM replicas
# ---------------------------------------------------------------------------------------------
def dlrm_record(ctx):
    import torch

    args, mm, datasets, ops, dev, world = ctx.args, ctx.mm, ctx.datasets, ctx.ops, ctx.dev, ctx.world
    B = args.batch or 65536
    schema, model = build_dlrm(mm, datasets)
    model.build(dev)
    n_bufs = 4
    hosts = host_batches(datasets, schema, B, n_bufs, seed0=1234 + 1000 * ctx.rank)
    widths = model.id_bytes()
    # packed pinned host batches (one allocation each, ids at 1/2/3 bytes) and their device-resident copies
    hbs = [mm.HostBatch.like(h, model.input_columns(), id_bytes=widths) for h in hosts]
    packed_dev = [hb.buffer.to(dev) for hb in hbs]
    devs = [{k: torch.from_numpy(v).to(dev) for k, v in h.items()} for h in hosts]
    torch.cuda.synchronize()

    # the public serving call: forward captured into a CUDA graph over static buffers
    cf = model.compile(hbs[0])
    ref_out = model(devs[0])  # int32 ids through the eager path
    cf.load_device(packed_dev[0])
    assert torch.equal(ref_out, cf.replay()), "graph replay on packed ids diverges from model.__call__ on int32 ids"

    # Steps are independent forward passes; `depth` graph instances on as many streams let the small kernels
    # of step i+1 (bottom MLP, narrow top layers) fill SMs that step i leaves idle — the same runtime
    # the host-buffer path uses.  K steps are still exactly K forward passes over K batches.
    depth = args.pipeline_depth
    pf = model.pipeline(hbs[0], depth=depth)
    pf.submit_device(packed_dev[1])
    pf.join()
    torch.cuda.synchronize()
    assert torch.equal(model(devs[1]), pf.output(0)), "pipelined replay diverges from model.__call__"

    elapsed_ms, clocks = timed_replay(ctx, pf, packed_dev, args.steps, args.warmup)
    ctx.dump("dlrm_predictions", last_output(pf))
    launches = cf.launches_per_replay * args.steps
    serial_ms = timed_serial(cf, packed_dev, args.steps)

    # ---- roofline of the dominant kernel: launched back to back on the same rotating (packed) inputs with a
    # CUDA-event pair around every launch (graph nodes cannot be bracketed individually)
    body = model.body
    slots = body.slots()
    names = body.embeddings.feature_names
    operand = body.use_operand_rows()  # split-bf16 table mirrors + operand-format bottom vector (what the step runs)
    tables = [body.embeddings.feature_to_table[f].operand_mirror() if operand else body.embeddings.feature_to_table[f].table
              for f in names]
    rows = [t.shape[0] for t in tables]
    slot_list = [slots[f] for f in names]
    bottoms = [body.bottom_forward(d, operand_out=operand) for d in devs]
    width = body.output_width_before_top()
    a_out = torch.empty((B, 2 * ops.tc_padded_k(width)), dtype=torch.bfloat16, device=dev)
    # packed id views of the device-resident batches (same layout the graph reads)
    from models_b200.graph import _view

    idx_lists = [[_view(pd, hbs[0].offsets[f], *hbs[0].spec[f]) for f in names] for pd in packed_dev]
    id_bytes_total = sum(ops.index_bytes_of(t) for t in idx_lists[0])

    def dominant(i):
        ops.dlrm_lookup_interact(tables, idx_lists[i % n_bufs], slot_list, rows, 64, bottoms[i % n_bufs],
                                 slots["bottom_block"], a_out, operand_rows=operand)

    kern_ms = event_times(dominant, args.steps, args.warmup)

    e2e_steps = max(5, args.steps)
    e2e_ms, res = timed_e2e(ctx, pf, hbs, e2e_steps, depth)
    ref_host = cf(hbs[(e2e_steps - 1) % n_bufs]).clone()
    assert torch.equal(res, ref_host), "pipelined e2e result differs from the serial graph call"
    h2d = int(hbs[0].payload_bytes())
    d2h = int(res.numel() * res.element_size())

    elapsed_ms, e2e_ms, kern_ms = ctx.max_over_ranks(elapsed_ms, e2e_ms, kern_ms)
    launches = ctx.sum_over_ranks(launches)
    peak, peak_src = measured_peaks()
    fused_b, _ = dlrm_bytes_per_sample(id_bytes_total=id_bytes_total)
    achieved = fused_b * B / (kern_ms * 1e-3) / 1e9
    traffic = ncu_traffic_bytes(ROOT / NCU_FUSED_SUMMARY) if B == 65536 else None
    line = {
        "metric": "DLRM fwd samples/sec (Criteo shape, batch 65536/GPU)",
        "value": world * B * args.steps / (elapsed_ms * 1e-3),
        "unit": "samples/s",
        "n_gpus": world,
        "steps": args.steps,
        "warmup": args.warmup,
        "ms_per_step": elapsed_ms / args.steps,
        "higher_is_better": True,
        "scaling": "weak",
        "vs_baseline": None,
        "dtype": "fp32 I/O; GEMM-shaped work as split-bf16 x3 (hi*hi + hi*lo + lo*hi, fp32 accumulate, |err| ~ 2^-16)",
        "data": "synthetic (uniform indices over bundled Criteo cardinalities; hash-initialised tables, random-init MLPs)",
        "config": {
            "workload": "mm.DLRMModel Criteo-shape (26 cat, 13 dense, emb_dim 64), bottom [128,64], top [128,64,32]",
            "batch_per_gpu": B, "global_batch": B * world,
            "index_dtype": f"packed per table (8 x u8, 10 x u16, 8 x u24 = {id_bytes_total} B/sample; Model.id_bytes())",
            "table_rows": 45621194,
            "table_gb": 11.68,
            "table_mirror": ("split-bf16 copy of every table (ops.split_rows, +11.68 GB): the lookup+interaction kernel loads MMA "
                             "fragments with ldmatrix instead of splitting fp32 rows per sample" if operand else "off (MM_TABLE_MIRROR=0)"),
            "parallelism": f"replicas x{world} (no data-path collective)",
            "l2": f"inputs larger than L2: 11.7 GB of tables, {n_bufs} rotating input batches, no flush",
            "runtime": f"CUDA graph replay, {depth} graph instances on {depth} streams (model.pipeline): independent steps overlap; "
                       "input refresh = one D2D copy of the packed batch per step",
            "ms_per_step_single_stream": serial_ms,
            "dense_engine": mm.dense_engine(),
        },
        "clocks": clocks,
        "e2e": {"value": world * B * e2e_steps / (e2e_ms * 1e-3), "unit": "samples/s",
                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": e2e_steps,
                "h2d_gbs_per_gpu": h2d * e2e_steps / (e2e_ms * 1e-3) / 1e9},
        "gpu_launches": launches,
        "roofline": {"bound": "hbm", "kernel": "interact_v2_kernel<lookup-fused> (mm_dlrm_lookup_interact)",
                     "timing": "CUDA events around each of K back-to-back launches on the same rotating inputs (graph nodes cannot be bracketed)",
                     "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "peak_source": peak_src, "algorithmic_bytes_per_launch": fused_b * B,
                     "kernel_ms": kern_ms,
                     "traffic": traffic,
                     "dram_frac": None if traffic is None else traffic / (kern_ms * 1e-3) / 1e9 / peak,
                     "traffic_source": f"{NCU_FUSED_SUMMARY} (ncu --set full of this round's kernel, one launch, B=65536; the 19 "
                                       "small tables are L2-resident, so DRAM traffic < algorithmic bytes)"},
    }
    return line, model, hosts


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="all", choices=["all", "dlrm", "dlrm-sharded", "twotower", "dcn", "dlrm-train"])
    ap.add_argument("--batch", type=int, default=None)
    ap.add_argument("--cpu-sample", type=int, default=None, help="samples per CPU pass (default: the full batch)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--pipeline-depth", type=int, default=3,
                    help="graph instances / streams of model.pipeline (3: one more pinned H2D in flight than 2)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what each timed path computed in its last timed step as DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.warmup < 3:
        args.warmup = 3

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    import torch

    import models_b200 as mm
    from models_b200 import datasets, ops

    cores = usable_cores()

    # ------------------------------------------------------------------ reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return 0
        return reference_arm(args, mm, datasets, cores)

    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device: the B200 hot path has no CPU fallback"}))
        return 1
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    import torch.distributed as dist

    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    ctx = Ctx(args, mm, datasets, ops, dev, rank, local_rank, world)

    def finish(line):
        if ctx.dumping:
            write_dumps(args.dump_outputs, ctx.dumps)
        if rank == 0:
            print(json.dumps(line))
        if dist.is_initialized():
            dist.destroy_process_group()
        return 0

    if args.workload == "dlrm-sharded":
        rec = sharded_record(ctx)
        rec.update({"n_gpus": world, "steps": args.steps, "warmup": args.warmup, "higher_is_better": True, "scaling": "weak",
                    "vs_baseline": None, "unit": "samples/s"})
        return finish(rec)
    if args.workload == "dlrm-train":
        rec = train_record(ctx)
        rec.update({"n_gpus": world, "steps": args.steps, "warmup": args.warmup, "higher_is_better": True, "scaling": "weak",
                    "vs_baseline": None})
        return finish(rec)
    if args.workload in ("twotower", "dcn"):
        rec = secondary_record(ctx, args.workload)
        rec.update({"n_gpus": world, "steps": args.steps, "warmup": args.warmup, "higher_is_better": True, "scaling": "weak",
                    "vs_baseline": None})
        return finish(rec)

    line, model, hosts = dlrm_record(ctx)
    if world == 1 and not args.no_cpu_baseline and rank == 0:
        try:
            line["cpu_baseline"] = time_cpu_baseline(model, hosts[0], min(args.cpu_sample or 16384, args.batch or 65536), cores)
        except Exception as e:  # the baseline must never take the bench line down
            line["cpu_baseline"] = {"error": f"{type(e).__name__}: {e}"}
    del model, hosts
    free_device_memory()
    if args.workload == "all":
        line["secondary"] = {}
        for kind in ("twotower", "dcn"):
            try:
                line["secondary"][kind] = secondary_record(ctx, kind)
            except Exception as e:  # a secondary record must never take the headline down
                line["secondary"][kind] = {"error": f"{type(e).__name__}: {e}"}
            free_device_memory()
        try:
            line["secondary"]["dlrm_train"] = train_record(ctx)
        except Exception as e:
            line["secondary"]["dlrm_train"] = {"error": f"{type(e).__name__}: {e}"}
        free_device_memory()
        if world > 1:
            try:
                line["sharded"] = sharded_record(ctx)
            except Exception as e:
                line["sharded"] = {"error": f"{type(e).__name__}: {e}"}
            free_device_memory()
    return finish(line)


def free_device_memory():
    import gc

    import torch

    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


def usable_cores() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def pick_threads(run, cores, candidates=None):
    """The CPU leg should use 'all the host threads it can use' — but more OpenMP threads than the
    small per-op work can feed makes PyTorch-CPU slower, not faster (128 threads: 4.7 s per 16 384-sample
    pass vs 37 ms at 8).  Time one pass at a few thread counts and keep the fastest."""
    import torch

    best, best_t = 1, float("inf")
    for n in sorted(candidates or {cores, min(cores, 64), min(cores, 32), min(cores, 16), min(cores, 8)}, reverse=True):
        torch.set_num_threads(n)
        run()
        t0 = time.perf_counter()
        run()
        dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = n, dt
    torch.set_num_threads(best)
    return best



# ---------------------------------------------------------------------------------------------
# configs[3]: row-sharded tables (N > 1)
# ---------------------------------------------------------------------------------------------
def sharded_record(ctx):
    """BASELINE config 4: Criteo-TB-shape tables (204 M rows x 64 fp32 = 52 GB) row-sharded over the ranks (row r on
    rank r % world), batch 65 536 per GPU, data-parallel MLPs.  The lookup is part of the interaction kernel: rows
    owned by other ranks are read over NVLink peer memory straight into shared memory (no exchange step, no barrier),
    so the step is graph-captured like the replicated one.  Three placements are reported: tables from 65 536 rows up
    sharded (shard_model's default), from 1 000 rows up, and every table sharded.  Parity: the sharded logits must be bit-identical to
    the unsharded model's on the same batch, on every rank.  The staged protocol of round 1 (NCCL all-gather of the
    ids + owner-computes push + symmetric-memory barriers, eager) is timed beside it as the baseline."""
    import torch
    import torch.distributed as dist

    args, mm, datasets, ops, dev, world, rank = ctx.args, ctx.mm, ctx.datasets, ctx.ops, ctx.dev, ctx.world, ctx.rank
    if not dist.is_initialized():
        dist.init_process_group("nccl", init_method="tcp://127.0.0.1:29577", rank=0, world_size=1, device_id=dev)
    B = args.batch or 65536
    steps = args.steps
    schema = datasets.criteo_tb_schema()
    rows_total = sum(datasets.CRITEO_TB_ROWS)

    def make(shard_below=None):
        mm.set_seed(4)
        m = mm.DLRMModel(schema, embedding_dim=64, bottom_block=mm.MLPBlock([128, 64]), top_block=mm.MLPBlock([128, 64, 32]),
                         embedding_options=mm.EmbeddingOptions(embeddings_initializers={"hash_seed": 4321}))
        if shard_below is not None:
            mm.shard_model(m, replicate_below_rows=shard_below)
        m.build(dev)
        return m

    n_bufs = 3
    hosts = []
    for i in range(n_bufs):
        b, _ = datasets.split_targets(schema, datasets.generate_batch(schema, B, seed=4000 + 100 * rank + i, index_law="uniform",
                                                                      index_dtype=np.int32))
        hosts.append(b)
    devs = [{k: torch.from_numpy(v).to(dev) for k, v in h.items()} for h in hosts]

    # unsharded model of the same shape (52 GB of tables on this GPU) -> the logits every placement must reproduce
    full = make()
    want = full(devs[0]).clone()
    del full
    free_device_memory()

    rec = {
        "metric": "DLRM fwd samples/sec (Criteo-TB shape, row-sharded tables, batch 65536/GPU)",
        "data": "synthetic (uniform indices; hash-initialised shards)", "dtype": "fp32 I/O; split-bf16 x3 GEMM work",
        "config": {"workload": "mm.DLRMModel Criteo-TB-shape (MLPerf DLRM-DCNv2 capped cardinalities), tables row-sharded "
                               "(row r on rank r % world at local row r / world), MLPs data-parallel",
                   "batch_per_gpu": B, "global_batch": B * world, "table_rows": rows_total, "table_gb": rows_total * 256 / 1e9,
                   "parallelism": f"tables row-sharded x{world}, MLPs dp{world}",
                   "exchange": "none as a separate step: mm_dlrm_lookup_interact reads remote rows over NVLink peer memory "
                               "(cp.async from the owner's shard into the consuming SM's shared memory)",
                   "runtime": f"CUDA graph replay, {args.pipeline_depth} graph instances (no collective, no barrier in the graph)"},
        "placements": {},
    }
    link_ref = 770.0  # GB/s per direction per GPU: measured peer copy (B200_PROFILING.md); nominal 900
    for label, below in (("sharded_from_65536_rows", 65536), ("sharded_from_1000_rows", 1000), ("all_tables_sharded", 0)):
        model = make(below)
        se = model.body.sharded
        got = model(devs[0])
        ok = int(torch.equal(got, want))
        flag = torch.tensor([ok], device=dev)
        if world > 1:
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        widths = model.id_bytes()
        hbs = [mm.HostBatch.like(h, model.input_columns(), id_bytes=widths) for h in hosts]
        packed_dev = [hb.buffer.to(dev) for hb in hbs]
        cf = model.compile(hbs[0])
        cf.load_device(packed_dev[0])
        graph_ok = int(torch.equal(cf.replay(), want))
        pf = model.pipeline(hbs[0], depth=args.pipeline_depth)
        elapsed_ms, clocks = timed_replay(ctx, pf, packed_dev, steps, args.warmup)
        ctx.dump(f"sharded_{label}_predictions", last_output(pf))
        serial_ms = timed_serial(cf, packed_dev, steps)
        # the fused lookup + interaction kernel alone
        body = model.body
        operand = body.use_operand_rows()
        bottoms = [body.bottom_forward(d) for d in devs]
        bottoms_k = [body.bottom_forward(d, operand_out=True) for d in devs] if operand else bottoms
        slots = body.slots()
        k_out = torch.empty((B, 2 * ops.tc_padded_k(body.output_width_before_top())), dtype=torch.bfloat16, device=dev)
        kern_ms = event_times(lambda i: se.lookup_interact(devs[i % n_bufs], slots, bottoms_k[i % n_bufs], k_out, operand_rows=operand),
                              max(5, steps // 2))
        e2e_steps = max(5, min(steps, 20))
        e2e_ms, _ = timed_e2e(ctx, pf, hbs, e2e_steps, args.pipeline_depth)
        # exact NVLink payload of this rank's batch 0: rows whose owner is another rank
        remote = 0
        n_sharded = 0
        for f in se.feature_names:
            name = body.embeddings.feature_to_table[f].table_name
            if se.is_sharded(name):
                n_sharded += 1
                remote += int((hosts[0][f].astype(np.int64) % world != rank).sum())
        remote_bytes = remote * 256
        elapsed_ms, serial_ms, kern_ms, e2e_ms, remote_b = ctx.max_over_ranks(elapsed_ms, serial_ms, kern_ms, e2e_ms, remote_bytes)
        rec["placements"][label] = {
            "replicate_below_rows": below, "tables_sharded": n_sharded, "tables_replicated": 26 - n_sharded,
            "shard_gb_per_gpu": float(se.arena.numel() * 4 / 1e9) if se.arena is not None else 0.0,
            "table_mirror": bool(operand),
            "parity": "bit-exact vs the unsharded model on every rank" if int(flag.item()) == 1 else "MISMATCH",
            "graph_replay_parity": bool(graph_ok),
            "value": world * B * steps / (elapsed_ms * 1e-3), "unit": "samples/s", "ms_per_step": elapsed_ms / steps,
            "ms_per_step_single_stream": serial_ms,
            "lookup_interact_kernel_ms": kern_ms,
            "nvlink_bytes_in_per_gpu_per_step": remote_b,
            "nvlink_gbs_per_gpu_kernel": remote_b / (kern_ms * 1e-3) / 1e9,
            "nvlink_gbs_per_gpu_step": remote_b / (elapsed_ms / steps * 1e-3) / 1e9,
            "nvlink_ref_gbs": link_ref, "nvlink_frac_kernel": remote_b / (kern_ms * 1e-3) / 1e9 / link_ref,
            "e2e": {"value": world * B * e2e_steps / (e2e_ms * 1e-3), "unit": "samples/s",
                    "h2d_bytes_per_step": int(hbs[0].payload_bytes()), "d2h_bytes_per_step": B * 4},
            "gpu_launches": ctx.sum_over_ranks(cf.launches_per_replay * steps), "clocks": clocks,
        }
        if world > 1:
            # NCCL baseline on the same shards: ids all-gather + local gather + ONE variable-size all-to-all of the vectors
            # (split sizes read back on the host) + scatter + interaction from the stack — torch ops + torch.distributed
            from models_b200.sharded import lookup_stack_nccl

            F_n = len(slots)
            out_n = torch.empty((B, 2 * ops.tc_padded_k(body.output_width_before_top())), dtype=torch.bfloat16, device=dev)

            def nccl_step(i):
                d = devs[i % n_bufs]
                stack = lookup_stack_nccl(se, d, slots, F_n)
                ops.concat_columns([bottoms[i % n_bufs]], stack, [slots["bottom_block"] * 64])
                ops.dot_interaction(stack.view(B, F_n, 64), out_n, prefix=bottoms[i % n_bufs])

            for i in range(2):
                nccl_step(i)
            ctx.barrier()
            n0_, n1_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            n_nc = 5
            n0_.record()
            for i in range(n_nc):
                nccl_step(i)
            n1_.record()
            ctx.barrier()
            (nc_ms,) = ctx.max_over_ranks(n0_.elapsed_time(n1_) / n_nc)
            rec["placements"][label]["nccl_all_to_all_ms"] = nc_ms
            rec["placements"][label]["nccl_all_to_all"] = ("baseline: NCCL all-gather of ids + torch gather + one variable-size NCCL all_to_all_single of "
                                                           "the rows + scatter + interaction from the stack (eager torch / torch.distributed; lookup + "
                                                           "interaction only, compare with lookup_interact_kernel_ms)")
        if below == 0 and world > 1:
            # staged baseline on the same shards: ids all-gathered by NCCL, owner-computes push into the destination
            # rank's (B,F,D) stack, barriers, interaction from the stack — eager, as in round 1
            F = len(slots)
            out = torch.empty((B, 2 * ops.tc_padded_k(body.output_width_before_top())), dtype=torch.bfloat16, device=dev)

            def staged(i):
                d = devs[i % n_bufs]
                stack = se.lookup_stack(d, slots, F)
                ops.concat_columns([bottoms[i % n_bufs]], stack, [slots["bottom_block"] * 64])
                ops.dot_interaction(stack.view(B, F, 64), out, prefix=bottoms[i % n_bufs])

            for i in range(3):
                staged(i)
            ctx.barrier()
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            n_st = max(5, min(steps, 10))
            t0.record()
            for i in range(n_st):
                staged(i)
            t1.record()
            ctx.barrier()
            (st_ms,) = ctx.max_over_ranks(t0.elapsed_time(t1) / n_st)
            rec["placements"][label]["staged_protocol_ms"] = st_ms
            rec["placements"][label]["staged_protocol"] = ("NCCL all-gather of ids + mm_shard_gather_push + symmetric-memory "
                                                           "barriers + interaction from the stack (eager; same shards)")
        del cf, pf, model, se, body, bottoms
        free_device_memory()
    best = rec["placements"]["sharded_from_65536_rows"]  # shard_model's default placement
    rec["value"], rec["ms_per_step"] = best["value"], best["ms_per_step"]
    rec["headline_placement"] = ("sharded_from_65536_rows: the 8 tables with >= 65 536 rows (99.9 % of the rows, 52.2 GB) row-sharded, "
                                 "the 18 small ones (55 MB) replicated; `all_tables_sharded` is reported beside it — tables of 3-155 rows "
                                 "then serialise every GPU on a few cache lines of one owner")
    return rec


# ---------------------------------------------------------------------------------------------
# configs[2] and configs[4]: two-tower and DCN-v2 (replicas under torchrun)
# ---------------------------------------------------------------------------------------------
def train_record(ctx):
    """SURVEY §8(f)-4: ONE TRAINING STEP of the headline DLRM (forward with saved activations + binary cross-entropy +
    backward + Adagrad update of every variable, embedding rows included) per batch of 65 536 samples — the reference's
    `model.fit` inner loop (models/base.py:1121-1177).  Replicas under torchrun (each rank trains its own copy: no
    gradient exchange is timed here).  `value`: CUDA-graph replay over rotating device-resident batches (a D2D refresh of
    the static input buffer is part of the step); `e2e`: packed pinned host batch (ids + dense + labels) -> one H2D ->
    graph -> D2H of the loss."""
    import torch

    args, mm, datasets, ops, dev, world = ctx.args, ctx.mm, ctx.datasets, ctx.ops, ctx.dev, ctx.world
    B = args.batch if (args.batch and args.workload == "dlrm-train") else 65536
    steps = args.steps
    mm.set_seed(1)
    schema, model = build_dlrm(mm, datasets)
    model.build(dev)
    model.compile(optimizer=mm.Adagrad(0.01))
    n_bufs = 4
    hosts = []
    for i in range(n_bufs):
        hosts.append(datasets.generate_batch(schema, B, seed=4321 + i + 1000 * ctx.rank, index_law="uniform", index_dtype=np.int32))
    label = schema.select_by_tag(mm.Tags.TARGET).column_names[0]
    names = model.input_columns() + [label]
    hbs = [mm.HostBatch.like(h, names, id_bytes=model.id_bytes()) for h in hosts]
    packed_dev = [hb.buffer.to(dev) for hb in hbs]
    from models_b200.graph import _view

    static = torch.empty(hbs[0].buffer.numel(), dtype=torch.uint8, device=dev)
    static.copy_(packed_dev[0])
    views = {name: _view(static, hbs[0].offsets[name], shp, dt) for name, (shp, dt) in hbs[0].spec.items()}
    inputs = {k: v for k, v in views.items() if k != label}
    tr = model.trainer(B)
    # per-phase device times of the eager step (CUDA events around each phase)
    phase = {}
    for name, fn in (("forward_backward", lambda i: tr.forward_backward(inputs, views[label])), ("update", lambda i: tr.apply_gradients())):
        phase[name + "_ms"] = event_times(fn, 10)
    n0 = ops.launch_count()
    tr.capture(inputs, views[label], clone=False)

    def run(n):
        for i in range(n):
            static.copy_(packed_dev[i % n_bufs], non_blocking=True)
            tr.replay()

    run(args.warmup)
    ctx.barrier()
    sampler = ClockSampler(ctx.local_rank)
    sampler.start()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    run(steps)
    t1.record()
    ctx.barrier()
    clocks = sampler.stop()
    ms = t0.elapsed_time(t1)
    loss_end = float(tr.loss.item())
    if ctx.dumping:
        # the loss of the last timed step and the variables it left: every Dense variable, and the embedding rows of a
        # seeded sample of that step's samples (rows it updated)
        ctx.dump("dlrm_train_loss", tr.loss)
        ctx.dump("dlrm_train_dense_variables", tr.arena.w)
        last = hosts[(steps - 1) % n_bufs]
        pos = np.sort(np.random.default_rng(DUMP_SEED).choice(B, size=min(256, B), replace=False))
        ctx.dump("dlrm_train_embedding_rows_sample",
                 torch.stack([t.table[torch.from_numpy(last[f].reshape(-1)[pos].astype(np.int64)).to(dev)] for f, t in zip(tr.feats, tr.tables)]))
    # e2e: pinned host batch -> H2D -> graph -> loss to the host
    loss_host = torch.zeros(1, dtype=torch.float32, pin_memory=True)

    def e2e(n):
        for i in range(n):
            static.copy_(hbs[i % n_bufs].buffer, non_blocking=True)
            tr.replay()
            loss_host.copy_(tr.loss, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    e2e(3)
    ctx.barrier()
    w0 = time.perf_counter()
    e2e(steps)
    e2e_ms = (time.perf_counter() - w0) * 1e3
    ctx.barrier()
    ms_max, e2e_max = ctx.max_over_ranks(ms, e2e_ms)
    rec = {
        "metric": "DLRM TRAIN samples/sec (Criteo shape, batch 65536/GPU, forward + BCE + backward + Adagrad)",
        "value": B * world * steps / (ms_max / 1e3), "unit": "samples/s", "ms_per_step": ms_max / steps,
        "dtype": "fp32 variables and I/O; split-bf16 x3 GEMM work", "data": "synthetic (uniform indices; hash-initialised tables)",
        "config": {"workload": "mm.DLRMModel Criteo-shape (26 cat, 13 dense, emb_dim 64), bottom [128,64], top [128,64,32]; "
                               "model.compile(Adagrad(0.01)); one optimizer step per batch",
                   "batch_per_gpu": B, "global_batch": B * world, "parallelism": f"replicas x{world} (no gradient exchange timed)",
                   "l2": "4 rotating input batches; tables, activations and slices exceed L2",
                   "runtime": "one CUDA graph per step (forward + backward + update), static buffers"},
        "clocks": clocks, "gpu_launches": tr.launches_per_step * steps, "launches_per_step": tr.launches_per_step,
        "eager_phase_ms": phase, "loss_after": loss_end,
        "e2e": {"value": B * world * steps / (e2e_max / 1e3), "unit": "samples/s", "h2d_bytes_per_step": int(hbs[0].buffer.numel()),
                "d2h_bytes_per_step": 4, "steps": steps},
        "fwd_only_ratio_note": "compare with the headline `value` (forward only) of the same line",
    }
    # roofline of the step's largest kernel (lookup + interaction backward), timed alone with CUDA events on this stream
    try:
        if tr.operand_rows:
            F_n = len(tr.slots)
            tabs = [t._mirror for t in tr.tables]
            rows = [t.table.shape[0] for t in tr.tables]
            tslots = [tr.slots[f] for f in tr.feats]
            idx = tr._indices(inputs)
            dA_view = tr.dA[:, :tr.OW]
            sl = [tr.slices[t] for t in range(len(tabs))]
            k_ms = event_times(lambda i: ops.dlrm_interact_backward(tabs, idx, tslots, rows, tr.D, tr.h_split[-1], tr.slots["bottom_block"], dA_view,
                                                                     sl, tr.dh[-1], mask_bottom=True, operand_rows=True), 20)
            id_bytes = sum(ops.index_bytes_of(i) for i in idx)
            T = len(tabs)
            per_sample = (T + 1) * 256 + tr.OW * 4 + T * 256 + 256 + id_bytes  # rows + bottom in, dA in, slices + d_bottom out, ids
            peak, peak_src = measured_peaks()
            ach = per_sample * B / (k_ms * 1e-3) / 1e9
            rec["roofline"] = {"bound": "hbm", "kernel": "interact_bwd_ps_kernel (mm_dlrm_interact_backward, operand-format rows)",
                               "unit": "GB/s", "achieved": ach, "peak": peak, "peak_source": peak_src, "frac": ach / peak, "kernel_ms": k_ms,
                               "algorithmic_bytes_per_launch": per_sample * B,
                               "traffic": 749990144.0, "dram_frac": 749990144.0 / (k_ms * 1e-3) / 1e9 / peak, "traffic_source": "profiles/r02_ncu_train_kernels.txt (ncu --set full, dram read + write of one launch)",
                               "share_of_step": k_ms / (ms_max / steps)}
    except Exception as e:  # evidence, never fatal
        rec["roofline"] = {"error": f"{type(e).__name__}: {e}"}
    if world == 1 and not args.no_cpu_baseline and ctx.rank == 0:
        try:
            rec["cpu_baseline"] = train_cpu_baseline(model, hosts[0], label, min(args.cpu_sample or 16384, B), usable_cores())
        except Exception as e:
            rec["cpu_baseline"] = {"error": f"{type(e).__name__}: {e}"}
    del tr, model
    return rec


def train_cpu_baseline(model, host_batch, label, sample_rows, cores, budget_s=8.0):
    """The same training step on the host cores (oracle/oracle_torch.py:DLRMTrainCPU: autograd with sparse embedding
    gradients + Adagrad) on a bounded sample of the batch — a reported baseline, not a target."""
    import torch
    from oracle import oracle_torch

    torch.set_num_threads(min(cores, 32))
    body = model.body
    tables = {n: t.embeddings.cpu() for n, t in body.embeddings.tables.items()}
    f2t = {f: t.table_name for f, t in body.embeddings.feature_to_table.items()}
    layers = lambda mlp: [{"kernel": l.kernel.cpu(), "bias": l.bias.cpu(), "activation": l.activation} for l in mlp.dense_layers]
    hd = model.prediction.to_call
    cpu = oracle_torch.DLRMTrainCPU(tables, f2t, layers(body.bottom_block), layers(body.top_block),
                                    {"kernel": hd.kernel.cpu(), "bias": hd.bias.cpu(), "activation": "linear"}, lr=0.01)
    del tables
    idx = {n: torch.from_numpy(host_batch[n][:sample_rows]) for n in f2t}
    dense = {n: torch.from_numpy(host_batch[n][:sample_rows]) for n in body.continuous.features}
    y = torch.from_numpy(host_batch[label][:sample_rows])
    # 128 OpenMP threads make these small ops ~100x slower than 8-32 (see pick_threads): only the small counts are tried
    cores = pick_threads(lambda: cpu.step(idx, dense, y), cores, candidates={min(cores, 32), min(cores, 16), min(cores, 8)})
    t0 = time.perf_counter()
    n = 0
    while True:
        cpu.step(idx, dense, y)
        n += 1
        dt = time.perf_counter() - t0
        if dt > budget_s or n >= 20:
            break
    return {"value": sample_rows * n / dt, "unit": "samples/s", "cores": cores, "kind": "port",
            "sample": f"{n} training steps on {sample_rows} samples of the same batch (PyTorch-CPU: autograd with sparse embedding "
                      "gradients + Adagrad; the reference's TF-CPU train_step is not runnable here)"}


def secondary_record(ctx, kind):
    """BASELINE configs[2] (two-tower, 10 M-item catalog, in-batch negatives, B = 16 384) and configs[4]
    (DCN-v2, depth 3, deep [256,128], B = 65 536): same timing protocol as the DLRM arm (graph replay on two
    streams for `value`, packed pinned host batches for `e2e`, CUDA events, clocks), replicas under torchrun."""
    import torch

    args, mm, datasets, ops, dev, world, rank = ctx.args, ctx.mm, ctx.datasets, ctx.ops, ctx.dev, ctx.world, ctx.rank
    steps = args.steps
    mm.set_seed(1)
    if kind == "twotower":
        B = args.batch if (args.batch and args.workload == "twotower") else 16384
        schema = datasets.retrieval_10m_schema()
        model = mm.TwoTowerModel(schema, query_tower=mm.MLPBlock([256, 128]),
                                 embedding_options=mm.EmbeddingOptions(embeddings_initializers={"hash_seed": 5}))
        call_kwargs = {"training": True}
        law = "zipf"
        label = "mm.TwoTowerModel 10M-item catalog, towers [256,128], in-batch sampled softmax (train-mode forward: (B, 1+B) logits)"
        metric = "TwoTower fwd samples/sec (10M-item catalog, in-batch negatives, batch 16384/GPU)"
    else:
        B = args.batch if (args.batch and args.workload == "dcn") else 65536
        schema = datasets.criteo_schema()
        model = mm.DCNModel(schema, depth=3, deep_block=mm.MLPBlock([256, 128]), embeddings_initializer={"hash_seed": 99})
        call_kwargs = {}
        law = "uniform"
        label = "mm.DCNModel (DCN-v2) cross depth 3 (d = 1037) + MLP[256,128]"
        metric = "DCN-v2 fwd samples/sec (Criteo shape, batch 65536/GPU)"
    n_bufs = 4
    hosts = []
    for i in range(n_bufs):
        b = datasets.generate_batch(schema, B, seed=1234 + 1000 * rank + i, index_law=law, index_dtype=np.int32)
        hosts.append(datasets.split_targets(schema, b)[0])
    model.build(dev)
    hbs = [mm.HostBatch.like(h, model.input_columns()) for h in hosts]
    packed_dev = [hb.buffer.to(dev) for hb in hbs]
    cf = model.compile(hbs[0], **call_kwargs)
    pf = model.pipeline(hbs[0], depth=2, **call_kwargs)
    elapsed_ms, clocks = timed_replay(ctx, pf, packed_dev, steps, args.warmup)
    if kind == "twotower":  # (B, 1+B) logits: 1 GB at B = 16 384
        if ctx.dumping:
            ctx.dump("twotower_logits_row_sample", sample_rows(last_output(pf)))
    else:
        ctx.dump("dcn_predictions", last_output(pf))
    serial_ms = timed_serial(cf, packed_dev, steps)

    # dominant kernel, one launch per CUDA-event pair
    if kind == "twotower":
        D = 128
        q = torch.randn((B, D), device=dev)
        it = torch.randn((B, D), device=dev)
        ids = torch.from_numpy(hosts[0][schema.select_by_tag(mm.Tags.ITEM_ID).first.name].astype(np.int64).reshape(-1)).to(dev)
        qs, its = ops.split_rows(q), ops.split_rows(it)
        logits = torch.empty((B, B + 4), dtype=torch.float32, device=dev)[:, 3:4 + B]  # (B, 1+B); negatives 16-byte aligned
        from models_b200 import _cabi

        lib = _cabi.load()

        def dominant(i):
            _cabi.check(lib.mm_inbatch_scores_tc(qs.data_ptr(), its.data_ptr(), B, B, D, ids.data_ptr(), ids.data_ptr(),
                                                 _cabi.MM_I64, 1, -655.04, None, 1.0, logits.data_ptr(), logits.stride(0),
                                                 torch.cuda.current_stream().cuda_stream), "mm_inbatch_scores_tc")

        algo = float(B) * (B + 1) * 4 + 2.0 * B * D * 4
        roof = {"bound": "hbm", "kernel": "dense_tc_kernel<scorer epilogue> (mm_inbatch_scores_tc)", "unit": "GB/s"}
    else:
        d = 1037
        x = torch.randn((B, d), device=dev)
        W = torch.randn((d, d), device=dev) * 0.03
        a, w = ops.split_rows(x), ops.split_weights(W)
        o = torch.empty((B, d), dtype=torch.float32, device=dev)
        nxt = torch.zeros((B, 2 * ops.tc_padded_k(d)), dtype=torch.bfloat16, device=dev)

        def dominant(i):
            ops.dense_tc(a, d, w, d, None, "linear", passes=3, out_f32=o, out_split=nxt, x0=x, xres=x)

        algo = 2.0 * B * d * d
        roof = {"bound": "tensor", "kernel": "dense_tc_kernel<cross epilogue> (mm_dense_tc, one of the 3 cross layers)",
                "unit": "TFLOP/s", "note": "algorithmic fp32 FLOPs; 3 bf16 passes are issued for fp32 parity (x3 tensor work)"}
    kern_ms = event_times(dominant, max(5, steps // 2))

    # e2e: pinned packed host batch in, predictions (logits for the two-tower) out, pipelined
    e2e_steps = max(5, min(steps, 20))
    e2e_ms, res = timed_e2e(ctx, pf, hbs, e2e_steps, 2)
    elapsed_ms, e2e_ms, kern_ms = ctx.max_over_ranks(elapsed_ms, e2e_ms, kern_ms)
    hbm, hbm_src = measured_peaks()
    tf_peak = None
    pth = ROOT / "MEASURED_PEAKS.json"
    if pth.exists():
        tf_peak = json.loads(pth.read_text()).get("bf16_tflops")
    if roof["bound"] == "hbm":
        achieved, peak, src = algo / (kern_ms * 1e-3) / 1e9, hbm, hbm_src
    else:
        achieved, peak, src = algo / (kern_ms * 1e-3) / 1e12, tf_peak or 1590.0, "measured (MEASURED_PEAKS.json)" if tf_peak else "fallback (B200_PROFILING.md)"
    roof.update({"achieved": achieved, "peak": peak, "frac": achieved / peak, "peak_source": src, "kernel_ms": kern_ms,
                 "algorithmic_per_launch": algo, "traffic": None})
    rec = {
        "metric": metric, "value": world * B * steps / (elapsed_ms * 1e-3), "unit": "samples/s",
        "ms_per_step": elapsed_ms / steps,
        "dtype": "fp32 I/O; split-bf16 x3 GEMM work",
        "data": f"synthetic ({law} indices; hash-initialised tables, random-init towers)",
        "config": {"workload": label, "batch_per_gpu": B, "global_batch": B * world,
                   "parallelism": f"replicas x{world} (no data-path collective)",
                   "l2": f"{n_bufs} rotating input batches; tables and the (B,1+B) logits exceed L2",
                   "runtime": "CUDA graph replay, 2 graph instances on 2 streams", "ms_per_step_single_stream": serial_ms},
        "clocks": clocks,
        "e2e": {"value": world * B * e2e_steps / (e2e_ms * 1e-3), "unit": "samples/s",
                "h2d_bytes_per_step": int(hbs[0].payload_bytes()), "d2h_bytes_per_step": int(res.numel() * res.element_size()),
                "steps": e2e_steps},
        "gpu_launches": cf.launches_per_replay * steps * world, "roofline": roof,
    }
    if kind == "twotower":
        # the same step with the soft-max cross-entropy folded into the scorer's epilogue (model(..., fused_loss=True)):
        # outputs (B,3) [max, log-sum-exp, positive logit] instead of the (B, 1+B) logits — nothing of size B^2 is written
        try:
            kw = dict(call_kwargs, fused_loss=True)
            cf2 = model.compile(hbs[0], **kw)
            pf2 = model.pipeline(hbs[0], depth=2, **kw)
            el2, _ = timed_replay(ctx, pf2, packed_dev, steps, args.warmup)
            ctx.dump("twotower_fused_loss_stats", last_output(pf2))
            ser2 = timed_serial(cf2, packed_dev, steps)
            e2e2, res2 = timed_e2e(ctx, pf2, hbs, e2e_steps, 2)
            el2, e2e2 = ctx.max_over_ranks(el2, e2e2)
            rec["fused_loss"] = {
                "what": "model(batch, training=True, fused_loss=True): in-batch soft-max CE statistics from the GEMM epilogue "
                        "(mm_inbatch_softmax_ce), no (B, 1+B) logits",
                "value": world * B * steps / (el2 * 1e-3), "unit": "samples/s", "ms_per_step": el2 / steps,
                "ms_per_step_single_stream": ser2,
                "e2e": {"value": world * B * e2e_steps / (e2e2 * 1e-3), "unit": "samples/s",
                        "h2d_bytes_per_step": int(hbs[0].payload_bytes()), "d2h_bytes_per_step": int(res2.numel() * res2.element_size())},
                "gpu_launches": cf2.launches_per_replay * steps * world}
            del cf2, pf2
        except Exception as e:
            rec["fused_loss"] = {"error": f"{type(e).__name__}: {e}"}
    del cf, pf, model
    return rec


def time_cpu_baseline(model, feats_host, sample_rows, cores, budget_s=20.0):
    run = cpu_baseline_dlrm(model, feats_host, sample_rows, cores)
    cores = pick_threads(run, cores)
    run()  # warm-up
    t0 = time.perf_counter()
    n = 0
    while True:
        run()
        n += 1
        dt = time.perf_counter() - t0
        if dt > budget_s or n >= 50:
            break
    return {"value": sample_rows * n / dt, "unit": "samples/s", "cores": cores, "kind": "port",
            "sample": f"{n} passes over {sample_rows} samples of the same batch, same tables/weights on the host; "
                      "PyTorch-CPU restatement of the reference TF op sequence (TensorFlow not installable)"}


def reference_arm(args, mm, datasets, cores):
    """`--impl reference`: the CPU restatement of the reference path on this box's host cores.
    Tables are generated on the host by the same hash initialiser (no GPU needed)."""
    import torch
    from oracle import oracle, oracle_torch

    torch.set_num_threads(cores)
    B = args.batch or 65536
    sample = min(args.cpu_sample or B, B)  # default: the SAME 65 536-sample step as our arm (same_config)
    schema = datasets.criteo_schema()
    rng = np.random.default_rng(4321)
    cat = schema.select_by_tag(mm.Tags.CATEGORICAL)
    # host tables: random rows are touched uniformly, so the table content is irrelevant to the
    # timing; sizes (rows x 64 fp32) are the real ones, filled by a cheap seeded generator
    gen = torch.Generator().manual_seed(4321)
    tables = {}
    for c in cat:
        rows = c.int_domain.max + 1
        t = torch.empty((rows, 64), dtype=torch.float32)
        t.uniform_(-0.05, 0.05, generator=gen)
        tables[c.name] = t
    f2t = {c.name: c.name for c in cat}

    def glorot(i, o):
        lim = np.sqrt(6.0 / (i + o))
        return torch.from_numpy(rng.uniform(-lim, lim, (i, o)).astype(np.float32))

    def layers(dims, width, last_act="relu"):
        out = []
        for d in dims:
            out.append({"kernel": glorot(width, d), "bias": torch.zeros(d), "activation": "relu"})
            width = d
        return out

    bottom, top = layers([128, 64], 13), layers([128, 64, 32], 64 + 351)
    head = {"kernel": glorot(32, 1), "bias": torch.zeros(1), "activation": "sigmoid"}
    batch = datasets.generate_batch(schema, sample, seed=1234, index_law="uniform", index_dtype=np.int32)
    feats, _ = datasets.split_targets(schema, batch)
    idx = {n: torch.from_numpy(feats[n]) for n in f2t}
    dense = {c.name: torch.from_numpy(feats[c.name]) for c in schema.select_by_tag(mm.Tags.CONTINUOUS)}

    def run():
        return oracle_torch.dlrm_forward(idx, dense, tables, f2t, bottom, top, head)

    cores = pick_threads(run, cores)
    for _ in range(max(1, min(args.warmup, 3))):
        run()
    done = args.steps
    t0 = time.perf_counter()
    for _ in range(done):
        out = run()
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        write_dumps(args.dump_outputs, {"reference_predictions": out.float().numpy()})
    value = sample * done / dt
    line = {
        "impl": "reference",
        "metric": "DLRM fwd samples/sec (Criteo shape, batch 65536/GPU)",
        "value": value, "unit": "samples/s", "n_gpus": args.gpus, "steps": done, "warmup": args.warmup,
        "ms_per_step": dt / done * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "fp32", "data": "synthetic (uniform indices over bundled Criteo cardinalities)",
        "config": {"workload": "mm.DLRMModel Criteo-shape (26 cat, 13 dense, emb_dim 64), bottom [128,64], top [128,64,32]",
                   "batch_per_gpu": sample, "global_batch": sample, "batch_per_step": sample,
                   "note": "each step = one pass of the CPU restatement over the same 65536-sample batch shape as the GPU arm"
                           if sample == B else "each step = a bounded sample of the batch"},
        "cpu_baseline": {"value": value, "unit": "samples/s", "cores": cores, "kind": "port",
                         "sample": f"{done} steps x {sample} samples; PyTorch-CPU restatement of the reference "
                                   "TF op sequence (TensorFlow/merlin-core not installable: no network)"},
        "e2e": {"value": value, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))
    return 0


if __name__ == "__main__":
    sys.exit(main())
