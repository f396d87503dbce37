#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native hot path (contract: see DESIGN.md section 6).

    python bench.py --gpus 1 --steps K --warmup W            # our arm
    python bench.py --impl reference --steps K --warmup W     # CPU restatement of the reference path
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
           --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR   # also write the last timed step's outputs

Metric (BASELINE.json): examples/sec (fwd+bwd) DeepFM batch=65536.  Workload at N=1 = config C2:
26 categorical slots x 1M-row tables, D=16, batch 65536, DNN [256,32]->1, synthetic uniform ids,
one step = forward + backward + SGD update (row-sparse on the tables, dense on the tower).
A step never skips work: every kernel of fwd, bwd and the optimizer runs inside the timed region.
Prints ONE JSON line (rank 0).
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
sys.path.insert(0, ROOT)

METRIC = "examples/sec (fwd+bwd) DeepFM batch=65536"
C2 = dict(slots=26, rows=1_000_000, dim=16, batch=65536, dnn=[256, 32])
# BASELINE config C5 (opt-in, --workload c5): 100M total rows over 26 tables, D=128, GLOBAL batch 65536 split over
# the ranks (strong scaling in the batch), rows sharded row-wise with the fused NVLink peer-memory gather / update.
# The tower is not specified by BASELINE.json; [512, 256] -> 1 is this repo's choice.
C5 = dict(slots=26, rows=3_846_154, dim=128, batch=65536, dnn=[512, 256])
# --dump-outputs writes the embedding vectors of a fixed, seeded sample of table rows, this many bytes of them: the tables
# themselves are 1.7 GB at C2 and 51 GB at C5
DUMP_EMBED_BYTES = 16 << 20


def measured_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback"


class ClockSampler:
    """nvidia-smi sampler running during the timed region (B200_PROFILING.md clocks line)."""

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def __exit__(self, *a):
        if self.proc is not None:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


def run_reference(args):
    """Reference arm: the reference's CPU path (restated in torch-CPU: TensorFlow is not in this image)."""
    import torch
    from oracle.torch_cpu import DeepFMCPU
    torch.manual_seed(0)
    cores = torch.get_num_threads()
    rows = [C2["rows"]] * C2["slots"]
    B = C2["batch"]
    model = DeepFMCPU(rows, C2["dim"], C2["dnn"], seed=0)
    g = torch.Generator().manual_seed(1)
    pool = [(torch.randint(0, C2["rows"], (B, C2["slots"]), generator=g),
             torch.randint(0, 2, (B,), generator=g).float()) for _ in range(2)]
    for i in range(max(1, args.warmup)):
        model.train_step(*pool[i % 2], 0.01)
    t0 = time.perf_counter()
    for i in range(args.steps):
        model.train_step(*pool[i % 2], 0.01)
    dt = time.perf_counter() - t0
    v = B * args.steps / dt
    sample = f"{args.steps} full train steps (fwd+bwd+SGD) at B={B}, torch-CPU restatement of the reference path"
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "examples/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args.gpus),
            "cpu_baseline": {"value": v, "unit": "examples/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": "examples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
            "note": "CPU restatement of the reference path (torch-CPU), not TensorFlow: TF is not installed in this image"}
    print(json.dumps(line), flush=True)


def dump_outputs(trainer, out_dir):
    """Writes what the trainer's last step left for its caller as float32 DIR/<name>.npy: the step's loss and
    probabilities, the dense tower, the FM bias, and the embedding vectors and first-order weights of a fixed sample of
    table rows (row indices drawn with seed 0, sorted), so that two builds run with the same arguments can be compared
    array for array.  main() calls it right after the timed loop and before the end-to-end passes step the trainer again:
    that order is what makes the files hold the last timed step.

    Under --optimizer adam_rows_tf the tables lag the rows' pending Adam steps, so this first replays them in place
    (flush_optimizer, what a caller does before reading the tables; a no-op for the other optimizers).  The end-to-end
    and per-kernel passes that follow then start with no pending steps, unlike a run without --dump-outputs; the
    headline timed region is not affected."""
    import numpy as np
    import torch
    trainer.flush_optimizer()
    coll = trainer.coll
    n = min(coll.total_rows, DUMP_EMBED_BYTES // (4 * coll.dim))
    rows = np.sort(np.random.default_rng(0).choice(coll.total_rows, n, replace=False))
    rows = torch.from_numpy(rows).to(coll.weight.device)
    out = {"loss": trainer.loss, "prob": trainer.prob, "fm_bias": coll.bias,
           "embed_rows": coll.emb_view().index_select(0, rows), "linear_rows": coll.lin_view().index_select(0, rows)}
    for i, (w, b) in enumerate(zip(trainer.w, trainer.b)):
        out[f"dense{i}_kernel"] = w
        if b is not None:
            out[f"dense{i}_bias"] = b
    os.makedirs(out_dir, exist_ok=True)
    for name, t in out.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), t.detach().float().cpu().numpy())


def workload_config(n, name="c2"):
    if name == "c5":
        return {"workload": f"C5 DLRM-shape DeepFM: {C5['slots']} slots x {C5['rows']} rows (100M total), D={C5['dim']}, "
                            f"GLOBAL batch {C5['batch']} ({C5['batch'] // n} per GPU), DNN {C5['dnn']}->1, BCE, SGD",
                "global_batch": C5["batch"], "parallelism": "single GPU" if n == 1 else f"row-sharded tables x{n} + data-parallel tower",
                "l2": "inputs larger than L2: 51.2 GB of tables, id batches rotate through a pool", "ids": "uniform int64"}
    return {"workload": f"C2 DeepFM: {C2['slots']} slots x {C2['rows']} rows, D={C2['dim']}, batch {C2['batch']} per GPU, "
                        f"DNN {C2['dnn']}->1, BCE, SGD (row-sparse tables + dense tower)",
            "global_batch": C2["batch"] * n, "parallelism": "single GPU" if n == 1 else f"row-sharded tables x{n} + data-parallel tower",
            "l2": "inputs larger than L2: 3.3 GB of tables (26 M fused 128-B rows), id batches and activations rotate through a pool",
            "ids": "uniform int64"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="launch the step eagerly (for ncu launch lists)")
    ap.add_argument("--workload", default="c2", choices=["c2", "c5"],
                    help="c2 (default, the headline config; weak scaling) or c5 (100M rows x D=128, global batch 65536)")
    ap.add_argument("--ids", default="uniform", choices=["uniform", "zipf"],
                    help="synthetic id distribution: uniform (headline) or Zipf(1.05) clipped to the table (SURVEY 8d second run)")
    ap.add_argument("--tune", action="append", default=[], metavar="KNOB=VALUE",
                    help="developer knob of libdeeprec_b200.so (dr_tune_set), e.g. --tune tc_min_n=32; recorded in the line")
    ap.add_argument("--optimizer", default="sgd", choices=["sgd", "adam", "lazy_adam", "adam_rows", "adam_rows_tf"],
                    help="N=1: sgd (default, fused row-sparse SGD), adam (TF-exact dense ApplyAdam over the arena), lazy_adam "
                         "(row-sparse, two kernels), adam_rows (row-sparse Adam fused into the backward scatter)")
    ap.add_argument("--embed-fwd", default="ldg", choices=["ldg", "tma"],
                    help="N=1: forward gather through register loads (default) or staged through TMA tile::gather4 (opt-in, measured slower)")
    ap.add_argument("--fwd-chunks", type=int, default=1,
                    help="N=1: run the gather and the first tower GEMM as this many alternating launches over slices of the batch")
    ap.add_argument("--dw-first", type=int, default=0, help="N=1: enqueue the layer-0 dW GEMM before the embedding update")
    ap.add_argument("--exchange", default="p2p", choices=["p2p", "nccl"],
                    help="N>1: fused NVLink peer-memory gather/update (p2p) or NCCL all-to-all pipeline (nccl)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="N=1: after the timed steps, write what the last one computed to DIR/<name>.npy (float32): loss, "
                         "probabilities, dense tower, FM bias and a fixed seeded sample of the embedding rows")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.dump_outputs and (args.impl != "ours" or world > 1):
        ap.error("--dump-outputs needs --impl ours in a single process")

    if args.impl == "reference":
        if rank == 0:
            run_reference(args)
        return

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the hot path has no CPU fallback; use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    from deep_recommenders_b200 import _lib, feature_column as fc
    from deep_recommenders_b200.keras.models.ranking import DeepFM
    from deep_recommenders_b200.training import DeepFMTrainStep

    for kv in args.tune:
        k, v = kv.split("=")
        _lib.tune(k, int(v))
    W = C5 if args.workload == "c5" else C2
    B, S, D = (W["batch"] // world if args.workload == "c5" else W["batch"]), W["slots"], W["dim"]
    gemm_note = None
    cols = [fc.categorical_column_with_identity(f"C{i}", W["rows"]) for i in range(S)]
    if world > 1:
        from deep_recommenders_b200.sharded import ShardedDeepFMTrainStep
        exchange_note = None
        def build_sharded(exchange):
            return ShardedDeepFMTrainStep(cols, D, W["dnn"], batch_size=B, lr=0.01, seed=1, device=dev,
                                          use_graph=not args.no_graph, exchange=exchange,
                                          dw_first=bool(args.dw_first)).capture()
        try:
            trainer = build_sharded(args.exchange)
        except Exception as e:
            trainer = None
            if _lib._tc_variant == 2:       # newest GEMM core first suspect: retry the same exchange on the tc core
                gemm_note = f"tc2 unavailable ({type(e).__name__}: {e}); used tc"
                _lib.enable_tensor_core_gemm(variant=1)
                try:
                    trainer = build_sharded(args.exchange)
                except Exception as e2:
                    e = e2
            if trainer is None:             # symmetric memory unavailable on this box: NCCL all-to-all pipeline instead
                if args.exchange != "p2p":
                    raise e
                exchange_note = f"p2p unavailable ({type(e).__name__}: {e}); used nccl"
                trainer = build_sharded("nccl")
    else:
        def build_single():
            model = DeepFM([fc.indicator_column(c) for c in cols], [fc.embedding_column(c, D) for c in cols],
                           dnn_units_size=W["dnn"], seed=1, device=dev, sparse_lr=0.01)
            return DeepFMTrainStep(model, batch_size=B, lr=0.01, use_graph=not args.no_graph,
                                   optimizer=args.optimizer, embed_fwd=args.embed_fwd,
                                   fwd_chunks=args.fwd_chunks, dw_first=bool(args.dw_first)).capture()
        try:
            trainer = build_single()
        except Exception as e:      # the newest GEMM core failing to launch must not cost the measurement: say so, use tc
            if _lib._tc_variant != 2:
                raise
            gemm_note = f"tc2 unavailable ({type(e).__name__}: {e}); used tc"
            _lib.enable_tensor_core_gemm(variant=1)
            torch.cuda.empty_cache()
            trainer = build_single()

    # synthetic MovieLens-shaped batches: pool resident in HBM (value) and in pinned host memory (e2e)
    NP = 8
    gen = torch.Generator(device=dev).manual_seed(100 + rank)
    if args.ids == "zipf":      # skewed ids: rank-1 rows are hit thousands of times per batch (L2 reuse, atomic contention)
        import numpy as np
        rng = np.random.default_rng(100 + rank)
        ids_pool = [torch.from_numpy(np.minimum(rng.zipf(1.05, size=(B, S)) - 1, W["rows"] - 1).astype(np.int64)).to(dev)
                    for _ in range(NP)]
    else:
        ids_pool = [torch.randint(0, W["rows"], (B, S), device=dev, generator=gen) for _ in range(NP)]
    lab_pool = [torch.randint(0, 2, (B,), device=dev, generator=gen).float() for _ in range(NP)]
    host_ids = [t.cpu().pin_memory() for t in ids_pool]
    host_lab = [t.cpu().pin_memory() for t in lab_pool]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t)
        return ms

    # ---- device-resident timed region ------------------------------------------------------------
    for i in range(args.warmup):
        trainer.step(ids_pool[i % NP], lab_pool[i % NP])
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clk:
        barrier()
        e0.record()
        for i in range(args.steps):
            trainer.step(ids_pool[i % NP], lab_pool[i % NP])
        e1.record()
        barrier()
    ms = max_over_ranks(e0.elapsed_time(e1))
    value = B * world * args.steps / (ms * 1e-3)
    if args.dump_outputs:               # before the end-to-end passes below step the trainer again
        dump_outputs(trainer, args.dump_outputs)
    final_loss = float(trainer.loss.item())

    # ---- end-to-end: host buffers in, loss out, copies inside the timed region --------------------
    # (a) the public epoch loop `trainer.fit_host(batches)`: per step the H2D copy of the batch from pinned host memory, the
    #     step, and a D2H read of the step's loss (asynchronous, read by the host two steps later) -- the headline e2e;
    # (b) `trainer.train_step_host(...)`, which blocks the host on `loss.item()` after every step -- reported beside it.
    seq = lambda n: [(host_ids[i % NP], host_lab[i % NP]) for i in range(n)]
    trainer._staged = None
    trainer.fit_host(seq(args.warmup))
    barrier()
    e0.record()
    losses = trainer.fit_host(seq(args.steps))
    e1.record()
    barrier()
    assert len(losses) == args.steps and all(l == l for l in losses), "fit_host must return every step's loss"
    ms_e2e = max_over_ranks(e0.elapsed_time(e1))
    trainer._staged = None
    for i in range(args.warmup):
        trainer.train_step_host(host_ids[i % NP], host_lab[i % NP], host_ids[(i + 1) % NP], host_lab[(i + 1) % NP])
    trainer._staged = None
    barrier()
    e0.record()
    for i in range(args.steps):
        trainer.train_step_host(host_ids[i % NP], host_lab[i % NP], host_ids[(i + 1) % NP], host_lab[(i + 1) % NP])
    e1.record()
    barrier()
    ms_blk = max_over_ranks(e0.elapsed_time(e1))
    trainer._staged = None
    e2e = {"value": B * world * args.steps / (ms_e2e * 1e-3), "unit": "examples/s",
           "h2d_bytes_per_step": (host_ids[0].numel() * host_ids[0].element_size() + host_lab[0].numel() * 4) * world,
           "d2h_bytes_per_step": 4 * world, "ms_per_step": ms_e2e / args.steps,
           "api": "trainer.fit_host(batches): pinned host ids/labels in, every step's loss out (async D2H, read 2 steps later)",
           "blocking_per_step": {"value": B * world * args.steps / (ms_blk * 1e-3), "ms_per_step": ms_blk / args.steps,
                                 "api": "trainer.train_step_host(...): host blocks on loss.item() after every step"}}

    # ---- per-kernel timing, live, CUDA events on the launching stream (every rank: the sharded
    # step contains collectives) -------------------------------------------------------------------
    roof, shares = trainer.profile_kernels(ids_pool, lab_pool, iters=max(10, args.steps))
    barrier()
    fwd_ms = trainer.time_embed_fwd(ids_pool, iters=max(30, args.steps))      # headline kernel, back-to-back launches
    barrier()
    if world > 1:
        dist.destroy_process_group()
    if rank != 0:
        return

    # ---- roofline of the headline kernel (fused gather+FM forward) ---------------------------------
    peaks, peak_kind = measured_peaks()
    # SURVEY 8(d): ids + rows + first-order weights + stacked write + logit (3 644 B / example at C2); the kernel also
    # writes the sum_e side output the backward reads (4 D B / example) -- reported separately, not in `frac`
    alg_bytes = B * (S * (8 + 4 * D + 4) + 4 * S * D + 4)
    alg_bytes_with_sum = alg_bytes + B * 4 * D
    traffic = None
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "embed_fwd_traffic.json")))["dram_bytes_per_launch"]
    except Exception:
        pass
    # duration of the headline kernel: (a) INSIDE the step -- CUDA events on the launching stream around the kernel in the
    # eager per-kernel pass over the timed region's batches (the L2 / DRAM state the kernel really meets in training);
    # (b) back to back -- the same launch repeated with nothing in between, where every launch also pays for writing back
    # the previous launch's 109 MB of dirty stacked output.  `achieved` / `frac` use (a); (b) is reported beside it.
    step_key = "embed_fm_fwd" if "embed_fm_fwd" in shares else "embed_fm_fwd_p2p"
    fwd_s = shares[step_key] * 1e-3
    b2b_s = fwd_ms * 1e-3
    roofline = {"kernel": "embed_fm_fwd_kernel (fused 26-slot gather + first-order + FM)", "bound": "hbm",
                "how": f"mean duration of the kernel inside the step (CUDA events on the launching stream before / after it, "
                       f"eager passes over {max(10, args.steps)} steps of the id pool) = kernel_ms.{step_key}; "
                       "back_to_back = the same launch repeated between two events",
                "achieved": alg_bytes / fwd_s / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                "frac": alg_bytes / fwd_s / 1e9 / peaks["hbm_gbs"], "traffic": traffic,
                "traffic_source": "profiles/embed_fwd_traffic.json (ncu --set full capture of this kernel at this config; "
                                  "not re-measured inside this run)",
                "peak_source": peak_kind, "algorithmic_bytes_per_launch": alg_bytes,
                "bytes_convention": "SURVEY 8(d): S*(8+4D+4) + 4*S*D + 4 per example",
                "frac_incl_sum_e_output": alg_bytes_with_sum / fwd_s / 1e9 / peaks["hbm_gbs"],
                "us_per_launch": fwd_s * 1e6,
                "back_to_back": {"us_per_launch": b2b_s * 1e6, "achieved": alg_bytes / b2b_s / 1e9,
                                 "frac": alg_bytes / b2b_s / 1e9 / peaks["hbm_gbs"]}}

    cpu = None
    if not args.no_cpu_baseline and world == 1 and args.workload == "c2":     # CPU arm on rank 0 at N=1 only (torchrun pins OMP threads to 1)
        from oracle.torch_cpu import time_deepfm_cpu
        r = time_deepfm_cpu([C2["rows"]] * S, D, C2["dnn"], B, steps=8, warmup=1, max_seconds=25.0)
        cpu = {"value": r["examples_per_sec"], "unit": "examples/s", "cores": r["cores"], "kind": "port",
               "sample": f"{r['steps']} full train steps at B={B} (torch-CPU restatement of the reference path, "
                         f"not TensorFlow), host has {os.cpu_count()} logical CPUs"}

    line = {"metric": METRIC, "value": value, "unit": "examples/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "strong" if args.workload == "c5" else "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": dict(workload_config(world, args.workload),
                           ids="uniform int64" if args.ids == "uniform" else "Zipf(1.05) clipped to the table, int64"),
            "clocks": clk.summary(), "e2e": e2e, "gpu_launches": int(trainer.launches_per_step * args.steps),
            "launches_per_step": int(trainer.launches_per_step), "roofline": roofline, "kernel_ms": shares,
            "cpu_baseline": cpu, "final_loss": final_loss,
            "cuda_graph": trainer.graph is not None,
            "gemm_core": {0: "ffma", 1: "tcgen05 3xTF32, pre-split planes (tc)",
                          2: "tcgen05 3xTF32, hi/lo split in kernel (tc2); outputs >= 128 wide on the CTA-pair kernel (cta_group::2)"}[_lib._tc_variant if _lib._tc_enabled and not gemm_note else (1 if gemm_note else 0)],
            "exchange": getattr(trainer, "exchange", None) if world > 1 else None,
            "optimizer": args.optimizer if world == 1 else "sgd", "embed_fwd": args.embed_fwd if world == 1 else "ldg",
            "fwd_chunks": args.fwd_chunks if world == 1 else 1, "dw_first": bool(args.dw_first)}
    if world > 1 and exchange_note:
        line["exchange_note"] = exchange_note
    if gemm_note:
        line["gemm_note"] = gemm_note
    if args.tune:
        line["tune"] = args.tune
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
