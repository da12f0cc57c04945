#!/usr/bin/env python3
"""Headline benchmark: GRU-HS[64] samples/s (BASELINE.json metric), one JSON line on stdout.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--mode f16|tf32|bf16|fp32] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
           bench.py --gpus N --steps K --warmup W

Workload (config.workload): BASELINE.json configs[1] -- the cfg-2 checkpoint (GRU-HS[64]-L[DCPreESR] AKAI),
1024 streams x 60 s of synthetic 48 kHz audio per GPU, predict() semantics (zero state -> 1024-sample warm
start -> the signal).  A "step" is one full pass over that batch.  Multi-GPU: streams are sharded, every rank
runs its own 1024 streams with no data-path collective (weak scaling); value = all samples / max-over-ranks time.

  value          device-resident: inputs and outputs in HBM, CUDA events around K steps on the launching stream
  e2e            the same pass through RNN.predict_host (ntm_gru_predict_host): pinned HOST input, HOST output,
                 host<->device copies inside the timed region
  roofline       contract asks for the tensor-pipe fraction: achieved = samples/s x 25088 FLOP (BASELINE.md
                 section 4) over the measured bf16 peak of MEASURED_PEAKS.json; extra keys give the honest bound of
                 the kernel that actually ran (fp32 FMA pipe / MUFU) and the (negligible) HBM rate
  strict         the same workload (10 s of it) in the strict tensor-core mode "f16x3" (fp32-grade: max-abs <= 1e-5 against
                 the reference like the CUDA-core fp32 mode), beside the f16-operand headline
  cpu_baseline   the reference's own RNN class (code/model.py staged under baseline/_ref by baseline/stage_ref.py; the
                 oracle's port of it if that is absent) on the host cores, bounded sample
  aux.cfg4_strong  BASELINE.json configs[3]: 65 536 streams x 10 s sharded over the N ranks (strong scaling, no collective)

--dump-outputs DIR writes what the last timed step of the device-resident pass returned (rank 0's streams), so that two
builds can be compared output for output: the inputs are seeded, identical for the same arguments.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
if "reference" in sys.argv[1:] and "--impl" in sys.argv[1:]:
    # the reference arm is the reference's CPU path: code/model.py pins its tensors to "cuda" whenever torch sees one
    # (code/model.py:61,223), so this process must not see the GPUs
    os.environ["CUDA_VISIBLE_DEVICES"] = ""

import numpy as np  # noqa: E402
import torch  # noqa: E402

FS = 48000
FLOP_PER_SAMPLE = 25088          # 2*(192*64 + 192 + 64), BASELINE.md section 4
BYTES_PER_SAMPLE = 8             # x in + y out
WORKLOAD = "cfg2: GRU-HS[64]-L[DCPreESR] AKAI _BEST, {B} streams x {sec:g} s synthetic 48 kHz audio per GPU"


def load_sd(tag):
    z = np.load(os.path.join(ROOT, "tests", "golden", f"ckpt_{tag}.npz"))
    return {k: torch.from_numpy(z[k]) for k in z.files if k not in ("model_type", "weights_dir")}


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["bf16_tflops_sustained"]), float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json, sustained)"
    except Exception:
        return 1400.0, 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.path = index, None, None

    def __enter__(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None
        return self

    def __exit__(self, *exc):
        if self.proc is not None:
            time.sleep(0.25)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()

    def summary(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        try:
            rows = [r.split(",") for r in open(self.path).read().strip().splitlines() if r.strip()]
            sm = sorted(float(r[0]) for r in rows)
            out["sm_mhz"] = sm[len(sm) // 2]
            out["sm_max_mhz"] = float(rows[0][1])
            out["power_w_max"] = max(float(r[2]) for r in rows)
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            out["reasons"] = [n for i, n in enumerate(names) if any("Active" == r[3 + i].strip() for r in rows)]
            out["samples"] = len(rows)
            os.unlink(self.path)
        except Exception:
            pass
        return out


def reference_runner():
    """-> (run(x) -> y, kind, description): the reference's CPU arithmetic for a (B, 1, T) batch with predict() semantics per
    stream.  kind "reference": the UNMODIFIED `RNN` class of code/model.py (staged under baseline/_ref, see
    baseline/stage_ref.py) -- zero state, its own warm_start(), the batch-1 warm state broadcast to the B streams (the
    reference's predict() itself only accepts B = 1, SURVEY 9.3 #3), then its forward() over 2048-sample segments exactly
    like the loop of RNN.predict (code/model.py:218-246).  kind "port": oracle/ref_torch.py, the same torch.nn.GRU + Linear
    calls restated (used only if baseline/_ref is absent)."""
    sys.path.insert(0, os.path.join(ROOT, "baseline"))
    import stage_ref
    if stage_ref.available():
        refmodel = stage_ref.load_reference()
        net = refmodel.RNN(input_size=1, hidden_size=64, output_size=1, skip=False)
        net.load_state_dict(stage_ref.load_checkpoint("cfg2"))
        net.eval()

        def run(x):
            B, T = x.shape[0], x.shape[2]
            with torch.no_grad():
                net.initialize_hidden()
                net.warm_start()
                net.hidden = net.hidden.expand(1, B, 64).contiguous()
                out = torch.empty_like(x)
                for s0 in range(0, T, 2048):
                    out[:, :, s0:s0 + 2048] = net.forward(x[:, :, s0:s0 + 2048])
            return out
        return run, "reference", "code/model.py RNN (baseline/_ref, unmodified): warm_start + forward over 2048-sample segments"
    from oracle import ref_torch
    net = ref_torch.RefNet(load_sd("cfg2"))
    return (lambda x: net.predict(x)[0]), "port", "oracle/ref_torch.py (torch.nn.GRU + Linear restated; baseline/_ref not staged)"


REF_SEGMENTS = int(os.environ.get("NTM_REF_SEGMENTS", "2"))   # 2048-sample segments per reference step (the --impl reference arm and cpu_baseline)
DUMP_SAMPLES = 1 << 23           # output samples --dump-outputs keeps at most (32 MB of float32)


def dump_outputs(out_dir, y, hidden):
    """DIR/y.npy: the (B, 1, T) output of the step, whole if it has at most DUMP_SAMPLES elements, else its elements at a
    fixed seeded set of flat indices (DUMP_SAMPLES draws of np.random.default_rng(0), sorted, so the same for every run
    with the same --streams / --seconds) as a 1-D array.  DIR/hidden.npy: the (1, B, 64) state the step left in the
    model.  Both float32."""
    os.makedirs(out_dir, exist_ok=True)
    if y.numel() > DUMP_SAMPLES:
        idx = np.sort(np.random.default_rng(0).integers(0, y.numel(), DUMP_SAMPLES))
        y = y.reshape(-1)[torch.from_numpy(idx).to(y.device)]
    np.save(os.path.join(out_dir, "y.npy"), y.float().cpu().numpy())
    np.save(os.path.join(out_dir, "hidden.npy"), hidden.float().cpu().numpy())


def cpu_baseline(B, seg_count, threads):
    """The reference on the host cores over a bounded sample: `seg_count` 2048-sample segments of B streams.  Runs in a child
    process that does not see the GPUs: the reference's RNN pins its state to "cuda" whenever torch sees one
    (code/model.py:61,223), and this leg is its CPU path."""
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="", NTM_REF_SEGMENTS=str(seg_count))
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT"):
        env.pop(k, None)
    r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "1", "--warmup", "1",
                        "--streams", str(B)], env=env, capture_output=True, text=True, timeout=900)
    if r.returncode != 0:
        raise RuntimeError("cpu_baseline child failed:\n" + r.stderr[-2000:])
    line = json.loads(r.stdout.strip().splitlines()[-1])
    c = line["cpu_baseline"]
    return c["value"], c["kind"], c["sample"] + f"; torch {torch.__version__}"


def run_reference(args, rank):
    """`--impl reference`: the reference's own CPU path with all host threads, on a bounded sample of the same workload
    (same streams, same checkpoint, the first REF_SEGMENTS x 2048 samples of every stream per step); rank 0 only."""
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    from ntm_b200 import signals
    torch.set_num_threads(threads)
    run, kind, desc = reference_runner()
    B, T = args.streams, 2048 * REF_SEGMENTS
    x = torch.from_numpy(signals.stream_batch(B, T, dur=60.0)).reshape(B, 1, T)
    for _ in range(args.warmup):
        run(x)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        y = run(x)
    dt = time.perf_counter() - t0
    value = B * T * args.steps / dt
    sample = (f"{B} streams x {T} samples per step (bounded sample of the {args.seconds:g} s workload: the loop is stationary in "
              f"time); {desc}")
    print(json.dumps({
        "impl": "reference", "metric": "GRU-HS64 samples/sec", "value": value, "unit": "samples/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD.format(B=args.streams, sec=args.seconds), "sample": sample,
                   "streams": B, "samples_per_stream_per_step": T, "same_config": False,
                   "same_config_note": "same checkpoint, streams and signal generator; the CPU arm times a bounded sample"},
        "cpu_baseline": {"value": value, "unit": "samples/s", "cores": threads, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "realtime_streams": value / FS, "checksum": float(y[:, :, ::257].double().sum()),
    }))


def bind_to_gpu_numa_node(index):
    """Multi-rank runs: pin this rank's threads (and so the first-touch placement of its pinned staging buffers) to the NUMA
    node its GPU hangs off -- what `numactl --cpunodebind --membind` would do per rank.  Returns the node or None."""
    try:
        p = torch.cuda.get_device_properties(index)
        bdf = f"{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return node
    except Exception:
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--mode", default="f16", choices=["fp32", "f16", "f16x3", "strict", "tf32", "bf16"])
    ap.add_argument("--streams", type=int, default=1024)
    ap.add_argument("--seconds", type=float, default=60.0)
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--no-aux", action="store_true", help="skip the batch-1 / large-batch side measurements")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-cfg4", action="store_true", help="skip the 65 536-stream strong-scaling leg (aux.cfg4_strong)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the output and final state of the last timed step as DIR/y.npy and DIR/hidden.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    import ntm_b200
    from ntm_b200 import lib, sharding, signals
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: ntm_b200 has no CPU path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        # keep stdout to the ONE JSON line: NCCL prints its version banner (and NCCL_DEBUG output) to stdout when the
        # communicator comes up, i.e. at the first collective -- do that here with fd 1 pointed at stderr
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize(dev)
        finally:
            os.dup2(saved, 1)
            os.close(saved)

    B, T = args.streams, int(round(args.seconds * FS))
    model = ntm_b200.RNN(input_size=1, hidden_size=64, output_size=1, skip=False).to(dev)
    model.load_state_dict(load_sd("cfg2"))
    model.mode = args.mode
    first, _ = sharding.weak_scaling_range(B, rank)         # this rank's own streams; nothing is exchanged
    x = signals.stream_batch_device(B, T, dev, first_stream=first, dur=args.seconds).reshape(B, 1, T)
    torch.cuda.synchronize(dev)

    def barrier():
        torch.cuda.synchronize(dev)
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    L = lib.load()
    with torch.inference_mode():
        # ---- device-resident pass -------------------------------------------------------------------
        for _ in range(args.warmup):
            y = model.predict(x)
        del y
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 * args.steps + 2)]
        barrier()
        launches0 = L.ntm_query(lib.Q_KERNEL_LAUNCHES)
        with ClockSampler(local_rank) as clk:
            ev[0].record()
            for i in range(args.steps):
                model.initialize_hidden()
                model.warm_start()
                model.hidden = model.hidden.expand(1, B, 64).contiguous()
                ev[2 + 2 * i].record()
                y = model(x)                       # the persistent kernel: all T steps of all B streams
                ev[3 + 2 * i].record()
            ev[1].record()
            barrier()
        launches = L.ntm_query(lib.Q_KERNEL_LAUNCHES) - launches0
        kernel_name = lib.KERNEL_NAMES.get(L.ntm_query(lib.Q_LAST_KERNEL), "?")
        total_ms = ev[0].elapsed_time(ev[1])
        kern_ms = sum(ev[2 + 2 * i].elapsed_time(ev[3 + 2 * i]) for i in range(args.steps)) / args.steps
        checksum = float(y[:, :, ::4801].double().sum())
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, y, model.hidden)
        del y
        model.static_io = False
        total_ms = sharding.max_over_ranks(total_ms, dev, dist)
        value = sharding.aggregate_rate(B * T * args.steps, world, total_ms * 1e-3)

        # ---- end to end: pinned host in -> engine pipeline -> pinned host out -------------------------
        import psutil
        avail = psutil.virtual_memory().available
        need = 3 * B * T * 4 * max(1, min(world, 8))          # pinned x and y (float32, then binary16) of every rank on this host
        T_e = T if need < 0.5 * avail else max(FS, int(0.25 * avail / (8 * B * max(1, world))) // FS * FS)
        numa_node = bind_to_gpu_numa_node(local_rank) if world > 1 else None
        xh = torch.empty((B, 1, T_e), dtype=torch.float32, pin_memory=True)
        xh.copy_(x[:, :, :T_e])
        yh = torch.empty((B, 1, T_e), dtype=torch.float32, pin_memory=True)      # result buffer reused across steps
        model.predict_host(xh, out=yh)
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            model.predict_host(xh, out=yh)
        torch.cuda.synchronize(dev)
        e2e_s = time.perf_counter() - t0
        e2e_value = sharding.aggregate_rate(B * T_e * args.e2e_steps, world, sharding.max_over_ranks(e2e_s, dev, dist))
        e2e_ok = bool(torch.isfinite(yh[:, :, ::4801]).all())
        # the same call with the opt-in 16-bit host transport (ntm_gru_predict_host_f16): binary16 samples over the host link
        xh16 = torch.empty((B, 1, T_e), dtype=torch.float16, pin_memory=True)
        xh16.copy_(x[:, :, :T_e])
        yh16 = torch.empty((B, 1, T_e), dtype=torch.float16, pin_memory=True)
        model.predict_host(xh16, out=yh16)
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            model.predict_host(xh16, out=yh16)
        torch.cuda.synchronize(dev)
        e2e16_s = time.perf_counter() - t0
        e2e16_value = sharding.aggregate_rate(B * T_e * args.e2e_steps, world, sharding.max_over_ranks(e2e16_s, dev, dist))
        sl = slice(0, None, 4801)
        d16 = (yh16[:, :, sl].double() - yh[:, :, sl].double())
        e2e16_esr = float((d16 ** 2).sum() / ((yh[:, :, sl].double() ** 2).sum() + 1e-12))
        del xh, yh, xh16, yh16

        # ---- the same workload in the strict (fp32-grade) tensor-core mode, every rank its own shard ------------
        strict = strict_leg(model, x, args, dev, barrier, sharding, dist, world, lib)
        del x
        # ---- BASELINE.json configs[3]: 65 536 streams x 10 s sharded over the ranks (strong scaling) ------------
        cfg4 = None if args.no_cfg4 else cfg4_strong_leg(ntm_b200, signals, sharding, lib, dev, dist, rank, world, barrier, args.mode)

        # ---- side measurements (rank 0, outside the timed regions) -------------------------------------
        aux = {}
        if rank == 0 and not args.no_aux:
            aux = aux_measurements(ntm_b200, signals, dev, args.mode)
        if cfg4 is not None:
            aux["cfg4_strong"] = cfg4

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    clocks = clk.summary()
    tensor_peak, hbm_peak, peak_src = measured_peaks()
    sps_kernel = B * T / (kern_ms * 1e-3)
    achieved_tflops = sps_kernel * FLOP_PER_SAMPLE / 1e12
    f_clk = (clocks.get("sm_mhz") or 1965.0) * 1e6
    sm_count = L.ntm_query(lib.Q_SM_COUNT)
    line = {
        "metric": "GRU-HS64 samples/sec", "value": value, "unit": "samples/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None,
        "dtype": {"fp32": "f32", "f16": "f16 operands, f32 accumulate/gates/state", "tf32": "tf32 operands, f32 accumulate/gates/state",
                  "bf16": "bf16 operands, f32 accumulate/gates/state",
                  "f16x3": "f16 hi/lo operand pairs (3 MMAs per product, fp32-grade), f32 accumulate/gates/state",
                  "strict": "f16 hi/lo operand pairs (3 MMAs per product, fp32-grade), f32 accumulate/gates/state"}[args.mode],
        "data": "synthetic",
        "config": {"workload": WORKLOAD.format(B=B, sec=args.seconds), "streams_per_gpu": B, "samples_per_stream": T,
                   "sample_rate": FS, "mode": args.mode, "parallelism": f"stream-sharded x{world}, no collective",
                   "l2": "inputs (%.1f GB per GPU) are larger than L2; no flush needed" % (B * T * 4 / 1e9)},
        "realtime_streams": value / FS,
        "e2e": {"value": e2e_value, "unit": "samples/s", "h2d_bytes_per_step": B * T_e * 4,
                "d2h_bytes_per_step": B * T_e * 4, "samples_per_stream": T_e, "finite": e2e_ok,
                "api": "RNN.predict_host -> ntm_gru_predict_host (pinned host buffers)",
                "rank0_numa_node": numa_node,
                "f16_transport": {"value": e2e16_value, "unit": "samples/s", "h2d_bytes_per_step": B * T_e * 2,
                                  "d2h_bytes_per_step": B * T_e * 2, "esr_vs_f32_transport_rank0": e2e16_esr,
                                  "api": "RNN.predict_host(float16 host tensor) -> ntm_gru_predict_host_f16 (opt-in: binary16 "
                                         "samples over the host link, same fp32-state kernels)"}},
        "gpu_launches": launches,
        "clocks": clocks,
        "roofline": {
            "bound": "tensor", "achieved": achieved_tflops, "peak": tensor_peak, "unit": "TFLOP/s",
            "frac": achieved_tflops / tensor_peak,
            # dram__bytes_read+write of this kernel from one `ncu --set full` capture (profiles/r02f_mma_b1024_ncu.txt,
            # gru_mma4_kernel: 395.7 MB read + 352.8 MB written for 1024 x 96 000 samples = 7.61 B per sample against 8
            # algorithmic -- the last ~10 % of the y writes were still in the 126 MB L2 when the kernel ended), scaled to this launch
            "traffic": round(748.5e6 / (1024 * 96000) * B * T), "algorithmic_bytes": BYTES_PER_SAMPLE * B * T,
            "traffic_source": "estimated_from_profile: bytes per sample of the ncu capture at 1024 x 96 000, scaled to this launch",
            "peak_source": peak_src,
            "kernel_ms": kern_ms, "kernel": kernel_name,
            "regime": "latency-bound recurrence: 1024 streams = 7 per SM, one dependent GRU step at a time (DESIGN.md section 4)",
            "legacy_mma_sync_peak_tflops": sm_count * 4 * 4096 / 8 * f_clk / 1e12,
            "frac_of_mma_sync_peak": achieved_tflops / (sm_count * 4 * 4096 / 8 * f_clk / 1e12),
            "ns_per_timestep": kern_ms * 1e6 / T,
            "fp32_fma_peak_tflops": sm_count * 128 * 2 * f_clk / 1e12,
            "frac_of_fp32_fma_peak": achieved_tflops / (sm_count * 128 * 2 * f_clk / 1e12),
            "mufu_bound_samples_per_s": sm_count * 16 * f_clk / 192,
            "hbm_gbs_achieved": sps_kernel * BYTES_PER_SAMPLE / 1e9, "hbm_frac": sps_kernel * BYTES_PER_SAMPLE / 1e9 / hbm_peak,
        },
        "strict": strict,
        "checksum": checksum,
        "aux": aux,
    }
    if not args.no_cpu:
        threads = os.cpu_count() or 1
        v, kind, sample = cpu_baseline(min(B, 1024), REF_SEGMENTS, threads)
        line["cpu_baseline"] = {"value": v, "unit": "samples/s", "cores": threads, "kind": kind, "sample": sample}
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


def strict_leg(model, x, args, dev, barrier, sharding, dist, world, lib):
    """The headline workload (its first 10 s) in the strict tensor-core mode: fp32-grade result (max-abs <= 1e-5 against the
    reference, tests/test_parity_gpu.py STRICT_CLASS) from f16 hi/lo operand pairs, 3 MMAs per product.  Device-resident,
    CUDA events, max over ranks, whole-job aggregate like `value`."""
    B = x.shape[0]
    Ts = min(x.shape[2], 10 * FS)
    xs = x[:, :, :Ts]
    prev = model.mode
    model.mode = "f16x3"
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    try:
        for _ in range(2):
            model.predict(xs[:, :, :FS])
        best = 1e30
        for _ in range(2):
            model.initialize_hidden()
            model.warm_start()
            model.hidden = model.hidden.expand(1, B, 64).contiguous()
            barrier()
            e0.record(); y = model(xs); e1.record()
            torch.cuda.synchronize(dev)
            best = min(best, sharding.max_over_ranks(e0.elapsed_time(e1), dev, dist))
        kernel = lib.KERNEL_NAMES.get(lib.load().ntm_query(lib.Q_LAST_KERNEL), "?")
        finite = bool(torch.isfinite(y[:, :, ::4801]).all())
        del y
    finally:
        model.mode = prev
    value = sharding.aggregate_rate(B * Ts, world, best * 1e-3)
    tflops = value / world * 3 * FLOP_PER_SAMPLE / 1e12          # executed tensor FLOPs per GPU: three MMAs per product
    peak = measured_peaks()[0]
    return {"mode": "f16x3", "value": value, "unit": "samples/s", "kernel": kernel, "ns_per_timestep": best * 1e6 / Ts,
            "samples_per_stream": Ts, "finite": finite, "tolerance": "fp32 class: max-abs <= 1e-5 vs the reference (tests)",
            "executed_tensor_tflops_per_gpu": tflops, "frac_of_measured_bf16_peak": tflops / peak,
            "algorithmic_frac": value / world * FLOP_PER_SAMPLE / 1e12 / peak}


def cfg4_strong_leg(ntm_b200, signals, sharding, lib, dev, dist, rank, world, barrier, mode):
    """BASELINE.json configs[3]: GRU-HS[64], 65 536 streams x 10 s, stream-sharded over the N ranks with no data-path
    collective.  Rank r owns streams shard_range(65536, r, N) and walks the 10 s in time chunks with the state carried on the
    device (the materialised signals would be 252 GB).  Inputs: per-stream synthetic signals generated on the device, four
    distinct chunks cycled (resident before the timed region, as for `value`); every chunk launch reads and writes its own
    1.6 GB of HBM, far beyond L2.  Timed with CUDA events over all launches of the pass, max over ranks."""
    TOTAL, T10 = 65536, 10 * FS
    lo, hi = sharding.shard_range(TOTAL, rank, world)
    Bs = hi - lo
    m = ntm_b200.RNN(1, 64, 1, False).to(dev)
    m.load_state_dict(load_sd("cfg2"))
    m.mode = mode
    Tc = 3000
    while Bs * Tc * 2 < 65536 * 3000 and Tc < 48000:       # ~0.8 GB per staged array whatever the shard size
        Tc *= 2
    nchunk = (T10 + Tc - 1) // Tc
    xs = [signals.stream_batch_device(Bs, Tc, dev, first_stream=lo + 977 * k, dur=10.0).reshape(Bs, 1, Tc) for k in range(4)]
    m.static_io = True                                      # y / state buffers reused across the chunk launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def one_pass():
        m.initialize_hidden()
        m.warm_start()
        m.hidden = m.hidden.expand(1, Bs, 64).contiguous()
        barrier()
        e0.record()
        done = 0
        for k in range(nchunk):
            n = min(Tc, T10 - done)
            y = m(xs[k & 3] if n == Tc else xs[k & 3][:, :, :n])
            done += n
        e1.record()
        torch.cuda.synchronize(dev)
        return e0.elapsed_time(e1), y

    one_pass()
    ms, y = one_pass()
    kernel = lib.KERNEL_NAMES.get(lib.load().ntm_query(lib.Q_LAST_KERNEL), "?")
    finite = bool(torch.isfinite(y[:, :, ::97]).all())
    ms = sharding.max_over_ranks(ms, dev, dist)
    value = TOTAL * T10 / (ms * 1e-3)
    del xs, y, m
    torch.cuda.empty_cache()
    return {"workload": "cfg4: GRU-HS[64] 65 536 streams x 10 s, stream-sharded (strong scaling), time-chunked with carried state",
            "value": value, "unit": "samples/s", "n_gpus": world, "scaling": "strong", "streams_per_gpu": Bs, "chunk_samples": Tc,
            "chunks": nchunk, "ms": ms, "kernel": kernel, "mode": mode, "finite": finite, "realtime_streams": value / FS,
            "per_gpu_samples_per_s": value / world,
            "tensor_tflops_per_gpu": value / world * FLOP_PER_SAMPLE / 1e12,
            "frac_of_measured_bf16_peak": value / world * FLOP_PER_SAMPLE / 1e12 / measured_peaks()[0]}


def aux_measurements(ntm_b200, signals, dev, mode):
    """cfg 5 (batch-1 real-time blocks) and a large-batch point, each a few hundred ms."""
    out = {}
    m1 = ntm_b200.RNN(1, 64, 1, False).to(dev)
    m1.load_state_dict(load_sd("cfg1"))
    x1 = torch.from_numpy(signals.signal("sweepnoise", 480000, seed=0)).to(dev).reshape(1, 1, -1)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    m1.predict(x1)
    m1.initialize_hidden(); m1.warm_start()
    e0.record(); m1(x1); e1.record(); torch.cuda.synchronize(dev)
    out["batch1_kernel_ns_per_sample"] = e0.elapsed_time(e1) * 1e6 / 480000
    nblk = 2000
    m1.initialize_hidden(); m1.warm_start()
    for k in range(50):
        m1(x1[:, :, 64 * k:64 * k + 64])
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    for k in range(nblk):
        m1(x1[:, :, 64 * k:64 * k + 64])
    torch.cuda.synchronize(dev)
    out["batch1_block64_ns_per_sample_incl_launch"] = (time.perf_counter() - t0) * 1e9 / (nblk * 64)
    # the same generic forward() with per-shape output buffers kept by the module (static_io), and captured in a CUDA Graph
    # (SURVEY 8d cfg 5: the torch.ops entry points launch on PyTorch's current stream and allocate nothing)
    for md in ("fp32", "f16"):
        m1.mode = md
        m1.static_io = True
        m1.initialize_hidden(); m1.warm_start()
        for k in range(50):
            m1(x1[:, :, 64 * k:64 * k + 64])
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        for k in range(nblk):
            m1(x1[:, :, 64 * k:64 * k + 64])
        torch.cuda.synchronize(dev)
        out[f"batch1_block64_ns_per_sample_forward_static_io_{md}"] = (time.perf_counter() - t0) * 1e9 / (nblk * 64)
        xs = torch.zeros((1, 1, 64), device=dev)
        m1.initialize_hidden(); m1.warm_start()
        m1.hidden = m1.hidden.clone()
        m1(xs)                                   # state now lives in the module's static buffer (updated in place)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            yg = m1(xs)
        for k in range(50):
            xs.copy_(x1[:, :, 64 * k:64 * k + 64]); graph.replay()
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        for k in range(nblk):
            xs.copy_(x1[:, :, 64 * k:64 * k + 64]); graph.replay()
        torch.cuda.synchronize(dev)
        out[f"batch1_block64_ns_per_sample_cuda_graph_{md}"] = (time.perf_counter() - t0) * 1e9 / (nblk * 64)
        del graph, yg
        m1.static_io = False
    m1.mode = "fp32"
    # the same through the block-stream API (one C call per block), exact fp32 and f16 tensor-core arithmetic
    for md in ("fp32", "f16"):
        m1.mode = md
        m1.initialize_hidden(); m1.warm_start()
        bs = m1.block_stream(1, 64)
        blocks = [x1[:, :, 64 * k:64 * k + 64] for k in range(nblk)]
        for k in range(50):
            bs.process(blocks[k])
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        for k in range(nblk):
            bs.process(blocks[k])
        torch.cuda.synchronize(dev)
        out[f"batch1_block64_ns_per_sample_blockstream_{md}"] = (time.perf_counter() - t0) * 1e9 / (nblk * 64)
        # per-block latency: submit one block, wait for it (what a real-time callback sees)
        lat = []
        for k in range(200):
            t1 = time.perf_counter()
            bs.process(blocks[k])
            torch.cuda.synchronize(dev)
            lat.append(time.perf_counter() - t1)
        lat.sort()
        out[f"batch1_block64_latency_us_median_{md}"] = lat[len(lat) // 2] * 1e6
    # the same blocks through the RESIDENT server kernel (ntm_rt_*): host block in -> host block out, no launch per block
    m1.mode = "f16"
    m1.initialize_hidden(); m1.warm_start()
    torch.cuda.synchronize(dev)
    x1h = x1.cpu().reshape(1, -1)
    hblocks = [x1h[:, 64 * k:64 * k + 64].contiguous() for k in range(nblk)]
    rt = m1.realtime_stream(1, 64)
    for k in range(50):
        rt.process(hblocks[k])
    lat = []
    t0 = time.perf_counter()
    for k in range(nblk):
        t1 = time.perf_counter()
        rt.process(hblocks[k])
        lat.append(time.perf_counter() - t1)
    out["batch1_block64_ns_per_sample_resident_server_f16"] = (time.perf_counter() - t0) * 1e9 / (nblk * 64)
    lat.sort()
    out["batch1_block64_latency_us_median_resident_server_f16"] = lat[len(lat) // 2] * 1e6
    out["batch1_block64_latency_us_p99_resident_server_f16"] = lat[int(len(lat) * 0.99)] * 1e6
    rt.close()
    m1.mode = "fp32"
    m1.initialize_hidden(); m1.warm_start()
    m1.mode = "f16"
    e0.record(); m1(x1); e1.record(); torch.cuda.synchronize(dev)
    out["batch1_kernel_ns_per_sample_f16"] = e0.elapsed_time(e1) * 1e6 / 480000
    m1.mode = "fp32"
    from ntm_b200 import lib
    L = lib.load()
    mb = ntm_b200.RNN(1, 64, 1, False).to(dev)
    mb.load_state_dict(load_sd("cfg2"))

    def timed(x, m, tuning=(0, 0)):
        B = x.shape[0]
        L.ntm_set_tuning(*tuning)
        m.predict(x[:, :, :1200])
        m.initialize_hidden(); m.warm_start()
        hw = m.hidden.expand(1, B, 64).contiguous()
        # one untimed full-size call first: the first call of a shape allocates its output inside torch's caching allocator
        # (a cudaMalloc of up to 0.8 GB in the timed region made single measurements here swing by a factor of 6), then best of two
        best = float("inf")
        for rep in range(3):
            m.hidden = hw.clone()
            e0.record(); m(x); e1.record(); torch.cuda.synchronize(dev)
            if rep:
                best = min(best, e0.elapsed_time(e1))
        L.ntm_set_tuning(0, 0)
        return B * x.shape[2] / (best * 1e-3)

    # the same 1024-stream workload (2 s of it) in every arithmetic mode, and the tcgen05 kernel forced
    x2 = signals.stream_batch_device(1024, 96000, dev, dur=60.0).reshape(1024, 1, 96000)
    per_mode = {}
    for md in ("fp32", "f16x3", "f16", "tf32", "bf16"):
        mb.mode = md
        per_mode[md] = timed(x2, mb)
    out["cfg2_samples_per_s_by_mode"] = per_mode
    del x2
    # throughput regime (cfg 4 per-GPU widths): the three tensor-core kernels.  "auto" is what the dispatcher picks
    # (mma.sync below ~110 streams per SM, the stream-major tcgen05 kernel above); sm_count x 256 streams is the
    # width at which every SM owns exactly two 128-stream tiles (no partial wave).
    big = {}
    sms = L.ntm_query(lib.Q_SM_COUNT)
    for Bb, Tb in ((8192, 12000), (sms * 256, 3000), (65536, 3000)):
        xb = signals.stream_batch_device(Bb, Tb, dev, dur=10.0).reshape(Bb, 1, Tb)
        mb.mode = "f16"
        big[str(Bb)] = {"auto": timed(xb, mb), "auto_kernel": lib.KERNEL_NAMES.get(L.ntm_query(lib.Q_LAST_KERNEL), "?"),
                        "mma_sync": timed(xb, mb, (8, 3))}
        if Bb >= sms * 64:
            big[str(Bb)]["tcgen05_stream_major"] = timed(xb, mb, (2 if Bb > sms * 128 else 1, 4))
        mb.mode = "f16x3"
        big[str(Bb)]["strict_f16x3_auto"] = timed(xb, mb)
        big[str(Bb)]["strict_f16x3_kernel"] = lib.KERNEL_NAMES.get(L.ntm_query(lib.Q_LAST_KERNEL), "?")
        mb.mode = "tf32"
        big[str(Bb)]["tf32_auto"] = timed(xb, mb)
        mb.mode = "fp32"
        big[str(Bb)]["fp32_cuda_core"] = timed(xb, mb)
        del xb
    # roofline of the throughput regime at the balanced width: tensor FLOP/s against the measured dense peak, and the
    # MUFU bound of the stream-major kernel
    bal = big[str(sms * 256)]["auto"]
    tensor_peak = measured_peaks()[0]
    out["large_batch_roofline"] = {
        "streams": sms * 256, "samples_per_s": bal, "kernel": big[str(sms * 256)]["auto_kernel"],
        "tensor_tflops": bal * FLOP_PER_SAMPLE / 1e12, "frac_of_measured_bf16_peak": bal * FLOP_PER_SAMPLE / 1e12 / tensor_peak,
        # MUFU work of the stream-major kernel: 3 ex2 per unit-step + the r/z reciprocal shared by two units + the n reciprocal
        # shared by four = 3.75 MUFU per unit-step (f16 / bf16 operands) at 16 lanes per clock and SM
        "mufu_per_unit_step": 3.75,
        "mufu_bound_samples_per_s_at_max_clock": sms * 16 * 1.965e9 / (64 * 3.75),
        "frac_of_mufu_bound": bal / (sms * 16 * 1.965e9 / (64 * 3.75)),
        "frac_of_round1_mufu_bound_4_per_unit": bal / (sms * 16 * 1.965e9 / (64 * 4.0))}
    out["large_batch_samples_per_s"] = big
    # cfg 3: DiffDelGRU (GRU + fused fractional-delay read), 256 streams x 30 s, predict() semantics
    Bd, Td = 256, 30 * FS
    md = ntm_b200.DiffDelRNN(1, 64, 1, False, max_delay=signals.DELAY_MAX).to(dev)
    md.load_state_dict(load_sd("cfg3"))
    xd = signals.stream_batch_device(Bd, Td, dev, dur=30.0).reshape(Bd, 1, Td)
    dd = signals.delay_trajectory_device(Bd, Td, dev).reshape(Bd, 1, Td)
    md.diffdel.check_delay = False            # the reference's assert costs a full extra pass + a stream sync
    cfg3 = {}
    for mdm in ("fp32", "f16"):
        md.mode = mdm
        md.predict(xd[:, :, :4800], dd[:, :, :4800])
        torch.cuda.synchronize(dev)
        best = float("inf")
        for _ in range(2):                        # (the first full-size call allocates its two outputs inside the timed region)
            e0.record(); yd, pd = md.predict(xd, dd); e1.record(); torch.cuda.synchronize(dev)
            best = min(best, e0.elapsed_time(e1))
            del yd, pd
        cfg3[mdm] = Bd * Td / (best * 1e-3)
    out["cfg3_diffdel_256x30s_samples_per_s"] = cfg3
    del xd, dd
    # evaluation losses on the device (SURVEY section 8f rank 2): one pass over 1024 streams x 30 s of (output, target);
    # HBM-bound by construction: 8 algorithmic bytes per sample against the measured copy bandwidth
    Bl, Tl = 1024, 30 * FS
    tl = 0.2 * torch.randn(Bl, 1, Tl, device=dev)
    ol = tl + 0.02 * torch.randn(Bl, 1, Tl, device=dev)
    hbm_peak = measured_peaks()[1]
    losses = {}
    for name, fn in (("ESR", ntm_b200.ESRLoss()), ("DCPreESR", ntm_b200.DCPreESR())):
        fn(ol, tl)
        best = 1e9
        for _ in range(3):
            e0.record(); fn(ol, tl); e1.record(); torch.cuda.synchronize(dev)
            best = min(best, e0.elapsed_time(e1))
        gbs = 8.0 * Bl * Tl / (best * 1e-3) / 1e9
        losses[name] = {"samples_per_s": Bl * Tl / (best * 1e-3), "hbm_gbs": gbs, "frac_of_measured_hbm_peak": gbs / hbm_peak}
    out["loss_pass_1024x30s"] = losses
    # stand-alone delay line (SURVEY section 8f rank 1, apply_delay): 12 algorithmic bytes per sample (x, d read; y written)
    dline = ntm_b200.TimeVaryingDelayLine(max_delay=signals.DELAY_MAX)
    dline.check_delay = False
    dtr = signals.delay_trajectory_device(Bl, Tl, dev).reshape(Bl, 1, Tl)
    dline.init_buffer(Bl)
    dline(ol, dtr)
    best = 1e9
    for _ in range(3):
        dline.init_buffer(Bl)
        e0.record(); dline(ol, dtr); e1.record(); torch.cuda.synchronize(dev)
        best = min(best, e0.elapsed_time(e1))
    gbs = 12.0 * Bl * Tl / (best * 1e-3) / 1e9
    out["delay_pass_1024x30s"] = {"samples_per_s": Bl * Tl / (best * 1e-3), "hbm_gbs": gbs,
                                  "frac_of_measured_hbm_peak": gbs / hbm_peak}
    del tl, ol, dtr
    out["existing_gpu_path_cudnn"] = cudnn_bar(dev)
    return out


def cudnn_bar(dev):
    """The "existing GPU kernel" bar of SURVEY.md section 8d: what `model.RNN(...).cuda()` runs today -- torch.nn.GRU (cuDNN)
    + nn.Linear in fp32, driven like code/model.py:218-246 (2048-sample segments with carried hidden state) -- on the cfg 2
    checkpoint, 1024 streams x 1 s, same B200, CUDA events.  Library code timed beside the product; it is not the product."""
    sd = load_sd("cfg2")
    B, T, SEG = 1024, FS, 2048
    gru = torch.nn.GRU(1, 64, batch_first=True).to(dev)
    head = torch.nn.Linear(64, 1).to(dev)
    gru.load_state_dict({k[4:]: v for k, v in sd.items() if k.startswith("GRU.")})
    head.load_state_dict({k[7:]: v for k, v in sd.items() if k.startswith("output.")})
    x = 0.1 * torch.randn(B, T, 1, device=dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def run():
        h, ys = None, []
        for s0 in range(0, T, SEG):
            hs, h = gru(x[:, s0:s0 + SEG], h)
            ys.append(head(hs))
        return ys

    with torch.inference_mode():
        run()
        torch.cuda.synchronize(dev)
        best = 1e9
        for _ in range(2):
            e0.record(); run(); e1.record(); torch.cuda.synchronize(dev)
            best = min(best, e0.elapsed_time(e1))
    return {"samples_per_s": B * T / (best * 1e-3), "ns_per_timestep": best * 1e6 / T,
            "sample": f"{B} streams x {T} samples in {SEG}-sample segments, torch.nn.GRU (cuDNN {torch.backends.cudnn.version()}) "
                      "+ nn.Linear, fp32"}


if __name__ == "__main__":
    main()
