#!/usr/bin/env python
"""bench.py — the hot path's headline measurement: RISC-V cycles PROVED per second at 2^20 rows (BASELINE.json `metric`).

One "step" = ONE WHOLE PROOF of the reference's v1 main component as recorded data (nexus_zkvm_b200/nexus_v1.py: the real 27 / 347 /
1012-column layout, 413 constraints of 13 transcribed chips, all 253 LogUp fractions, two multiplicity tables; padding-only witness —
`--machine add21` selects round 1's synthetic ADD machine instead) at 2^log_rows rows, i.e. everything
/root/reference prover/src/machine.rs:186-290 hands to Stwo: three tree commits (Circle iFFT, LDE, Blake2s Merkle), the LogUp
interaction trace, constraint quotients, the composition commit, OODS evaluation, DEEP quotients, FRI, proof of work, query
decommitments and the postcard proof bytes.  Host-side trace FILLING is outside the step (the north star keeps it on the CPU).

    python bench.py --gpus N --steps K --warmup W            # our arm (one process per GPU under torchrun for N > 1)
    python bench.py --impl reference ...                     # CPU arm: the oracle's whole proof of the SAME machine, really executed (2^18-row sample; --ref-log-rows 20 = full size)
    python bench.py --fft-sweep [--gpus N]                   # BASELINE configs[4]: Circle-FFT M31 elems/s, 2^16..2^26
    python bench.py --log-rows 22 --steps 2 --warmup 1       # BASELINE configs[2]: a 2^22-row full proof on one GPU
    python bench.py --dump-outputs DIR ...                   # also writes the last timed proof's outputs as DIR/*.npy (compare two builds)

  value   cycles/s with the filled trace (trees 0+1 evaluations) already RESIDENT in HBM when the timed region starts;
  e2e     the same proof through the public host-column API: pinned HOST trace columns in (packed: byte-valued columns travel as
          u8, the device widens them and applies finalize_columns) -> proof bytes on the host; H2D and D2H inside the timed region;
  stages / roofline   the commit transforms (iFFT + LDE of every committed column: the dominant kernel group) timed alone with
          CUDA events on the launching stream, against MEASURED_PEAKS.json's HBM bandwidth at 12 algorithmic bytes per trace element;
  N > 1   `value` is weak scaling: every rank proves its own 2^log_rows-row trace segment; the Merkle roots are all-gathered over NCCL.
          Two strong-scaling legs follow (on the world sizes the sharded paths were validated on: STRONG_VALIDATED_WORLDS): `strong_commit` = one
          1012-column tree committed by all ranks through nb200_commit_sharded, and `strong_proof` = ONE whole 2^log_rows-row proof by all ranks
          together (machine.prove_sharded: column-/row-sharded main component, re-shard fused into the last LDE pass over NVLink), whose bytes are
          compared with the single-GPU proof inside the run.
Inputs (1.4 GB of evaluations, 45 GB of intermediates per proof) are far larger than L2: no flush is needed between steps.
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

P = (1 << 31) - 1
METRIC = "RISC-V cycles proved/sec @ 2^20 rows"
UNIT = "cycles/s"
STRONG_VALIDATED_WORLDS = {2, 4, 8}    # world sizes on which the sharded commit / sharded proof ran on real GPUs this round (profiles/bench_n{2,4,8}_r02*.json)
CONFIG = dict(pow_bits=5, log_blowup=1, log_last=0, n_queries=3)   # PcsConfig::default() as restated in DESIGN.md


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--log-rows", type=int, default=20)
    ap.add_argument("--lanes", type=int, default=21)
    ap.add_argument("--machine", default="nexus_v1", choices=["nexus_v1", "add21"],
                    help="nexus_v1: the reference's v1 main component as recorded data (nexus_zkvm_b200/nexus_v1.py: 27/347/1012 columns, 413 constraints); "
                         "add21: the round-1 synthetic ADD machine (3/339/1012 columns, 424 constraints)")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--cpu-sample-log-rows", type=int, default=16)
    ap.add_argument("--ref-log-rows", type=int, default=18,
                    help="--impl reference: rows of the ONE whole proof the CPU arm executes (a bounded sample of the workload: a complete proof of the same "
                         "machine, not a partial one; 20 = the full-size run, ~6-10 min on 128 host threads: profiles/bench_ref_r02a.json)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-breakdown", action="store_true")
    ap.add_argument("--no-strong-proof", action="store_true", help="N > 1: skip the one-proof-over-all-ranks measurement")
    ap.add_argument("--strong-any-world", action="store_true",
                    help="run strong_commit / strong_proof at every world size (default: only at the sizes listed in STRONG_VALIDATED_WORLDS — a collective that "
                         "misbehaves on an unvalidated size would hang the whole bench line)")
    ap.add_argument("--no-verify", action="store_true")
    ap.add_argument("--fft-sweep", action="store_true")
    ap.add_argument("--sweep-logs", default="16,18,20,22,24,26")
    ap.add_argument("--sweep-mib", type=int, default=1024, help="MiB of evaluations per sweep point and GPU")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed proof returned (rank 0's) as DIR/<name>.npy in float64: proof bytes, "
                         "claimed LogUp sums, the three tree roots, the lookup parameters; inputs are seeded, so two builds can be compared file by file")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.fft_sweep:
        ap.error("--dump-outputs writes a proof's outputs; --fft-sweep computes none")
    return args


class ClockSampler:
    """SM clock and throttle reasons DURING the timed region (B200_PROFILING.md recipe).  NVML is polled from a thread every few ms
    (a 5-step timed region lasts ~0.15 s, too short for `nvidia-smi -lms`); nvidia-smi is the fallback when pynvml is unusable."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NVML_REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index=0, uuid=None):
        self.index, self.uuid = index, uuid
        self.rows = []          # nvidia-smi rows
        self.samples = []       # (sm_mhz, reasons bitmask) from NVML
        self.proc = None
        self.nvml = None
        self.stop_flag = threading.Event()

    def _nvml_handle(self):
        import pynvml
        pynvml.nvmlInit()
        if self.uuid:
            try:
                u = self.uuid if str(self.uuid).startswith("GPU-") else "GPU-" + str(self.uuid)
                return pynvml, pynvml.nvmlDeviceGetHandleByUUID(u.encode() if hasattr(u, "encode") else u)
            except Exception:
                pass
        vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
        idx = self.index
        if vis:
            ent = vis.split(",")
            if self.index < len(ent) and ent[self.index].strip().isdigit():
                idx = int(ent[self.index])
        return pynvml, pynvml.nvmlDeviceGetHandleByIndex(idx)

    def start(self):
        try:
            self.nvml, self.h = self._nvml_handle()
            self.max_mhz = int(self.nvml.nvmlDeviceGetMaxClockInfo(self.h, self.nvml.NVML_CLOCK_SM))
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _poll(self):
        n = self.nvml
        while not self.stop_flag.is_set():
            try:
                mhz = int(n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM))
                try:
                    rs = int(n.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:
                    rs = int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                self.samples.append((mhz, rs))
            except Exception:
                pass
            time.sleep(0.004)

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.nvml is not None:
            self.stop_flag.set()
            self.t.join(timeout=1)
            sm = sorted(m for m, _ in self.samples)
            reasons = set()
            for _, rs in self.samples:
                for bit, name in self.NVML_REASONS.items():
                    if rs & bit:
                        reasons.add(name)
            return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(reasons),
                    "samples": len(sm), "source": "nvml"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm = sorted(int(r[1]) for r in self.rows if len(r) >= 9 and r[1].isdigit())
        mx = [int(r[2]) for r in self.rows if len(r) >= 9 and r[2].isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) >= 9:
                for nme, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nme)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi"}


def workload_config(args, m, world):
    nc = m.air.n_columns()
    return {"workload": f"full STARK proof (stwo::prover::prove + the 3 trace-tree commits + LogUp interaction trace) of a 2^{args.log_rows}-row synthetic "
                        f"trace, {nc[0]}+{nc[1]}+{nc[2]} M31 columns, blow-up {1 << CONFIG['log_blowup']}, Blake2s Merkle, per GPU",
            "log_rows": args.log_rows, "columns": int(sum(nc)), "constraints": int(sum(len(c.constraints) for c in m.air.components)), "machine": args.machine,
            "pcs_config": CONFIG, "l2": "working set (tens of GB per proof) far larger than L2; no flush needed",
            "sharding": "one trace segment per GPU (weak scaling) + NCCL all-gather of the Merkle roots" if world > 1 else "single GPU"}


def make_machine(args, log_rows=None):
    from nexus_zkvm_b200 import machine as M
    if args.machine == "nexus_v1":
        from nexus_zkvm_b200.nexus_v1 import NexusV1Machine
        return NexusV1Machine(log_rows or args.log_rows)
    return M.AddMachine(log_size=log_rows or args.log_rows, n_lanes=args.lanes)


def fill_trace(m, seed):
    """(main_cols, mult) as nexus_zkvm_b200.machine.prove takes them (plain host arrays; the CPU arm and the verifier use these)."""
    if hasattr(m, "n_main"):           # NexusV1Machine: a list of all tree-1 columns (multiplicities included)
        return m.fill_main_trace(seed=seed), None
    return m.fill_main_trace(seed=seed)


def oracle_full_prove(m, cols, mult):
    """One whole proof by the oracle (CPU restatement of the same pipeline), all host threads; returns (seconds, proof, claimed, aux)."""
    from nexus_zkvm_b200 import machine as M
    from tests.oracle_backend import OracleBackend
    t0 = time.perf_counter()
    proof, claimed, aux = M.prove(m, OracleBackend(), cols, mult, config=CONFIG)
    return time.perf_counter() - t0, proof, claimed, aux


def run_reference(args):
    """CPU arm: the reference's own prover cannot be built here (Rust + un-vendored stwo, no cargo: DESIGN.md §2), so this times the
    oracle port's WHOLE proof of the same machine, really executed on every host core — every stage, every column, nothing extrapolated.
    The bounded sample the contract asks for is the row count: one complete proof at 2^ref_log_rows rows (default 2^18: about two
    minutes on the GPU box's 128 threads; the metric is per row, and the port's rate still rises with size — 1.8 k cycles/s at 2^16, 3.0 k at
    2^20 — so the smaller sample is stated, not hidden: `--ref-log-rows 20` runs the full-size proof)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import pyoracle as orc
    orc.set_num_threads(os.cpu_count() or 1)   # torchrun exports OMP_NUM_THREADS=1; the CPU arm uses every host core
    ref_rows = min(args.ref_log_rows, args.log_rows)
    m = make_machine(args, ref_rows)
    cols, mult = fill_trace(m, 0)
    t, proof, claimed, aux = oracle_full_prove(m, cols, mult)   # ONE step: a CPU proof of this size takes minutes
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, proof, claimed, aux)
    value = (1 << ref_rows) / t
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": 1, "warmup": 0,
            "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32 (M31)",
            "data": "synthetic", "impl": "reference", "config": workload_config(args, m, 1),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": orc.num_threads(), "kind": "port",
                             "sample": f"one whole 2^{ref_rows}-row proof of the same machine ({t:.1f} s, {len(proof)} proof bytes): every stage and column executed, "
                                       f"no extrapolation; the GPU arm's config is 2^{args.log_rows} rows (--ref-log-rows {args.log_rows} runs that size on the CPU)"},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "reference_log_rows": ref_rows, "note": "steps/warmup fixed to 1/0: one CPU proof takes minutes"}
    print(json.dumps(line), flush=True)


def dump_outputs(d, proof, claimed, aux):
    """What a caller of machine.prove receives, as float64 arrays (every value is a byte or an M31 element < 2^31: exact in float64)."""
    import numpy as np
    os.makedirs(d, exist_ok=True)
    out = {"proof": np.frombuffer(proof, dtype=np.uint8),
           "claimed_sums": np.array(claimed, dtype=np.uint32).reshape(-1, 4),
           "roots": np.frombuffer(b"".join(aux["roots"]), dtype=np.uint8).reshape(-1, 32),
           "params": np.array(aux["params"], dtype=np.uint32).reshape(-1, 4)}
    for name, a in out.items():
        np.save(os.path.join(d, name + ".npy"), a.astype(np.float64))


def load_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)

    import numpy as np
    import torch
    import nexus_zkvm_b200 as nb
    from nexus_zkvm_b200 import machine as M
    from nexus_zkvm_b200.prover import CudaBackend

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    stream = torch.cuda.Stream(device=dev)
    ctx = nb.Context(local, stream=stream.cuda_stream)
    if args.fft_sweep:
        with torch.cuda.stream(stream):
            run_fft_sweep(args, ctx, torch, dist, dev, stream, rank, world)
        if world > 1:
            dist.destroy_process_group()
        return

    n_rows = 1 << args.log_rows
    m = make_machine(args)
    be = CudaBackend(ctx)
    # ---- the filled trace, in pinned host memory, packed: byte-valued main columns (limbs, flags, register indices) travel as u8
    if args.machine == "nexus_v1":
        all_cols, mult = fill_trace(m, rank)
        byte_block = ctx.host_alloc_bytes(m.n_main << args.log_rows).reshape(m.n_main, n_rows)
        for i in range(m.n_main):
            byte_block[i] = all_cols[i]                       # every one of the 347 main columns holds values < 256
        small = all_cols[m.n_main:]                           # the extension components' multiplicity columns (2^8, 2^5 rows)
        host_cols = [byte_block] + small
        wide_blocks = [byte_block]
        h2d = byte_block.nbytes + sum(c.nbytes for c in small) + sum(c.nbytes for c in m.preprocessed_columns())
        host_format = "packed: %d u8 columns (widened on the device) + %d small u32 columns" % (m.n_main, len(small))
        del all_cols
        pre = m.preprocessed_columns()                        # cached; the big block goes to pinned memory once
        pinned_pre = ctx.host_alloc_bytes(pre[0].size).reshape(pre[0].shape)
        pinned_pre[:] = pre[0]
        m._pre_cache[0] = pinned_pre
    else:
        pc_block = ctx.host_alloc(1, args.log_rows)
        byte_block = ctx.host_alloc_bytes((m.n_main_columns() - 1) << args.log_rows).reshape(m.n_main_columns() - 1, n_rows)
        host_cols, mult = m.fill_main_trace(seed=rank, packed_out=(pc_block, byte_block))
        small = [mult]
        wide_blocks = [pc_block, byte_block]
        h2d = pc_block.nbytes + byte_block.nbytes + mult.nbytes + sum(c.nbytes for c in m.preprocessed_columns())
        host_format = "packed: 1 u32 column + %d u8 columns (widened on the device)" % (m.n_main_columns() - 1)

    with torch.cuda.stream(stream):
        ctx.precompute_twiddles(args.log_rows + 3)
        # resident copies of trees 0 + 1 (finalized order) for the HBM-resident headline
        up = be.prover(m.words, CONFIG)
        pre_cols = []
        for c_ in m.preprocessed_columns():
            a_ = np.asarray(c_)
            pre_cols += list(a_.astype(np.uint32)) if a_.ndim == 2 else [a_]
        t0_res = up._batches_from_host(pre_cols, True)
        del pre_cols
        wide = np.concatenate([b.astype(np.uint32) for b in wide_blocks])
        t1_res = [ctx.upload(wide, coset_order=True)] + [ctx.upload(np.asarray(c, dtype=np.uint32)[None, :], coset_order=True) for c in small]
        del wide, up
        roots_dev = torch.zeros((4, 32), dtype=torch.uint8, device=dev)
        gathered = [torch.zeros_like(roots_dev) for _ in range(world)] if world > 1 else None
        last = {}

        def exchange_roots(aux):
            if world > 1:   # the caps exchange of the north star: 3 x 32 bytes per rank
                roots_dev[:3].copy_(torch.frombuffer(bytearray(b"".join(aux["roots"])), dtype=torch.uint8).view(3, 32), non_blocking=True)
                dist.all_gather(gathered, roots_dev)

        def step_resident():
            proof, claimed, aux = M.prove(m, be, None, None, config=CONFIG, resident=(t0_res, t1_res))
            exchange_roots(aux)
            last.update(proof=proof, claimed=claimed, aux=aux)
            return proof

        def step_e2e():
            proof, claimed, aux = M.prove(m, be, host_cols, mult, config=CONFIG)
            exchange_roots(aux)
            last.update(proof_e2e=proof)
            return proof

        def barrier():
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()

        for _ in range(args.warmup):
            step_resident()
        barrier()
        sampler = ClockSampler(local, getattr(torch.cuda.get_device_properties(dev), "uuid", None)) if rank == 0 else None
        if sampler:
            sampler.start()
        l0 = ctx.launches
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(args.steps):
            step_resident()
        e1.record(stream)
        barrier()
        clocks = sampler.stop() if sampler else None
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        ms_per_step = float(ms.item()) / args.steps
        launches = (ctx.launches - l0) * world
        value = world * n_rows / (ms_per_step * 1e-3)
        if rank == 0 and args.dump_outputs:
            dump_outputs(args.dump_outputs, last["proof"], last["claimed"], last["aux"])

        # ---- e2e: pinned host columns -> proof bytes on the host, copies inside the timed region
        e2e = None
        if not args.no_e2e:
            step_e2e()
            barrier()
            f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            f0.record(stream)
            for _ in range(args.e2e_steps):
                pe = step_e2e()
            f1.record(stream)
            barrier()
            assert pe == last["proof"], "the proof from host columns differs from the HBM-resident one"
            ems = torch.tensor([f0.elapsed_time(f1)], device=dev)
            if world > 1:
                dist.all_reduce(ems, op=dist.ReduceOp.MAX)
            e2e = {"value": world * n_rows / (float(ems.item()) / args.e2e_steps * 1e-3), "unit": UNIT, "ms_per_step": float(ems.item()) / args.e2e_steps,
                   "h2d_bytes_per_step": int(h2d) * world, "d2h_bytes_per_step": (len(pe) + 4 * 32) * world, "steps": args.e2e_steps,
                   "host_format": host_format}

        # ---- stage breakdown + roofline of the dominant kernel group (rank 0): CUDA events on the launching stream
        stages, roofline = None, None
        if rank == 0 and not args.no_breakdown:
            stages, roofline = commit_breakdown(args, ctx, torch, dev, stream, m)

        # ---- N > 1: ONE commitment over all ranks through the library's NCCL path (strong scaling of the commit stage; not replicas)
        strong, strong_pf = None, None
        if world > 1 and (world in STRONG_VALIDATED_WORLDS or args.strong_any_world):
            strong = strong_commit(args, ctx, torch, dist, dev, stream, rank, world, m)
            if not args.no_strong_proof:
                strong_pf = strong_proof(args, ctx, be, torch, dist, dev, stream, rank, world, m)
        elif world > 1:
            strong = strong_pf = {"skipped": f"the in-library sharded paths were exercised on {sorted(STRONG_VALIDATED_WORLDS)} GPUs this round; pass --strong-any-world to run them on {world}"}

    verified = None
    if rank == 0 and not args.no_verify:
        try:
            # the oracle's independent verifier accepts the proof (transcript replayed from the returned roots with the ORACLE's channel)
            from tests.oracle_backend import verify_with_replayed_transcript
            verify_with_replayed_transcript(m, last["proof"], last["claimed"], last["aux"])
            verified = True
        except Exception as e:
            verified = f"failed: {e!r}"

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            from oracle import pyoracle as orc
            orc.set_num_threads(os.cpu_count() or 1)
            ms_ = make_machine(args, args.cpu_sample_log_rows)
            cs, mu = fill_trace(ms_, 0)
            tcpu, _p, _c, _a = oracle_full_prove(ms_, cs, mu)
            cpu_baseline = {"value": (1 << args.cpu_sample_log_rows) / tcpu, "unit": UNIT, "cores": orc.num_threads(), "kind": "port",
                            "sample": f"one whole proof of the same machine at 2^{args.cpu_sample_log_rows} rows ({tcpu:.1f} s); `--impl reference` runs a 2^{min(args.ref_log_rows, args.log_rows)}-row proof"}
        except Exception as e:  # the GPU numbers must still be reported
            cpu_baseline = {"value": None, "unit": UNIT, "cores": None, "kind": "port", "sample": f"failed: {e!r}"}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "u32 (M31)", "data": "synthetic", "config": workload_config(args, m, world),
                "clocks": clocks, "e2e": e2e, "gpu_launches": launches, "roofline": roofline, "cpu_baseline": cpu_baseline,
                "stages": stages, "strong_commit": strong if world > 1 else None, "strong_proof": strong_pf if world > 1 else None, "proof_bytes": len(last["proof"]), "verified_by_oracle_verifier": verified,
                "claimed_sums_cancel": M.verify_claimed_sums(last["claimed"]), "roots": [r.hex()[:16] for r in last["aux"]["roots"]]}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def strong_proof(args, ctx, be, torch, dist, dev, stream, rank, world, m, reps=3):
    """ONE proof of the 2^log_rows-row machine by ALL ranks together (machine.prove_sharded: BASELINE configs[3], SURVEY §8e) — the same trace on
    every rank (rank 0's), trees 0/1 resident as column shards, every collective inside the library.  The proof bytes are compared with the
    single-GPU proof of the same trace computed on rank 0."""
    from nexus_zkvm_b200 import machine as M
    from nexus_zkvm_b200.prover import CudaBackend
    cols, mult = fill_trace(m, 0)
    pr = be.prover(m.words, CONFIG)
    res = [M.shard_host_tree(m, pr, m.preprocessed_columns(), rank, world),
           M.shard_host_tree(m, pr, list(cols) + ([mult] if mult is not None else []), rank, world)]
    del pr
    ts, proof = [], None
    for rep in range(reps + 1):
        dist.barrier(); torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        proof, claimed, aux = M.prove_sharded(m, be, None, None, rank, world, config=CONFIG, resident=res)
        b.record(stream)
        torch.cuda.synchronize()
        if rep:
            ts.append(a.elapsed_time(b))
    t = torch.tensor([min(ts)], device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    same_single = None
    if rank == 0:
        import nexus_zkvm_b200 as nb
        ctx1 = nb.Context(dev.index)          # no communicator: the ordinary single-GPU proof of the same trace
        p1, _c1, _a1 = M.prove(m, CudaBackend(ctx1), cols, mult, config=CONFIG)
        same_single = bool(p1 == proof)
        ctx1.close()
    h = torch.frombuffer(bytearray(__import__("hashlib").sha256(proof).digest()), dtype=torch.uint8).to(dev)
    allh = [torch.zeros_like(h) for _ in range(world)]
    dist.all_gather(allh, h)
    same = all(bool((x == h).all().item()) for x in allh)
    ms = float(t.item())
    return {"ms": ms, "value": (1 << args.log_rows) / (ms * 1e-3), "unit": UNIT, "log_rows": args.log_rows, "scaling": "strong",
            "same_proof_on_all_ranks": bool(same), "equals_single_gpu_proof": same_single, "proof_bytes": len(proof)}


def strong_commit(args, ctx, torch, dist, dev, stream, rank, world, m, reps=3):
    """One tree (the interaction tree's 2^log_rows-row columns) committed by ALL ranks together: nb200_commit_sharded = column-sharded fused
    iFFT+LDE -> grouped ncclSend/Recv of packed row slices over NVLink -> row-sharded sub-tree hashing -> ncclAllGather of the caps."""
    import nexus_zkvm_b200 as nb
    total = sum(1 for ls in m.column_log_sizes()[2] if ls == args.log_rows)
    ctx.comm_init_from_torch(dist, dev)
    first, count = nb.Context.shard_range(total, world, rank)
    g = torch.Generator(device=dev); g.manual_seed(1234 + rank)
    ev_t = torch.randint(0, P, (max(count, 1), 1 << args.log_rows), device=dev, dtype=torch.int32, generator=g)
    ev = ctx.wrap_device(ev_t.data_ptr(), count, args.log_rows) if count else None
    ts, root = [], None
    for rep in range(reps + 1):
        dist.barrier(); torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        co, rows, sub, caps, root = ctx.commit_sharded(ev, total, args.log_rows, CONFIG["log_blowup"])
        b.record(stream)
        torch.cuda.synchronize()
        co.free(); sub.free(); rows.free()
        if rep:
            ts.append(a.elapsed_time(b))
    t = torch.tensor([min(ts)], device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    r_t = torch.frombuffer(bytearray(root), dtype=torch.uint8).to(dev)
    allr = [torch.zeros_like(r_t) for _ in range(world)]
    dist.all_gather(allr, r_t)
    same = all(bytes(x.cpu().numpy().tobytes()) == root for x in allr)
    lde_bytes = total * (4 << (args.log_rows + CONFIG["log_blowup"]))
    return {"ms": float(t.item()), "columns": int(total), "log_rows": args.log_rows, "rows_per_s": (1 << args.log_rows) / (float(t.item()) * 1e-3),
            "same_root_on_all_ranks": bool(same), "root": root.hex()[:16],
            "limiting_collective": "grouped ncclSend/ncclRecv row re-shard of the LDE", "exchanged_bytes_per_rank": int(lde_bytes / world * (world - 1) / world)}


def commit_breakdown(args, ctx, torch, dev, stream, m):
    """iFFT + LDE (nb200_interpolate_evaluate) and Merkle (nb200_merkle_commit) of the proof's three trace trees, each timed alone."""
    peaks = load_peaks()
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    big = [sum(1 for ls in tree if ls == args.log_rows) for tree in m.column_log_sizes()]   # the 2^log_rows-row columns of each trace tree
    n_rows = 1 << args.log_rows
    t_fft = t_mrk = 0.0
    reps = 3
    for c in big:
        ev_t = torch.randint(0, P, (c, n_rows), device=dev, dtype=torch.int32)
        ev = ctx.wrap_device(ev_t.data_ptr(), c, args.log_rows)
        co, lde = ctx.interpolate_evaluate(ev, CONFIG["log_blowup"])
        for rep in range(reps + 1):
            a, b, d = (torch.cuda.Event(enable_timing=True) for _ in range(3))
            a.record(stream); ctx.interpolate_evaluate(ev, CONFIG["log_blowup"], co, lde); b.record(stream)
            tr = ctx.merkle_commit([lde]); d.record(stream)
            torch.cuda.synchronize()
            tr.free()
            if rep > 0:
                t_fft += a.elapsed_time(b) / reps; t_mrk += b.elapsed_time(d) / reps
        co.free(); lde.free(); del ev_t
    elems = sum(big) * n_rows
    fft_bytes = 12.0 * elems  # SURVEY §8(d): fused LDE commit = read 4 + write 8 per trace element
    ach = fft_bytes / (t_fft * 1e-3) / 1e9
    stages = {"commit_transforms_ms": t_fft, "merkle_ms": t_mrk, "columns": int(sum(big)),
              "fft_Melems_per_s": elems * (1 + (1 << CONFIG["log_blowup"])) / (t_fft * 1e-3) / 1e6,
              "merkle_GBps_read": 4.0 * elems * (1 << CONFIG["log_blowup"]) / (t_mrk * 1e-3) / 1e9}
    traffic = None
    try:   # measured once per build with ncu (tools/ncu_traffic.py writes it); never a constant baked into this file
        tj = json.load(open(os.path.join(ROOT, "profiles", "fft_traffic.json")))
        traffic = float(tj["dram_bytes_per_trace_element"]) * elems
    except Exception:
        pass
    roofline = {"bound": "hbm", "kernel": "commit transforms: fft_tile_async_kernel<inv> + fft_mid_kernel + fft_tile_async_kernel<fwd> (Circle iFFT + LDE FFT of every committed column)",
                "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak, "traffic": traffic,
                "traffic_unit": "B per step (profiles/fft_traffic.json: ncu dram bytes of the three kernels)" if traffic else None,
                "algorithmic": fft_bytes, "peak_source": peak_src,
                "algorithmic_bytes": "12 B per trace element (read 4, write 8) for iFFT+LDE; x columns x 2^log_rows",
                "int_pipe_note": "the butterflies are INT32 work: 4 ALU-pipe instructions each, 30 butterflies per trace element (DESIGN.md §4)"}
    return stages, roofline


def run_fft_sweep(args, ctx, torch, dist, dev, stream, rank, world):
    """BASELINE configs[4]: Circle-FFT throughput 2^16..2^26 M31 elements, columns sharded over the ranks (independent transforms)."""
    out = []
    for lg in [int(x) for x in args.sweep_logs.split(",")]:
        n_cols = max(1, (args.sweep_mib << 20) // (4 << lg))
        ev_t = torch.randint(0, P, (n_cols, 1 << lg), device=dev, dtype=torch.int32)
        ev = ctx.wrap_device(ev_t.data_ptr(), n_cols, lg)
        ctx.precompute_twiddles(lg)
        res = {}
        for name, fn in (("ifft", lambda: ctx.interpolate(ev)), ("fft", lambda: ctx._chk(nbl().nb200_evaluate(ctx._h, ev._h, 0, ev._h)))):
            ts = []
            for _ in range(4):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                if world > 1:
                    dist.barrier()
                torch.cuda.synchronize()
                a.record(stream); fn(); b.record(stream)
                torch.cuda.synchronize()
                ts.append(a.elapsed_time(b))
            t = torch.tensor([min(ts[1:])], device=dev)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            res[name] = float(t.item())
        elems = world * n_cols * (1 << lg)
        out.append({"log_size": lg, "columns_per_gpu": n_cols, "ifft_ms": res["ifft"], "fft_ms": res["fft"],
                    "ifft_Gelems_per_s": elems / (res["ifft"] * 1e-3) / 1e9, "fft_Gelems_per_s": elems / (res["fft"] * 1e-3) / 1e9})
        del ev_t
    if rank == 0:
        peaks = load_peaks()
        hbm = float(peaks.get("hbm_gbs", 6650.0))
        best = max(o["ifft_Gelems_per_s"] for o in out)
        print(json.dumps({"metric": "Circle-FFT M31 elems/sec", "value": best * 1e9, "unit": "elems/s", "n_gpus": world, "higher_is_better": True,
                          "scaling": "weak", "data": "synthetic", "dtype": "u32 (M31)",
                          "config": {"workload": "configs[4]: Circle iFFT / FFT sweep, in place, %d MiB of columns per GPU per point" % args.sweep_mib},
                          "roofline_elems_per_s_at_8B": world * hbm / 8.0 * 1e9, "sweep": out}), flush=True)


def nbl():
    import nexus_zkvm_b200 as nb
    return nb.lib()


if __name__ == "__main__":
    main()
