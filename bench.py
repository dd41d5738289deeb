#!/usr/bin/env python
"""bench.py — batched Plonk-by-hand prove + verify throughput on B200 (BASELINE.json's metric).

    python bench.py --gpus 1 --steps K --warmup W            # this repo's CUDA path
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...   # one rank per GPU, weak scaling
    python bench.py --impl reference ...                     # the CPU path (oracle port of the reference) on host cores

A step is one pass of the hot path over one batch: prove 2^20 D_fullpath witnesses per GPU (configs[1] of
BASELINE.json), verify the 2^20 proofs, pack the verdict bitmap and digest the proof bytes; with N > 1 every rank does
that on its own shard (digest fused into the prover, bitmap into the verifier) and the bitmaps + digests are all-gathered
over NCCL (the only collective: one per ring cycle, overlapped with the next cycle's kernels).  The K timed steps are ONE
CUDA graph (kernels and collectives), so the host is out of the timed path; the K-step region is repeated `--reps` times
and the median of the per-repetition maxima over ranks is reported.  `value` counts proof+verify pairs per second over
all ranks with inputs resident in HBM; `e2e` is the same work through the host-pointer C-ABI calls (host buffers, H2D and
D2H inside the timed region).  Inputs rotate through a ring of distinct batches larger than L2.

After the timed region the line's `check` object is filled: the exact 2^20-item batch of ring slot 0 is replayed through
the CPU oracle byte for byte, and with N > 1 rank 0 recomputes the whole N-rank index range alone and compares the
gathered bitmaps and digests with it.
"""
import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "plonk-by-fingers_b200", "python"))
sys.dont_write_bytecode = True      # the benchmark leaves the tree as it found it (it may be read-only)

METRIC = "plonk_by_hand_prove_plus_verify_throughput"
UNIT = "proof+verify/s"
N_PER_GPU = 1 << 20
SEED = 0xB200
WORKLOAD = "batched prover+verifier: 2^20 D_fullpath witnesses of the pbh circuit per GPU per step, shared SRS (s=2, 7 points)"
MASK64 = (1 << 64) - 1
DUMP_ITEMS = 1 << 18                # --dump-outputs: items sampled from the per-item outputs
DUMP_BITMAP_BYTES = 1 << 22         # --dump-outputs: leading bytes of the verdict bitmap kept


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU through NVML while the timed region runs."""

    def __init__(self, index, period=0.002):
        super().__init__(daemon=True)
        self.index, self.period, self.samples, self.reasons, self.max_mhz = index, period, [], set(), None
        self.power_w = []
        self._stop_evt = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM)
        except Exception as e:  # pragma: no cover - NVML missing
            self.nv, self.err = None, str(e)

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM))
                if len(self.samples) % 4 == 2:      # NVML queries take milliseconds each: power only every fourth round
                    try:
                        self.power_w.append(nv.nvmlDeviceGetPowerUsage(self.handle) / 1000.0)
                    except Exception:
                        pass
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        s = sorted(self.samples)
        pw = sorted(self.power_w)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s), "sm_mhz_min": (s[0] if s else None), "power_w_median": (pw[len(pw) // 2] if pw else None),
                "power_w_max": (pw[-1] if pw else None)}


_CPU_INPUTS = {}


def cpu_leg(sample_items, threads):
    """Oracle (C++ restatement of the reference) prove + verify on host cores; returns (pairs/s, seconds).  The D_fullpath
    inputs are generated once per sample size and reused (drawing them costs about twenty prove+verify attempts per
    item, none of it timed)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle as O
    if sample_items not in _CPU_INPUTS:
        biggest = max(_CPU_INPUTS, default=0)
        if biggest >= sample_items:
            _CPU_INPUTS[sample_items] = tuple(np_slice(a, sample_items) for a in _CPU_INPUTS[biggest])
        else:
            _CPU_INPUTS[sample_items] = O.generate_inputs(sample_items, seed=SEED, dist=1, threads=threads)[:4]
    w, r, c, u = _CPU_INPUTS[sample_items]
    t0 = time.perf_counter()
    proof, status = O.prove_batch(w, r, c, threads=threads)
    O.verify_batch(proof, c, u, threads=threads, want_gt=False)
    dt = time.perf_counter() - t0
    return sample_items / dt, dt


def cpu_model():
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return None


def np_slice(a, n):
    import numpy as np
    return np.ascontiguousarray(a[..., :n])


def run_reference(args):
    """--impl reference: the reference's CPU algorithm (oracle port; the Rust crate cannot be built here) on all host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle as O
    threads = max(1, O.hardware_threads())
    if args.cpu_sample is None:
        # bounded sample: size the step so that the whole --steps K run stays near one minute of wall clock
        # (drawing the D_fullpath inputs, once, costs about twenty times one step on top)
        rate, _ = cpu_leg(2000 * threads, threads)
        sample = int(max(1000 * threads, min(6000 * threads, rate * 60.0 / max(1, args.steps))))
    else:
        sample = args.cpu_sample
    cpu_leg(sample, threads)                        # draws the inputs (untimed) and warms the caches
    for _ in range(max(0, args.warmup - 1)):
        cpu_leg(max(1000, sample // 10), threads)
    t_total = 0.0
    for _ in range(args.steps):
        _, dt = cpu_leg(sample, threads)
        t_total += dt
    value = sample * args.steps / t_total
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * t_total / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8 (F_17 / F_101 residues, u64 arithmetic)", "data": "synthetic",
        "config": {"workload": WORKLOAD, "sample_per_step": sample},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "cpu_model": cpu_model(), "nproc": os.cpu_count(),
                         "sample": f"{sample} D_fullpath items per step, prove then verify, C++ restatement of the reference, {threads} threads"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


# ---- static inputs of the roofline: executed instructions per item, from the committed ncu captures -------------------
def instr_table():
    """profiles/instr_per_item.json: thread instructions per item (total, FMA pipe, ALU pipe) of each fused kernel, read
    from the ncu reports named there.  STATIC: these are properties of the compiled code, not of this run; the times,
    the clocks and the pipe peaks they are combined with below ARE measured in this run."""
    try:
        with open(os.path.join(ROOT, "profiles", "instr_per_item.json")) as f:
            return json.load(f)
    except Exception:
        return {}


def roofline_entry(name, table_key, ms, items, bytes_per_item, peaks, instr):
    """One kernel against its four ceilings: HBM bytes, issue slots, FMA pipe, ALU pipe.  `bound` names the largest."""
    sec = ms * 1e-3
    ent = {"kernel": name, "ms": ms, "items": items, "items_per_s": items / sec,
           "hbm": {"achieved_GBps": bytes_per_item * items / sec / 1e9, "peak_GBps": peaks["hbm_gbs"],
                   "frac": bytes_per_item * items / sec / 1e9 / peaks["hbm_gbs"], "algorithmic_bytes_per_item": bytes_per_item}}
    fr = {"hbm": ent["hbm"]["frac"]}
    ins = instr.get(table_key)
    if ins:
        ent["instr_per_item_static"] = {k: ins[k] for k in ("total", "fma", "fp32", "imad", "alu") if k in ins}
        ent["instr_source_static"] = ins.get("source")

        def add(pipe, count, peak):
            if count is not None and peak:
                ach = count * items / sec
                ent[pipe] = {"achieved_thread_instr_per_s": ach, "peak_thread_instr_per_s": peak, "frac": ach / peak}
                fr[pipe] = ach / peak

        add("issue", ins.get("total"), peaks["issue_thread_instr_per_s"])
        # FP32 ops issue on both FMA pipes (peak: the FFMA rate), IMAD on the heavy one only (peak: the IMAD rate)
        add("fma-pipe", ins.get("fma"), peaks["fma_thread_ops_per_s"])
        if ins.get("imad", 0) > ins.get("fp32", 0):
            add("imad-pipe", ins.get("imad"), peaks.get("imad_thread_ops_per_s"))
        add("alu-pipe", ins.get("alu"), peaks["alu_thread_ops_per_s"])
    ent["bound"] = max(fr, key=fr.get)
    ent["frac"] = fr[ent["bound"]]
    return ent


def dump_outputs(out_dir, proof, status, result, bitmap, digest):
    """Write what one step hands its caller as .npy files in float32 / float64 (under 64 MB in all), so that two builds
    can be compared output for output: the proof planes, prover status and verdicts of a fixed, seeded sample of
    DUMP_ITEMS items (their indices in item_index.npy), the verdict bitmap (its first DUMP_BITMAP_BYTES bytes when longer)
    and the 64-bit proof digest as two exact 32-bit halves, low first."""
    import numpy as np
    n = status.numel()
    if n > DUMP_ITEMS:
        idx = np.sort(np.random.default_rng(SEED).choice(n, DUMP_ITEMS, replace=False))
    else:
        idx = np.arange(n)
    d = int(digest.item()) & MASK64
    arrays = {"item_index": idx.astype(np.float64),
              "proof": proof.cpu().numpy()[:, idx].astype(np.float32),
              "status": status.cpu().numpy()[idx].astype(np.float32),
              "result": result.cpu().numpy()[idx].astype(np.float32),
              "verdict_bitmap": bitmap[:DUMP_BITMAP_BYTES].cpu().numpy().astype(np.float32),
              "proof_digest": np.array([d & 0xFFFFFFFF, d >> 32], dtype=np.float64)}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--reps", type=int, default=7, help="repetitions of the K-step timed region (the median is reported)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--algo", default="table", choices=["table", "arith"])
    ap.add_argument("--items", type=int, default=N_PER_GPU, help="items per GPU per step")
    ap.add_argument("--ring", type=int, default=8, help="distinct input/output batches cycled through (L2 defeat)")
    ap.add_argument("--cpu-sample", type=int, default=None)
    ap.add_argument("--e2e-steps", type=int, default=None)
    ap.add_argument("--e2e-lanes", type=int, default=4, help="batches in flight on the packed end-to-end path (2..4)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg and the full-batch oracle replay")
    ap.add_argument("--no-arith", action="store_true", help="skip timing the PBH_ALGO_ARITH kernels")
    ap.add_argument("--no-fs", action="store_true", help="skip timing the Fiat-Shamir kernels")
    ap.add_argument("--no-uniform", action="store_true", help="skip timing the kernels on D_uniform inputs")
    ap.add_argument("--no-sweeps", action="store_true", help="skip the kernel sweeps of BASELINE.json configs[3] (N = 1 only)")
    ap.add_argument("--no-config2", action="store_true", help="skip the 16 M-proof verifier of BASELINE.json configs[2] (N = 1 only)")
    ap.add_argument("--no-config4", action="store_true", help="skip the 256 M-witness sharded run of BASELINE.json configs[4]")
    ap.add_argument("--config4-log2", type=int, default=28)
    ap.add_argument("--sweep-log2", type=str, default="24,28")
    ap.add_argument("--gather", default="window", choices=["window", "nccl"],
                    help="N > 1: how the shard summaries reach every rank: 'window' = stored into the peers' windows over NVLink by the "
                         "prover / verifier kernels themselves (pbh_window_*), 'nccl' = one NCCL all-gather per ring cycle")
    ap.add_argument("--no-gather", action="store_true",
                    help="DIAGNOSTIC ONLY: leave the all-gathers out of the timed region (the line is marked invalid); shows what the collective costs")
    ap.add_argument("--no-graph", action="store_true", help="launch the step's kernels directly instead of replaying one CUDA graph per K-step region")
    ap.add_argument("--no-overlap-prove", dest="overlap_prove", action="store_false",
                    help="launch every prover from one stream (default: odd steps launch from a second prover stream, so prove(k+1) fills the SMs prove(k) leaves)")
    ap.add_argument("--no-overlap-verify", dest="overlap_verify", action="store_false",
                    help="keep verify(k) and prove(k+1) on one stream inside the graph (default: verify(k) runs on a second stream beside prove(k+1))")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (proofs, status, verdicts, bitmap, digest; rank 0) "
                         "as DIR/<name>.npy in float32 / float64, per-item outputs as a fixed seeded sample")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)

    # Only the JSON line may reach stdout: libraries that print there (NCCL's version banner under NCCL_DEBUG, for one)
    # are sent to stderr for the whole run; the line itself is written to the saved descriptor at the end.
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    import numpy as np
    import torch
    import pbh_b200

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU fallback (use --impl reference for the CPU baseline)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    n = args.items
    K = args.steps
    ctx = pbh_b200.Context(device=local, algo=args.algo)
    stream = ctx.torch_stream()

    # ---- synthetic shard of this rank: item i of ring slot r has global index ((r * world) + rank) * n + i
    ring = max(1, args.ring)
    nb = (n + 7) // 8
    assert nb % 8 == 0, "items per GPU must be a multiple of 64"
    ins, outs = [], []
    # Summaries (verdict bitmap, then the 64-bit proof digest) of a whole ring cycle are contiguous so that ONE all-gather
    # can carry them; two sets, so that cycle c+1's kernels write set (c+1)%2 while set c%2 is still being gathered.
    row = nb + 8
    # How the N ranks exchange the summaries.  "window" (default): every rank owns a peer window (pbh_window_*) whose row r is rank
    # r's region; the prover and verifier kernels store their digest / bitmap into the own row AND, over NVLink, into the same
    # row of every peer's window, so the all-gather is complete when the kernels are and the timed region holds no collective.
    # "nccl": one all_gather_into_tensor per ring cycle on a side stream.
    collective = None
    window = None
    if world > 1:
        collective = args.gather
        if collective == "window":
            try:
                bpr = (2 * ring * row + 15) // 16 * 16
                window, handle = ctx.window_create(bpr, rank, world)
                hs = torch.zeros((world, 64), dtype=torch.uint8, device=dev)
                dist.all_gather_into_tensor(hs, torch.from_numpy(handle).to(dev))
                ctx.window_attach(hs.cpu().numpy())
            except Exception as e:   # no peer access between these devices: the NCCL path is the fallback FOR THE COLLECTIVE only
                print(f"[rank {rank}] peer window unavailable ({type(e).__name__}: {e}); using the NCCL all-gather", file=sys.stderr)
                window = None
            flag = torch.tensor([1 if window is not None else 0], dtype=torch.int32, device=dev)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            if int(flag.item()) == 0:
                window, collective = None, "nccl"
    if window is not None:
        win_sets = window[:, :2 * ring * row].view(world, 2, ring * row)
        summary_all = [win_sets[rank, b] for b in range(2)]
        gathered_all = [None, None]
    else:
        summary_all = [torch.zeros(ring * row, dtype=torch.uint8, device=dev) for _ in range(2)]
        gathered_all = [torch.empty(world * ring * row, dtype=torch.uint8, device=dev) if world > 1 else None for _ in range(2)]
    for r in range(ring):
        first = (r * world + rank) * n
        w, rd, c, u = ctx.generate_inputs(n, first_index=first, seed=SEED, dist=pbh_b200.DIST_FULLPATH)
        ins.append((w, rd, c, u, first))
        views = []
        for b in range(2):
            summary = summary_all[b][r * row:(r + 1) * row]
            views.append(dict(summary=summary, bitmap=summary[:nb], digest=summary[nb:].view(torch.int64)))
        outs.append(dict(proof=torch.empty((27, n), dtype=torch.uint8, device=dev), status=torch.empty((n,), dtype=torch.uint8, device=dev),
                         result=torch.empty((n,), dtype=torch.uint8, device=dev), sets=views, **views[0]))
    ctx.sync()
    torch.cuda.synchronize()
    comm_stream = torch.cuda.Stream(device=dev) if world > 1 else None
    KERNELS_PER_STEP = 2   # prover (+ fused proof digest), verifier (+ fused verdict bitmap)
    ctx_v = vstream = ctx_p1 = pstream1 = None
    if args.overlap_verify:
        # the verifier of step k runs on a second context (its own stream) beside the prover of step k + 1: the two touch
        # different ring slots, and the tail of one kernel fills the SMs the other has not reached yet
        ctx_v = pbh_b200.Context(device=local, algo=args.algo)
        vstream = ctx_v.torch_stream()
        if args.overlap_prove and ring >= 2:
            # the provers of consecutive steps are independent too (different ring slots): odd steps launch from a third
            # context's stream, so the persistent blocks of prove(k+1) take over each SM as the blocks of prove(k) leave it
            # instead of waiting for the whole grid to drain
            ctx_p1 = pbh_b200.Context(device=local, algo=args.algo)
            pstream1 = ctx_p1.torch_stream()
    if window is not None:
        for other in (ctx_v, ctx_p1):
            if other is not None:
                ctx.window_share(other)

    def enqueue_region(steps):
        """Enqueue exactly `steps` steps on `stream` (+ `vstream`, + the cycle all-gathers on `comm_stream`), joined back into
        `stream` at the end.  Cycle c (steps c*ring .. c*ring+ring-1, ring slots 0..) writes summary set c % 2; its ONE
        all-gather overlaps the kernels of cycle c + 1.  Used both directly and under stream capture."""
        gather_done = {}
        verified = {}                                          # ring slot -> event: the verifier that last read the slot's proof
        nccl_mode = world > 1 and window is None and not args.no_gather
        cycles = (steps + ring - 1) // ring
        for cyc in range(cycles):
            b = cyc % 2
            if nccl_mode and cyc >= 2:
                stream.wait_event(gather_done[cyc - 2])       # the all-gather that read this summary set has finished
                if vstream is not None:
                    vstream.wait_event(gather_done[cyc - 2])
            if pstream1 is not None and (nccl_mode or cyc == 0):
                pstream1.wait_stream(stream)                  # fork; with NCCL also everything `stream` waited for (previous cycle, gathers)
            for slot in range(min(ring, steps - cyc * ring)):
                w, rd, c, u, first = ins[slot]
                o = outs[slot]
                pst = pstream1 if (pstream1 is not None and slot % 2 == 1) else stream
                if slot in verified and not nccl_mode:
                    # the only dependency between cycles: this slot's proof planes are rewritten, so the verifier that read them
                    # a whole ring ago must be done (it is, long since: no stall, and no drain of the streams at the cycle's end)
                    pst.wait_event(verified[slot])
                if pst is pstream1:
                    with torch.cuda.stream(pstream1):
                        ctx_p1.prove_digest_batch(w, rd, c, o["proof"], o["status"], o["sets"][b]["digest"], first_index=first)
                else:
                    ctx.prove_digest_batch(w, rd, c, o["proof"], o["status"], o["sets"][b]["digest"], first_index=first)
                if vstream is None:
                    ctx.verify_bitmap_batch(o["proof"], c, u, o["result"], o["sets"][b]["bitmap"])
                else:
                    proved = torch.cuda.Event()
                    proved.record(pst)
                    vstream.wait_event(proved)
                    with torch.cuda.stream(vstream):
                        ctx_v.verify_bitmap_batch(o["proof"], c, u, o["result"], o["sets"][b]["bitmap"])
                        verified[slot] = torch.cuda.Event()
                        verified[slot].record(vstream)
            if nccl_mode or cyc == cycles - 1:
                if pstream1 is not None:
                    stream.wait_stream(pstream1)
                if vstream is not None:
                    stream.wait_stream(vstream)
            if nccl_mode:
                ev_ = torch.cuda.Event()
                ev_.record(stream)
                comm_stream.wait_event(ev_)
                with torch.cuda.stream(comm_stream):
                    dist.all_gather_into_tensor(gathered_all[b], summary_all[b])   # the only collective
                    gather_done[cyc] = torch.cuda.Event()
                    gather_done[cyc].record(comm_stream)
        if world > 1 and window is None and not args.no_gather:
            stream.wait_stream(comm_stream)
        return cycles

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # warm-up (direct launches; also warms NCCL), then capture the K-step region into ONE graph
    W = max(3, args.warmup)
    with torch.cuda.stream(stream):
        enqueue_region(W + ring)
    barrier()
    region_graph, launch_mode = None, "direct launches"
    if not args.no_graph and 2 * K + 64 < 30000:
        try:
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=stream):
                enqueue_region(K)
            region_graph = g
            launch_mode = (f"one CUDA graph per {K}-step region: {2 * K} kernels" +
                           (f" + {(K + ring - 1) // ring} NCCL all-gathers (one per {ring}-step cycle, overlapping the next cycle)" if world > 1 and window is None else "") +
                           ("; summaries stored into the peers' windows by the kernels (no collective)" if window is not None else "") +
                           ("; verify(k) on a second stream beside prove(k+1)" if vstream is not None else "") +
                           ("; provers alternate between two streams" if pstream1 is not None else ""))
        except Exception as e:   # pragma: no cover - capture not supported
            region_graph, launch_mode = None, f"direct launches (graph capture failed: {type(e).__name__}: {e})"
            torch.cuda.synchronize()

    def run_region():
        if region_graph is not None:
            region_graph.replay()
        else:
            enqueue_region(K)

    with torch.cuda.stream(stream):
        run_region()                                  # one untimed replay
    barrier()

    # ---- timed region: exactly K steps per repetition, device-timed on the launching stream, max over ranks per
    # repetition, median over repetitions
    reps = max(1, args.reps)
    sampler = ClockSampler(local)
    sampler.start()
    rep_ms = []
    def aligned_start():
        """After the barrier the ranks still leave it tens of microseconds apart, and the first collective of the region makes
        the early ones wait for the last: with a 2 ms region that skew is a few per cent of every rank's time.  All ranks
        therefore agree on one instant of the node's monotonic clock (the maximum of their proposals) and launch then."""
        if world == 1:
            return
        t = torch.tensor([time.monotonic() + 0.002], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        deadline = float(t.item())
        torch.cuda.synchronize()
        while time.monotonic() < deadline:
            pass

    for _ in range(reps):
        t_begin, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        aligned_start()
        with torch.cuda.stream(stream):
            t_begin.record(stream)
            run_region()
            t_end.record(stream)
        barrier()
        rep_ms.append(t_begin.elapsed_time(t_end))
    per_rank_ms = None
    if world > 1:
        t = torch.tensor(rep_ms, dtype=torch.float64, device=dev)
        allt = torch.empty((world, len(rep_ms)), dtype=torch.float64, device=dev)
        dist.all_gather_into_tensor(allt, t)
        per_rank_ms = [statistics.median(r_) for r_ in allt.tolist()]        # each rank's own median: shows a slow device
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        rep_ms = [float(x) for x in t.tolist()]
    ms_total = statistics.median(rep_ms)
    launches = KERNELS_PER_STEP * K * reps
    value = n * world * K / (ms_total * 1e-3)
    last_set = (((K + ring - 1) // ring) - 1) % 2       # summary set written by the last cycle of a region
    last_outputs = None
    if args.dump_outputs and rank == 0:
        # copied before the kernel timings below rewrite these buffers; written to DIR at the end
        o = outs[(K - 1) % ring]
        last_outputs = [t.clone() for t in (o["proof"], o["status"], o["result"], o["sets"][last_set]["bitmap"], o["sets"][last_set]["digest"])]
        torch.cuda.synchronize()

    # ---- per-kernel durations for the roofline: each kernel alone, back to back over the ring, CUDA events on its stream
    def time_kernel(fn, reps_):
        with torch.cuda.stream(stream):
            for k in range(3):
                fn(k % ring)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for k in range(reps_):
                fn(k % ring)
            e1.record(stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps_

    kreps = max(10, min(K, 100))
    prove_ms = time_kernel(lambda s_: ctx.prove_batch(ins[s_][0], ins[s_][1], ins[s_][2], proof=outs[s_]["proof"], status=outs[s_]["status"]), kreps)
    verify_ms = time_kernel(lambda s_: ctx.verify_batch(outs[s_]["proof"], ins[s_][2], ins[s_][3], result=outs[s_]["result"]), kreps)
    prove_digest_ms = time_kernel(lambda s_: ctx.prove_digest_batch(ins[s_][0], ins[s_][1], ins[s_][2], outs[s_]["proof"], outs[s_]["status"],
                                                                    outs[s_]["digest"], first_index=ins[s_][4]), kreps)
    verify_bitmap_ms = time_kernel(lambda s_: ctx.verify_bitmap_batch(outs[s_]["proof"], ins[s_][2], ins[s_][3], outs[s_]["result"],
                                                                      outs[s_]["bitmap"]), kreps)
    clocks = sampler.stop()
    if world > 1:
        # every rank samples its own device: a box that slows all its GPUs down when they run together shows up here
        mine = torch.tensor([float(clocks.get("sm_mhz") or 0), float(clocks.get("sm_mhz_min") or 0), float(clocks.get("power_w_median") or 0),
                             float(len(clocks.get("reasons") or []))], dtype=torch.float64, device=dev)
        allc = torch.empty((world, 4), dtype=torch.float64, device=dev)
        dist.all_gather_into_tensor(allc, mine)
        clocks["per_rank"] = [{"sm_mhz": r_[0], "sm_mhz_min": r_[1], "power_w_median": r_[2], "throttle_reasons": int(r_[3])} for r_ in allc.tolist()]
    # the same kernels with per-item curve arithmetic (PBH_ALGO_ARITH: fixed-base MSM commitments, Straus MSM, Miller loops,
    # final exponentiations): reported beside the default group-table algorithm, both bit-exact
    arith = None
    if args.algo == "table" and not args.no_arith:
        ctx.set_algo("arith")
        ap_ms = time_kernel(lambda s_: ctx.prove_batch(ins[s_][0], ins[s_][1], ins[s_][2], proof=outs[s_]["proof"], status=outs[s_]["status"]), 20)
        av_ms = time_kernel(lambda s_: ctx.verify_batch(outs[s_]["proof"], ins[s_][2], ins[s_][3], result=outs[s_]["result"]), 20)
        ctx.set_algo("table")
        arith = {"prove_ms": ap_ms, "verify_ms": av_ms, "proofs_per_s_per_gpu": n / (ap_ms * 1e-3), "verifies_per_s_per_gpu": n / (av_ms * 1e-3),
                 "prove_plus_verify_per_s_per_gpu": n / ((ap_ms + av_ms) * 1e-3)}

    # ---- sanity inside the bench: every timed item proved (status 0) and reached the pairing check
    o = outs[(K - 1) % ring]
    ok_status = int((o["status"] != 0).sum().item()) == 0
    accept = int((o["result"] == 1).sum().item())
    reached = int(((o["result"] == 1) | (o["result"] == 0)).sum().item())

    # ---- check (a): the N-rank result against ONE GPU.  Ring slot 0 of the N ranks is the contiguous global index range
    # [0, N n): rank 0 recomputes all of it alone and requires gathered bitmap == its bitmap and the sum of the gathered
    # digests == its digest.  Every rank also finds its own summary at its place in the gathered buffer.
    gather_ok = sharded_equals_single = single_ref = None
    if world > 1 and not args.no_gather:
        torch.cuda.synchronize()
        if window is not None:
            dist.barrier()                                   # every rank's kernels (and with them its stores into this window) are done
            torch.cuda.synchronize()
            g_ = win_sets[:, last_set].reshape(world, ring, row)
        else:
            g_ = gathered_all[last_set].view(world, ring, row)
        gather_ok = bool(torch.equal(g_[rank].reshape(-1), summary_all[last_set]))
        flag = torch.tensor([1 if gather_ok else 0], dtype=torch.int32, device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        gather_ok = bool(flag.item())
        if rank == 0:
            tot = world * n
            w1, r1, c1, u1 = ctx.generate_inputs(tot, first_index=0, seed=SEED, dist=pbh_b200.DIST_FULLPATH)
            p1 = torch.empty((27, tot), dtype=torch.uint8, device=dev)
            s1 = torch.empty((tot,), dtype=torch.uint8, device=dev)
            v1 = torch.empty((tot,), dtype=torch.uint8, device=dev)
            b1 = torch.empty((tot // 8,), dtype=torch.uint8, device=dev)
            d1 = torch.zeros((1,), dtype=torch.int64, device=dev)
            ctx.prove_digest_batch(w1, r1, c1, p1, s1, d1, first_index=0)
            ctx.verify_bitmap_batch(p1, c1, u1, v1, b1)
            ctx.sync()
            torch.cuda.synchronize()
            bits_n = g_[:, 0, :nb].reshape(-1)
            digs_n = g_[:, 0, nb:].contiguous().view(torch.int64).reshape(-1).tolist()
            sum_n = sum(int(x) & MASK64 for x in digs_n) & MASK64
            sharded_equals_single = bool(torch.equal(bits_n, b1)) and sum_n == (int(d1.item()) & MASK64)
            single_ref = (b1.cpu().numpy(), int(d1.item()) & MASK64)
            del w1, r1, c1, u1, p1, s1, v1, b1, d1

    # ---- the other input distribution of SURVEY.md 8(d): D_uniform (attempt 0 only; ~89 % of the items end in one of the
    # reference's panics).  Reported beside the headline, which is on D_fullpath where every item does all the work.
    d_uniform = None
    if not args.no_uniform:
        uw, ur, uc, uu = ctx.generate_inputs(n, first_index=0, seed=SEED, dist=pbh_b200.DIST_UNIFORM)
        u_proof = torch.empty((27, n), dtype=torch.uint8, device=dev)
        u_status = torch.empty((n,), dtype=torch.uint8, device=dev)
        u_result = torch.empty((n,), dtype=torch.uint8, device=dev)
        up_ms = time_kernel(lambda s_: ctx.prove_batch(uw, ur, uc, proof=u_proof, status=u_status), 20)
        uv_ms = time_kernel(lambda s_: ctx.verify_batch(u_proof, uc, uu, result=u_result), 20)
        hist = torch.bincount(u_status.to(torch.int64), minlength=6)[:6].tolist()
        d_uniform = {"prove_ms": up_ms, "verify_ms": uv_ms, "proofs_per_s_per_gpu": n / (up_ms * 1e-3),
                     "verifies_per_s_per_gpu": n / (uv_ms * 1e-3), "status_histogram_0_to_5": hist,
                     "accepted": int((u_result == 1).sum().item()), "items": n,
                     "note": "one batch (no ring): inputs and outputs of 2^20 items stay L2-resident; the kernels are issue-bound"}
        del uw, ur, uc, uu, u_proof, u_status, u_result

    # ---- Fiat-Shamir variants (SURVEY.md 8(f) row 1): same witnesses and blinders, challenges derived on the device
    fs = None
    if args.algo == "table" and not args.no_fs:
        f_proof = torch.empty((27, n), dtype=torch.uint8, device=dev)
        f_status = torch.empty((n,), dtype=torch.uint8, device=dev)
        f_result = torch.empty((n,), dtype=torch.uint8, device=dev)
        f_chal = torch.empty((6, n), dtype=torch.uint8, device=dev)
        fp_ms = time_kernel(lambda s_: ctx.prove_fs_batch(ins[s_][0], ins[s_][1], proof=f_proof, status=f_status, chal=f_chal), 10)
        produced = int((f_status == 0).sum().item())
        fv_ms = time_kernel(lambda s_: ctx.verify_fs_batch(f_proof, result=f_result, chal=f_chal), 10)
        fs = {"prove_fs_ms": fp_ms, "verify_fs_ms": fv_ms, "proofs_per_s_per_gpu": n / (fp_ms * 1e-3), "verifies_per_s_per_gpu": n / (fv_ms * 1e-3),
              "proofs_produced": produced, "accepted": int((f_result == 1).sum().item()), "items": n,
              "hash": "SHA-256, 5 compressions per proof and per verification"}
        del f_proof, f_status, f_result, f_chal

    # ---- end-to-end through the host-pointer C-ABI calls: every rank on its own device.  Three host-memory cases:
    #   lanes     page-locked buffers from pbh_host_alloc, pbh_prove_batch_async + pbh_verify_batch_async on two lanes: two
    #             batches in flight, verify(k) shares the full-duplex link with prove(k+1)           <- the headline `e2e`
    #   pinned    the same buffers through the two synchronous calls (round 1's number)
    #   pageable  ordinary numpy arrays (what a Rust Vec<u8> is), the two synchronous calls, staged copies
    e2e = None
    if args.e2e_steps != 0:
        host_in = [t.cpu().numpy() for t in ins[0][:4]]

        def alloc_set():
            hw = [ctx.host_alloc(a.shape) for a in host_in]
            for h, a in zip(hw, host_in):
                h[...] = a
            return dict(w=hw[0], r=hw[1], c=hw[2], u=hw[3], proof=ctx.host_alloc((27, n)), status=ctx.host_alloc((n,)), result=ctx.host_alloc((n,)))

        sets = [alloc_set() for _ in range(2)]
        ksteps = args.e2e_steps or max(6, min(K, 50))

        def timed(fn, steps_):
            barrier()
            t0 = time.perf_counter()
            for i in range(steps_):
                fn(i)
            ctx.sync()
            dt = time.perf_counter() - t0
            if world > 1:
                t = torch.tensor([dt], dtype=torch.float64, device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                dt = float(t.item())
            return dt

        def lanes_step(i):
            s_ = sets[i % 2]
            ctx.lane_sync(i % 2)                    # the batch that used these buffers two steps ago is complete
            ctx.prove_batch_async(i % 2, s_["w"], s_["r"], s_["c"], s_["proof"], s_["status"])
            ctx.verify_batch_async(i % 2, s_["proof"], s_["c"], s_["u"], s_["result"])

        def pinned_step(i):
            s_ = sets[0]
            ctx.prove_batch(s_["w"], s_["r"], s_["c"], proof=s_["proof"], status=s_["status"])
            ctx.verify_batch(s_["proof"], s_["c"], s_["u"], result=s_["result"])

        pg = dict(proof=np.empty((27, n), np.uint8), status=np.empty((n,), np.uint8), result=np.empty((n,), np.uint8))

        def pageable_step(i):
            ctx.prove_batch(host_in[0], host_in[1], host_in[2], proof=pg["proof"], status=pg["status"])
            ctx.verify_batch(pg["proof"], host_in[2], host_in[3], result=pg["result"])

        def fused_step(i):
            s_ = sets[0]
            ctx.prove_verify_batch(s_["w"], s_["r"], s_["c"], s_["u"], proof=s_["proof"], status=s_["status"], result=s_["result"])

        # packed wire format (include/pbh_b200.h): 16-byte prover inputs, 12-byte proofs, 4-byte challenge words - 32 bytes up
        # and 13 bytes down per proof + verification instead of 59 and 29
        packed_in0 = pbh_b200.pack_witness(*host_in)              # host-side format conversion, outside the timed region
        pk_sets = []
        L = max(2, min(4, args.e2e_lanes))               # batches in flight (PBH_LANES = 4)
        for _ in range(L):
            d_ = dict(pin=ctx.host_alloc_as(n, pbh_b200.PACKED_WITNESS), out=ctx.host_alloc_as(n, pbh_b200.PACKED_PROOF),
                      cu=ctx.host_alloc_as(n, "<u4"), res=ctx.host_alloc_as(n, np.uint8))
            d_["pin"][...] = packed_in0
            d_["cu"][...] = pbh_b200.pack_chal_u(host_in[2], host_in[3])
            pk_sets.append(d_)

        pgk = dict(pin=np.array(packed_in0), cu=pbh_b200.pack_chal_u(host_in[2], host_in[3]), out=np.zeros(n, pbh_b200.PACKED_PROOF), res=np.zeros(n, np.uint8))

        def pageable_packed_step(i):
            ctx.prove_packed(pgk["pin"], out=pgk["out"])
            ctx.verify_packed(pgk["out"], pgk["cu"], result=pgk["res"])

        def packed_lanes_step(i):
            s_ = pk_sets[i % L]
            ctx.lane_sync(i % L)
            ctx.prove_packed_async(i % L, s_["pin"], s_["out"])
            ctx.verify_packed_async(i % L, s_["out"], s_["cu"], s_["res"])

        def packed_fused_step(i):
            s_ = pk_sets[0]
            ctx.prove_verify_packed(s_["pin"], out=s_["out"], result=s_["res"])

        def packed_fused_lanes_step(i):
            s_ = pk_sets[i % L]
            ctx.lane_sync(i % L)
            ctx.prove_verify_packed_async(i % L, s_["pin"], s_["out"], s_["res"])

        for fn in (lanes_step, pinned_step, pageable_step, fused_step, packed_lanes_step, packed_fused_step, pageable_packed_step, packed_fused_lanes_step):
            for i in range(L + 1):
                fn(i)
            ctx.sync()
        for s_ in sets:
            s_["proof"][...] = 0; s_["status"][...] = 255; s_["result"][...] = 255
        for s_ in pk_sets:
            s_["out"].view(np.uint8)[...] = 0xEE; s_["res"][...] = 0xEE
        dt_packed = timed(packed_lanes_step, ksteps)
        ctx.set_option(pbh_b200.OPT_PROOF_RESIDENT, 0)      # the same two calls with the proofs uploaded again for the verifier
        for i in range(L):
            packed_lanes_step(i)
        ctx.sync()
        dt_packed_reupload = timed(packed_lanes_step, ksteps)
        ctx.set_option(pbh_b200.OPT_PROOF_RESIDENT, 1)
        ref_packed = pbh_b200.pack_proofs(outs[0]["proof"].cpu().numpy(), outs[0]["status"].cpu().numpy())
        ref_result0 = outs[0]["result"].cpu().numpy()
        packed_equal = all(np.array_equal(s_["out"], ref_packed) and np.array_equal(s_["res"], ref_result0) for s_ in pk_sets)
        dt_packed_fused = timed(packed_fused_step, ksteps)
        packed_equal = packed_equal and np.array_equal(pk_sets[0]["out"], ref_packed) and np.array_equal(pk_sets[0]["res"], ref_result0)
        for s_ in pk_sets:
            s_["out"].view(np.uint8)[...] = 0xEE; s_["res"][...] = 0xEE
        dt_packed_fused_lanes = timed(packed_fused_lanes_step, ksteps)
        packed_equal = packed_equal and all(np.array_equal(s_["out"], ref_packed) and np.array_equal(s_["res"], ref_result0) for s_ in pk_sets)
        dt_lanes = timed(lanes_step, ksteps)             # the library's default PBH_OPT_LANE_MODE
        lane_modes = {}
        for mode, what in ((0, "kernels read and write the host buffers in place"), (1, "copy-engine upload, in-place stores"),
                           (3, "copy engine both ways")):
            ctx.set_option(pbh_b200.OPT_LANE_MODE, mode)
            for i in range(2):
                lanes_step(i)
            ctx.sync()
            dtm = timed(lanes_step, ksteps)
            lane_modes[str(mode)] = {"value": n * world * ksteps / dtm, "ms_per_step": 1e3 * dtm / ksteps, "how": what}
        ctx.set_option(pbh_b200.OPT_LANE_MODE, 3)
        # every byte the lane pipeline produced equals the device-resident path of ring slot 0
        ref_proof, ref_status, ref_result = (outs[0][k].cpu().numpy() for k in ("proof", "status", "result"))
        e2e_equal = all(np.array_equal(s_["proof"], ref_proof) and np.array_equal(s_["status"], ref_status) and
                        np.array_equal(s_["result"], ref_result) for s_ in sets)
        dt_pinned = timed(pinned_step, ksteps)
        dt_pageable = timed(pageable_step, max(3, ksteps // 2))
        dt_pageable_packed = timed(pageable_packed_step, max(3, ksteps // 2))
        packed_equal = packed_equal and np.array_equal(pgk["out"], ref_packed) and np.array_equal(pgk["res"], ref_result0)
        ctx.set_option(pbh_b200.OPT_HOST_STAGE, 0)
        pageable_step(0)
        dt_pageable_driver = timed(pageable_step, 3)
        ctx.set_option(pbh_b200.OPT_HOST_STAGE, 1)
        e2e_equal = e2e_equal and np.array_equal(pg["proof"], ref_proof) and np.array_equal(pg["result"], ref_result)
        dt_fused = timed(fused_step, ksteps)
        per = lambda dt, st: {"value": n * world * st / dt, "ms_per_step": 1e3 * dt / st}
        # Headline: every input of both calls is read from the host buffers (PBH_OPT_PROOF_RESIDENT 0), i.e. the proofs cross PCIe
        # twice, down as prove's output and up again as verify's input.  The library's default (the verifier reads the device-resident
        # copy of the proofs the prove call on the same lane has just produced) is reported beside it.
        e2e = {"value": n * world * ksteps / dt_packed_reupload, "unit": UNIT, "h2d_bytes_per_step": n * (16 + 12 + 4) * world,
               "d2h_bytes_per_step": n * (12 + 1) * world, "steps": ksteps, "ms_per_step": 1e3 * dt_packed_reupload / ksteps,
               "api": f"pbh_prove_packed_async + pbh_verify_packed_async on {L} lanes ({L} batches in flight), pbh_lane_sync before a lane's buffers are reused; "
                      "the two reference calls, Plonk::prove then Plonk::verify, on the packed wire format",
               "wire_format": "packed records (include/pbh_b200.h): prove 16 B in / 12 B out per item, verify 12 + 4 B in / 1 B out; the proofs cross PCIe twice "
                              "(down from prove, up into verify: PBH_OPT_PROOF_RESIDENT 0 for this measurement); unpacking and packing run on the GPU inside "
                              "the timed region",
               "packed_lanes_proofs_resident": dict(per(dt_packed, ksteps), h2d_bytes_per_step=n * (16 + 4) * world, d2h_bytes_per_step=n * 13 * world,
                                                    api="the same two calls with the library's default PBH_OPT_PROOF_RESIDENT 1: the verify call names the very buffer the prove "
                                                        "call on the same lane is still filling (no synchronisation in between, so by the lane contract the caller cannot have "
                                                        "touched it), and the verifier reads the device-resident copy of those proofs instead of uploading them again; the "
                                                        "proofs still travel to the host as prove's output; results identical"),
               "host_memory": "page-locked (pbh_host_alloc), whole-batch copy-engine transfers both ways on the lane's stream",
               "numa_node_of_device": ctx.numa_node,
               "timing": "host wall clock around the C-ABI calls up to the final pbh_ctx_sync, max over ranks",
               "bytes_equal_device_path": bool(e2e_equal and packed_equal),
               "packed_equals_pack_of_device_path": bool(packed_equal),
               "byte_plane_lanes": dict(per(dt_lanes, ksteps), h2d_bytes_per_step=n * (26 + 33) * world, d2h_bytes_per_step=n * (28 + 1) * world,
                                        api="pbh_prove_batch_async + pbh_verify_batch_async on two lanes, one byte per field element (default PBH_OPT_LANE_MODE 3)"),
               "packed_fused_call": dict(per(dt_packed_fused, ksteps), h2d_bytes_per_step=n * 16 * world, d2h_bytes_per_step=n * 13 * world,
                                         api="pbh_prove_verify_packed (extension: the proof does not cross PCIe twice)"),
               "packed_fused_call_lanes": dict(per(dt_packed_fused_lanes, ksteps), h2d_bytes_per_step=n * 16 * world, d2h_bytes_per_step=n * 13 * world,
                                               api=f"pbh_prove_verify_packed_async on {L} lanes (extension)"),
               "lane_modes": lane_modes,
               "two_sync_calls_pinned": dict(per(dt_pinned, ksteps), api="pbh_prove_batch then pbh_verify_batch, page-locked buffers"),
               "two_sync_calls_pageable": dict(per(dt_pageable, max(3, ksteps // 2)), api="pbh_prove_batch then pbh_verify_batch, pageable numpy buffers (what a plain Vec<u8> is): "
                                               "staged chunks through page-locked mirrors filled by the library's copy threads (PBH_OPT_HOST_STAGE 1)",
                                               driver_staging=dict(per(dt_pageable_driver, 3), api="the same with PBH_OPT_HOST_STAGE 0: the driver stages the pageable copies")),
               "two_sync_calls_pageable_packed": dict(per(dt_pageable_packed, max(3, ksteps // 2)), api="pbh_prove_packed then pbh_verify_packed, pageable numpy buffers"),
               "fused_call": dict(per(dt_fused, ksteps), h2d_bytes_per_step=n * 27 * world, d2h_bytes_per_step=n * 29 * world,
                                  api="pbh_prove_verify_batch (extension: the proof does not cross PCIe twice)")}
        for s_ in sets + pk_sets:
            for a in s_.values():
                ctx.host_free(a)
        del sets, pg, pk_sets, pgk

    # ---- BASELINE.json configs[4]: 2^28 witnesses in total, sharded over the N ranks (strong scaling), ONE all-gather of
    # the verdict bitmaps + digests at the end of each pass
    config4 = None
    if not args.no_config4:
        tot4 = 1 << args.config4_log2
        n4 = tot4 // world
        first4 = rank * n4
        w4, r4, c4, u4 = ctx.generate_inputs(n4, first_index=first4, seed=SEED, dist=pbh_b200.DIST_FULLPATH)
        p4 = torch.empty((27, n4), dtype=torch.uint8, device=dev)
        s4 = torch.empty((n4,), dtype=torch.uint8, device=dev)
        v4 = torch.empty((n4,), dtype=torch.uint8, device=dev)
        sum4 = torch.zeros(n4 // 8 + 8, dtype=torch.uint8, device=dev)
        gat4 = torch.empty(world * (n4 // 8 + 8), dtype=torch.uint8, device=dev) if world > 1 else None

        def pass4():
            ctx.prove_digest_batch(w4, r4, c4, p4, s4, sum4[n4 // 8:].view(torch.int64), first_index=first4)
            ctx.verify_bitmap_batch(p4, c4, u4, v4, sum4[:n4 // 8])
            if world > 1:
                dist.all_gather_into_tensor(gat4, sum4)

        steps4 = 3
        with torch.cuda.stream(stream):
            pass4()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            e0.record(stream)
            for _ in range(steps4):
                pass4()
            e1.record(stream)
        barrier()
        ms4 = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms4], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms4 = float(t.item())
        ok4 = int((s4 != 0).sum().item()) == 0 and int(((v4 != 0) & (v4 != 1)).sum().item()) == 0
        if world > 1:
            ok4 = ok4 and bool(torch.equal(gat4.view(world, -1)[rank], sum4))
        config4 = {"workload": f"BASELINE.json configs[4]: end-to-end prove+verify of 2^{args.config4_log2} witnesses sharded over {world} GPU(s), NCCL all-gather of verdict bitmaps + digests",
                   "items_total": tot4, "items_per_gpu": n4, "passes": steps4, "ms_per_pass": ms4 / steps4, "value": tot4 * steps4 / (ms4 * 1e-3),
                   "unit": UNIT, "scaling": "strong", "all_proved_and_reached_pairing": bool(ok4),
                   "accepted_on_rank0": int((v4 == 1).sum().item())}
        del w4, r4, c4, u4, p4, s4, v4, sum4, gat4
        torch.cuda.empty_cache()

    def finish():
        """Multi-rank teardown: final barrier, then leave without destroy_process_group() — tearing the communicator down
        while CUDA graphs that captured its collectives are alive was observed to hang."""
        if world > 1:
            torch.cuda.synchronize()
            dist.barrier()
            sys.stdout.flush()
            sys.stderr.flush()
            os._exit(0)

    if rank != 0:
        finish()
        return

    # ---- pipe peaks measured in THIS run (independent register chains, no memory traffic)
    hbm_peak, peak_src = measured_peaks()
    int32 = {}
    try:
        names = ["imad", "lop3_iadd3", "half_imad_half_alu", "ffma", "hfma2_instr", "dp4a_instr", "imad_hi_iadd", "half_ffma_half_imad", "ffma_3reg", "imad_3reg",
                 "ffma2_3pair_instr", "ffma2_bcast_instr", "shf"]
        int32 = {f"{nm}_thread_ops_per_s": ctx.measure_int32_peak(i) for i, nm in enumerate(names)}
    except Exception as e:  # pragma: no cover
        int32 = {"error": str(e)}
    sm_count = torch.cuda.get_device_properties(dev).multi_processor_count
    sm_hz = 1e6 * float(clocks.get("sm_mhz") or clocks.get("sm_max_mhz") or 1965)
    peaks = {"hbm_gbs": hbm_peak,
             # one warp instruction per clock per SM sub-partition: 4 x 32 thread instructions per clock per SM at the SM clock sampled under load
             "issue_thread_instr_per_s": sm_count * 128 * sm_hz,
             "fma_thread_ops_per_s": int32.get("ffma_thread_ops_per_s"),       # FFMA on both FMA pipes (measured above)
             "imad_thread_ops_per_s": int32.get("imad_thread_ops_per_s"),      # IMAD issues on the heavy FMA pipe only
             "alu_thread_ops_per_s": int32.get("shf_thread_ops_per_s")}        # SHF = one ALU-pipe instruction per chain step
    instr = instr_table()
    # the two kernels of the timed step first (prover with its fused digest, verifier with its fused bitmap), then the same
    # kernels without the fused summaries
    kernels_rf = [roofline_entry(("prove_f32_tma_kernel<TABLE>" if args.algo == "table" else "prove_f32_tma_kernel<ARITH>") + " + fused digest (the step's prover)",
                                 "prove_table_digest" if args.algo == "table" else "prove_arith", prove_digest_ms, n, 54, peaks, instr),
                  roofline_entry(("verify_tma_kernel<TABLE>" if args.algo == "table" else "verify_tma_kernel<ARITH>") + " + fused bitmap (the step's verifier)",
                                 "verify_table_bitmap" if args.algo == "table" else "verify_arith", verify_bitmap_ms, n, 34, peaks, instr),
                  roofline_entry("prove_f32_tma_kernel<TABLE>" if args.algo == "table" else "prove_f32_tma_kernel<ARITH>",
                                 "prove_table" if args.algo == "table" else "prove_arith", prove_ms, n, 54, peaks, instr),
                  roofline_entry("verify_tma_kernel<TABLE>" if args.algo == "table" else "verify_tma_kernel<ARITH>",
                                 "verify_table" if args.algo == "table" else "verify_arith", verify_ms, n, 34, peaks, instr)]
    if arith:
        kernels_rf.append(roofline_entry("prove_f32_tma_kernel<ARITH>", "prove_arith", arith["prove_ms"], n, 54, peaks, instr))
        kernels_rf.append(roofline_entry("verify_tma_kernel<ARITH>", "verify_arith", arith["verify_ms"], n, 34, peaks, instr))
    if fs:
        kernels_rf.append(roofline_entry("prove_fs_kernel<TABLE>", "prove_fs", fs["prove_fs_ms"], n, 49 + 6, peaks, instr))
        kernels_rf.append(roofline_entry("verify_fs_kernel<TABLE>", "verify_fs", fs["verify_fs_ms"], n, 27 + 1 + 6, peaks, instr))
    if d_uniform:
        kernels_rf.append(roofline_entry("prove_f32_tma_kernel<TABLE> on D_uniform", "prove_table_uniform", d_uniform["prove_ms"], n, 54, peaks, instr))
    dom = max(kernels_rf[:2], key=lambda e: e["ms"])          # the dominant kernel of the step
    traffic = None
    try:   # per-launch DRAM bytes of the dominant kernel from the committed ncu capture (profiles/): STATIC
        with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as f:
            tj = json.load(f)
        ent = tj.get("prove_f32_tma_kernel") if (args.algo == "table" and dom is kernels_rf[0]) else None
        if ent and n == N_PER_GPU:
            traffic = ent["dram_read_bytes"] + ent["dram_write_bytes"]
    except Exception:
        traffic = None
    if dom["bound"] == "hbm":
        rf_main = {"bound": "hbm", "achieved": dom["hbm"]["achieved_GBps"], "peak": hbm_peak, "unit": "GB/s", "frac": dom["hbm"]["frac"]}
    else:
        b_ = dom[dom["bound"]]
        rf_main = {"bound": dom["bound"], "achieved": b_["achieved_thread_instr_per_s"] / 1e12, "peak": b_["peak_thread_instr_per_s"] / 1e12,
                   "unit": "T thread-instr/s", "frac": b_["frac"]}

    # ---- N = 1 only: BASELINE.json configs[2] (16 M-proof verifier) and configs[3] (kernel sweeps, 2^24 .. 2^28 items)
    config2 = sweeps = None
    if world == 1 and not args.no_config2:
        n2 = 1 << 24
        w2, r2, c2, u2 = ctx.generate_inputs(n2, first_index=0, seed=SEED, dist=pbh_b200.DIST_FULLPATH)
        p2, s2 = ctx.prove_batch(w2, r2, c2)
        v2 = torch.empty((n2,), dtype=torch.uint8, device=dev)
        v2a = torch.empty((n2,), dtype=torch.uint8, device=dev)
        ms2 = time_kernel(lambda s_: ctx.verify_batch(p2, c2, u2, result=v2), 5)
        ctx.set_algo("arith")
        ms2a = time_kernel(lambda s_: ctx.verify_batch(p2, c2, u2, result=v2a), 3)
        ctx.set_algo("table")
        config2 = {"workload": "BASELINE.json configs[2]: batched verifier, 2^24 proofs, one B200", "items": n2, "verify_ms": ms2,
                   "verifies_per_s": n2 / (ms2 * 1e-3), "hbm_frac": 34.0 * n2 / (ms2 * 1e-3) / 1e9 / hbm_peak,
                   "arith_verify_ms": ms2a, "arith_verifies_per_s": n2 / (ms2a * 1e-3), "table_equals_arith": bool(torch.equal(v2, v2a)),
                   "accepted": int((v2 == 1).sum().item()), "all_reached_pairing": int(((v2 != 0) & (v2 != 1)).sum().item()) == 0}
        del w2, r2, c2, u2, p2, s2, v2, v2a
        torch.cuda.empty_cache()
        # the verifier against its ceilings at this size: a 2^20-item launch carries ~9 us of fixed cost (launch, first tile, tail)
        kernels_rf.append(roofline_entry("verify_tma_kernel<TABLE> at 2^24 items (configs[2])", "verify_table", ms2, n2, 34, peaks, instr))
        kernels_rf.append(roofline_entry("verify_tma_kernel<ARITH> at 2^24 items (configs[2])", "verify_arith", ms2a, n2, 34, peaks, instr))
    if world == 1 and not args.no_sweeps:
        import bench_sweeps
        sweeps = []
        for lg in [int(x) for x in args.sweep_log2.split(",") if x]:
            sweeps.append({"log2_items": lg, "kernels": bench_sweeps.run_sweeps(ctx, lg, reps=5 if lg >= 27 else 10, hbm_peak=hbm_peak, peaks=peaks)})
            torch.cuda.empty_cache()

    # ---- check (b) and the CPU baseline: the exact 2^20-item batch of ring slot 0 replayed through the oracle, byte for byte
    cpu = None
    oracle_full = generator_sample_ok = None
    if world >= 1 and not args.no_cpu:
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import oracle as O
        threads = max(1, O.hardware_threads())
        h_w, h_r, h_c, h_u = (t.cpu().numpy() for t in ins[0][:4])
        t0 = time.perf_counter()
        o_proof, o_status = O.prove_batch(h_w, h_r, h_c, threads=threads)
        o_result = O.verify_batch(o_proof, h_c, h_u, threads=threads, want_gt=False)
        dt_full = time.perf_counter() - t0
        if isinstance(o_result, tuple):
            o_result = o_result[0]
        oracle_full = (np.array_equal(o_proof, outs[0]["proof"].cpu().numpy()) and np.array_equal(o_status, outs[0]["status"].cpu().numpy())
                       and np.array_equal(o_result, outs[0]["result"].cpu().numpy()))
        # the device generator against the oracle's on a prefix of the same slot (the oracle needs ~20 attempts per item)
        g_w, g_r, g_c, g_u = O.generate_inputs(4096, first_index=ins[0][4], seed=SEED, dist=1, threads=threads)[:4]
        generator_sample_ok = bool(np.array_equal(g_w, h_w[:, :4096]) and np.array_equal(g_r, h_r[:, :4096]) and
                                   np.array_equal(g_c, h_c[:, :4096]) and np.array_equal(g_u, h_u[:4096]))
        if world == 1:
            v1, dt1 = cpu_leg(20000, 1)
            cpu = {"value": n / dt_full, "unit": UNIT, "cores": threads, "kind": "port", "cpu_model": cpu_model(), "nproc": os.cpu_count(),
                   "sample": f"the whole 2^20-item D_fullpath batch of ring slot 0 (the batch the GPU is checked against), prove then verify, C++ restatement of the reference (oracle/), {threads} threads, {dt_full:.1f} s",
                   "single_thread": {"value": v1, "cores": 1, "sample": f"20000 items, {dt1:.1f} s"}}

    # ---- the same sharded pass from ONE process through the C ABI's multi-device entry points (pbh_multi_*: one stream per
    # device, ncclCommInitAll, one in-library ncclAllGather): rank 0 drives all the GPUs of the job while the other ranks wait
    # at the final barrier.  Checked against what one GPU computed for the same global index range.
    multi = None
    try:
        if single_ref is None:
            bm0 = ctx.pack_verdicts(outs[0]["result"])
            single_ref = (bm0.cpu().numpy(), int(ctx.digest(outs[0]["proof"], first_index=ins[0][4]).item()) & MASK64)
            ctx.sync()
        with pbh_b200.MultiContext(world, algo=args.algo) as mc:
            mc.prove_verify_sharded(world * n, first_index=0, seed=SEED)          # warm-up (allocations, NCCL channels)
            runs = [mc.prove_verify_sharded(world * n, first_index=0, seed=SEED) for _ in range(5)]
            best = min(runs, key=lambda r_: r_["ms"])
            multi = {"api": "pbh_multi_create + pbh_multi_prove_verify_sharded (generate -> prove -> verify on every device, one ncclAllGather of bitmaps + digests)",
                     "n_dev": mc.device_count, "items_total": world * n, "ms_per_pass_incl_generation": best["ms"],
                     "accepted": best["accepted"], "equals_single_gpu": bool(np.array_equal(best["bitmap"], single_ref[0]) and best["total_digest"] == single_ref[1])}
    except Exception as e:   # pragma: no cover - reported, not fatal for the headline
        multi = {"error": f"{type(e).__name__}: {e}"}
    if last_outputs is not None:
        dump_outputs(args.dump_outputs, *last_outputs)

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "fp32/int32 registers holding exact F_17 / F_101 residues (u8 on the wire)", "data": "synthetic",
        "config": {"workload": WORKLOAD, "items_per_gpu_per_step": n, "algo": args.algo, "distribution": "D_fullpath seed 0xB200",
                   "l2": f"ring of {ring} distinct input/output batches ({ring * n * 88 / 1e6:.0f} MB) cycled, larger than the 126 MB L2",
                   "parallelism": f"shard x{world}, all-gather of verdict bitmaps + digests" if world > 1 else "single GPU",
                   "collective": ({"window": "peer windows: the verifier / prover kernels store bitmap / digest into every peer's buffer over NVLink (pbh_window_*); "
                                             "no collective call in the timed region; the NCCL all-gather is timed in config4_256m_sharded",
                                   "nccl": "NCCL all_gather_into_tensor, one per ring cycle, on a side stream"}[collective] if world > 1 else None),
                   "timing": f"median of {reps} repetitions of the exactly-{K}-step region (CUDA events on the launching stream, max over ranks per repetition)"},
        "timed_region_ms": {"median": ms_total, "all_repetitions": rep_ms, "median_of_each_rank": per_rank_ms},
        "clocks": clocks,
        "e2e": e2e,
        "gpu_launches": launches,
        "roofline": {"bound": rf_main["bound"], "achieved": rf_main["achieved"], "peak": rf_main["peak"], "unit": rf_main["unit"],
                     "frac": rf_main["frac"], "traffic": traffic, "kernel": dom["kernel"],
                     "traffic_source": "profiles/roofline_traffic.json (ncu --set full; STATIC, not measured in this run)",
                     "hbm_frac": dom["hbm"]["frac"], "hbm_achieved_GBps": dom["hbm"]["achieved_GBps"], "hbm_peak_GBps": hbm_peak, "peak_source": peak_src,
                     "algorithmic_bytes_per_item": dom["hbm"]["algorithmic_bytes_per_item"],
                     "how": "frac = max over {HBM bytes, issue slots, FMA pipe, ALU pipe} of achieved / peak for the step's dominant kernel; times, clocks "
                            "and pipe peaks are measured in this run, instructions per item are the committed ncu counts (profiles/instr_per_item.json)",
                     "peaks_measured_in_this_run": peaks, "kernels": kernels_rf,
                     # SURVEY.md 8(d): the work the reference's algorithm does per item, in its own modular operations
                     "reference_equivalent_modops_per_item": {"prove": 5170 + 3719 + 318, "verify": 3552 + 1309 + 256},
                     "reference_equivalent_modops_per_s": value * (5170 + 3719 + 318 + 3552 + 1309 + 256)},
        "launch": launch_mode,
        "kernels": {"how": "each kernel alone, back to back over the ring, CUDA events on the context's stream",
                    "prove_ms": prove_ms, "verify_ms": verify_ms, "prove_with_digest_ms": prove_digest_ms,
                    "verify_with_bitmap_ms": verify_bitmap_ms, "proofs_per_s_per_gpu": n / (prove_ms * 1e-3),
                    "verifies_per_s_per_gpu": n / (verify_ms * 1e-3)},
        "arith_algo_kernels": arith,
        "fiat_shamir_kernels": fs,
        "d_uniform_kernels": d_uniform,
        "config2_verifier_16m": config2,
        "config4_256m_sharded": config4,
        "sweeps": sweeps,
        "single_process_multi_device": multi,
        "int32_peak": int32,
        "cpu_baseline": cpu,
        "check": {"all_status_ok": ok_status, "accepted": accept, "reached_pairing": reached, "items": n,
                  "oracle_full_batch": oracle_full, "generator_prefix_equals_oracle": generator_sample_ok,
                  "gathered_summaries_ok": gather_ok, "sharded_equals_single": sharded_equals_single},
    }
    if args.no_gather:
        line["INVALID"] = "--no-gather: diagnostic run without the exchange of the summaries"
    sys.stdout.flush()
    os.write(json_fd, (json.dumps(line) + "\n").encode())
    finish()


if __name__ == "__main__":
    main()
