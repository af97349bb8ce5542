#!/usr/bin/env python
"""bench.py -- CTC loss forward+backward throughput on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W

One "step" = one pass of the hot path (loss forward + gradient) over one batch of synthetic
input: BASELINE.json configs[1], CTC B=64, T=800, V=3500, label length <= 80, variable lengths,
PER GPU (weak scaling: N GPUs = configs[3]'s B=512 at N=8, batch-sharded, the loss summed over the ranks by one small asynchronous all-reduce per four steps).

Printed JSON (rank 0, one line):
  value     padded utterance-frames/s = N*B*T*K / max-over-ranks device time, inputs resident in HBM
  e2e       the same through the public API with HOST (pinned) buffers: activations H2D, gradient and
            loss D2H inside the timed region
  roofline  dominant kernel (the fused gradient kernel: 2/3 of the algorithmic bytes) against the
            measured HBM copy bandwidth in MEASURED_PEAKS.json; whole-step figure in "step_roofline"
  cpu_baseline  the oracle's C port (oracle/ctc_oracle.c, OpenMP) on this box's host cores, rank 0, N=1

--impl reference times the CPU implementation alone (the reference itself is Python/Chainer and
cannot travel to the GPU box, so this is the oracle port -- kind "port").

--dump-outputs DIR (rank 0) writes what the headline path returned in its last timed step: DIR/loss.npy (the float32
scalar loss) and DIR/grad_rows.npy (float32 (DUMP_FRAMES, V): the gradient rows of the frames dump_frames() picks with
a fixed seed out of the (T,B,V) gradient, which at 717 MB is too large to keep whole).  The inputs are seeded, so two
builds run with the same arguments can be compared output for output.
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOAD = {"B": 64, "T": 800, "V": 3500, "L": 80}
METRIC = "CTC fwd+bwd utterance-frames/sec at B=64,T=800,V=3500"
UNIT = "frames/s"
FALLBACK_HBM_GBS = 6650.0
REF_SAMPLE_UTTS = 4        # utterances of the workload the reference's NumPy path processes per timed step (~1.5 s)
DUMP_FRAMES = 2048         # gradient rows --dump-outputs keeps: 2048 * V * 4 bytes = 28.7 MB


def config_dict(world):
    """`config` of the JSON line: identical in both arms (the driver compares them)."""
    B = WORKLOAD["B"]
    return {"workload": "CTC fwd+bwd B=64,T=800,V=3500,L<=80 per GPU, variable lengths "
                        "(BASELINE configs[1]; N GPUs = batch-sharded configs[3])",
            "global_batch": world * B, "parallelism": "batch-sharded dp%d, loss all-reduce (asynchronous, one per 4 steps)" % world,
            "layout": "(T,B,V) float32", "l2": "inputs (717 MB) and outputs exceed the 126 MB L2; no flush needed"}


def synth():
    return importlib.import_module("chainer-speech-recognition_b200.synth")


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback"


def profiled_traffic(kernel):
    """DRAM bytes (read + write) per launch of `kernel` from the committed `ncu --set full` capture of this workload
    (profiles/r1_ncu_full_summary.json, written by tools/ncu_summary.py); None if there is no capture."""
    try:
        names = [n for n in ("r2_ncu_full_summary.json", "r1_ncu_full_summary.json")
                 if os.path.exists(os.path.join(ROOT, "profiles", n))]
        with open(os.path.join(ROOT, "profiles", names[0])) as f:
            for k in json.load(f):
                if kernel in k["kernel"]:
                    def to_bytes(v):
                        num, unit = v.split()
                        return float(num) * {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}[unit]
                    return int(to_bytes(k["dram__bytes_read.sum"]) + to_bytes(k["dram__bytes_write.sum"]))
    except Exception:
        pass
    return None


class ClockSampler(object):
    """nvidia-smi clocks + throttle reasons sampled while the timed region runs."""
    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.FIELDS,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.lines:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1]))
            except ValueError:
                continue
            for n, v in zip(names, parts[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        # "under load": keep the upper half of the samples (idle samples before/after the region read low)
        sm_sorted = sorted(sm)
        load = sm_sorted[len(sm_sorted) // 2:] if sm_sorted else []
        return {"sm_mhz": float(np.median(load)) if load else None,
                "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm)}


def host_threads():
    """All the host threads this process may use (torchrun exports OMP_NUM_THREADS=1, which is not what the CPU arm
    should be limited to)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return max(1, os.cpu_count() or 1)


def algorithmic_bytes(V, in_len, B, T):
    """SURVEY.md 8d: read activations once (softmax), once more (gradient), write the gradient once."""
    valid = int(np.sum(in_len))
    k1 = 4 * V * valid                       # kernel 1: one read of the valid frames
    k3 = 4 * V * valid + 4 * V * B * T       # kernel 3: re-read valid frames + write every frame
    return k1, k3


def dump_frames(T, B):
    """Flat frame indices t * B + b (ascending) of the gradient rows --dump-outputs writes: a fixed seeded sample."""
    return np.sort(np.random.RandomState(0).choice(T * B, min(DUMP_FRAMES, T * B), replace=False))


def sample_outputs(loss, grad):
    """Device copies of a step's outputs that --dump-outputs keeps: the loss and the dump_frames() rows of the gradient."""
    import torch
    T, B, V = grad.shape
    rows = torch.from_numpy(dump_frames(T, B)).to(grad.device)
    return {"loss": loss.detach().clone(), "grad_rows": grad.detach().reshape(T * B, V).index_select(0, rows)}


def write_outputs(dirname, outputs):
    os.makedirs(dirname, exist_ok=True)
    for name, t in outputs.items():
        np.save(os.path.join(dirname, name + ".npy"), t.cpu().numpy().astype(np.float32))


def port_baseline(prob, threads, budget_s=6.0):
    """Oracle C port (banded restatement of the reference algorithm, float64, OpenMP), forward+backward over the WHOLE
    64-utterance workload, repeated for ~budget_s seconds."""
    from oracle import c_oracle
    args = (0, prob["x"], prob["labels"], None, prob["input_length"], prob["label_length"], prob["blank"])
    c_oracle.run(*args, nthreads=threads)                      # warm-up: page in, spin up the thread pool
    t0 = time.perf_counter()
    c_oracle.run(*args, nthreads=threads)
    one = time.perf_counter() - t0
    reps = max(1, min(200, int(budget_s / max(one, 1e-3))))
    t0 = time.perf_counter()
    for _ in range(reps):
        c_oracle.run(*args, nthreads=threads)
    dt = time.perf_counter() - t0
    T, B = prob["x"].shape[0], prob["x"].shape[1]
    return B * T * reps / dt, dt, reps


class ReferenceSample(object):
    """The reference's own implementation (asr/loss/gram_ctc.py, unmodified, NumPy path under oracle/ref_stub.py;
    every bigram id -1 = plain CTC, SURVEY.md 8c) on the first REF_SAMPLE_UTTS utterances of the workload.  One step =
    GramCTC.forward + GramCTC.backward, exactly what a training step of the reference runs.  Its cost is linear in the
    number of utterances (every op is per utterance, SURVEY.md 8e), so frames/s of the sample is frames/s of the
    workload.  Available wherever the reference's files are (oracle/ref_stub.py: REFERENCE_ROOT)."""

    def __init__(self, prob, n=REF_SAMPLE_UTTS):
        from oracle import ref_stub
        self.ok = ref_stub.available()
        if not self.ok:
            return
        self.ref = ref_stub.load()
        self.n = n
        T = prob["x"].shape[0]
        xs = tuple(np.ascontiguousarray(prob["x"][t, :n]) for t in range(T))
        lab = np.ascontiguousarray(prob["labels"][:n], np.int32)
        self.inputs = (np.asarray(prob["input_length"][:n], np.int32), np.asarray(prob["label_length"][:n], np.int32),
                       lab, np.full_like(lab, -1)) + xs
        self.frames = n * T
        self.threads = 1                                     # NumPy elementwise/reduction code: one thread

    def step(self):
        f = self.ref.GramCTC(0, "mean")                      # fresh object: backward mutates the saved softmax (:290-296)
        t0 = time.perf_counter()
        loss = f.forward(self.inputs)[0]
        t1 = time.perf_counter()
        f.backward(self.inputs, (np.float32(1.0),))
        t2 = time.perf_counter()
        return float(loss), t1 - t0, t2 - t1

    def describe(self):
        return ("the reference itself: asr/loss/gram_ctc.py unmodified, NumPy path (bigram ids -1 = plain CTC), "
                "forward+backward of the first %d of the 64 utterances per step; cost is linear in utterances" % self.n)


def torch_cpu_ctc(prob, steps=2):
    """Secondary CPU line (BASELINE.md section 3): torch.nn.functional.ctc_loss on the host, float32, all threads."""
    import torch
    threads = host_threads()
    torch.set_num_threads(threads)
    x = torch.tensor(prob["x"], requires_grad=True)
    lab = torch.tensor(prob["labels"], dtype=torch.long)
    il = torch.tensor(prob["input_length"], dtype=torch.long)
    ll = torch.tensor(prob["label_length"], dtype=torch.long)

    def one():
        x.grad = None
        lp = torch.log_softmax(x, dim=2)
        torch.nn.functional.ctc_loss(lp, lab, il, ll, blank=0, reduction="none").mean().backward()
    one()
    t0 = time.perf_counter()
    for _ in range(steps):
        one()
    dt = (time.perf_counter() - t0) / steps
    T, B = prob["x"].shape[0], prob["x"].shape[1]
    return {"value": B * T / dt, "unit": UNIT, "threads": threads, "ms_per_step": 1e3 * dt,
            "what": "torch.nn.functional.ctc_loss + log_softmax, CPU float32, whole workload (cross-check, not the reference)"}


def run_reference_arm(args, rank, world, emit):
    """--impl reference: the reference's own CPU implementation alone, rank 0 only."""
    if rank != 0:
        return
    W = WORKLOAD
    prob = synth().ctc_problem(W["B"], W["T"], W["V"], W["L"], seed=0)
    ref = ReferenceSample(prob)
    threads = host_threads()
    if ref.ok:
        for _ in range(max(min(args.warmup, 2), 1)):
            ref.step()
        fwd = bwd = 0.0
        for _ in range(args.steps):
            _, f, b = ref.step()
            fwd += f; bwd += b
        dt = fwd + bwd
        value = ref.frames * args.steps / dt
        kind, cores, sample, dtype = "reference", ref.threads, ref.describe(), "f32"
        extra = {"fwd_ms": 1e3 * fwd / args.steps, "bwd_ms": 1e3 * bwd / args.steps}
    else:                                                     # no reference files on this machine: the banded C port
        from oracle import c_oracle
        xargs = (0, prob["x"], prob["labels"], None, prob["input_length"], prob["label_length"], prob["blank"])
        for _ in range(max(args.warmup, 1)):
            c_oracle.run(*xargs, nthreads=threads)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            c_oracle.run(*xargs, nthreads=threads)
        dt = time.perf_counter() - t0
        value = W["B"] * W["T"] * args.steps / dt
        kind, cores, dtype = "port", threads, "f64"
        sample = "oracle C port (oracle/ctc_oracle.c, float64, OpenMP x%d), all 64 utterances of the workload per step" % threads
        extra = {}
    out = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": dtype, "data": "synthetic",
        "config": config_dict(max(args.gpus, 1)),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "host_cores": threads,
    }
    out.update(extra)
    if ref.ok:                                               # the faster CPU restatements beside it, for context
        v, secs, reps = port_baseline(prob, threads, budget_s=4.0)
        out["port_baseline"] = {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
                                "sample": "oracle C port (banded O(T*N) restatement, float64, OpenMP x%d), whole workload, %d passes" % (threads, reps)}
        try:
            out["torch_cpu_ctc"] = torch_cpu_ctc(prob)
        except Exception as exc:
            sys.stderr.write("bench.py: torch CPU line skipped (%s)\n" % exc)
    emit(out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="do not also time the step as a CUDA graph replay")
    ap.add_argument("--no-kernel-loop", action="store_true",
                    help="skip the kernel-only loop of the dominant kernel (for ncu launch lists: steps only)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the loss and a fixed sample of the gradient rows of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 path")
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    # Exactly ONE line goes to stdout: the JSON.  Libraries write banners there (NCCL prints its version on the first
    # collective), so everything else -- at file-descriptor level -- is sent to stderr.
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        os.write(json_fd, (json.dumps(obj) + "\n").encode())

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference_arm(args, rank, world, emit)
        return

    import torch
    import torch.distributed as dist
    import b200ctc

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    group = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"                      # keep NCCL's version banner off stdout (one JSON line)
        dist.init_process_group("nccl", device_id=dev)
        group = dist.group.WORLD

    W = WORKLOAD
    B, T, V, L = W["B"], W["T"], W["V"], W["L"]
    prob = synth().ctc_problem(B, T, V, L, seed=rank)            # each rank owns its own shard of utterances
    x = torch.tensor(prob["x"], device=dev).requires_grad_(True)  # (T,B,V), the reference's stacked layout
    labels = torch.tensor(prob["labels"], device=dev)
    in_len = torch.tensor(prob["input_length"], device=dev)
    lab_len = torch.tensor(prob["label_length"], device=dev)
    # Batch-sharded step (SURVEY.md 8e): every rank scales its partial loss sum by 1/B_global in-kernel
    # (batch_global), the gradient needs no communication, and the ONE collective of the path -- a small NCCL
    # all-reduce of the loss -- is issued after the gradient kernel has been enqueued, so no rank's backward ever
    # waits for a peer's forward.
    kw = {"batch_global": world * B} if world > 1 else {}
    kDepth = 4                                       # all-reduce buffers per rank
    kEvery = max(1, int(os.environ.get("B200CTC_BENCH_REDUCE_EVERY", "4")))      # steps per all-reduce
    red = {"buf": [torch.zeros(kEvery, dtype=torch.float32, device=dev) for _ in range(kDepth)], "work": [None] * kDepth,
           "n": 0, "open": False}

    def reduce_loss(loss):
        """The loss all-reduce, asynchronous and off the critical path: the rank-local partial loss of a step is copied
        into the next slot of a small buffer, and every kEvery steps NCCL sums that buffer over the ranks on its own
        stream (every step's global loss is computed, each at most kEvery steps after its step -- what a training loop
        that logs the loss does).  The compute stream waits for a reduce only when its buffer comes round again or is
        read.  Measured at 8 GPUs: ranks as independent replicas 0.362 ms per step, one scalar all-reduce per step
        0.377 (the NCCL kernel takes SMs from the persistent row kernels while it waits for its peers), so it is
        issued once per four steps.  B200CTC_BENCH_REDUCE_EVERY=1 restores the per-step collective."""
        if world > 1 and os.environ.get("B200CTC_BENCH_NO_REDUCE") != "1":        # (diagnostic: ranks as independent replicas)
            g, i = (red["n"] // kEvery) % kDepth, red["n"] % kEvery
            red["n"] += 1
            if i == 0 and red["work"][g] is not None:
                red["work"][g].wait()
                red["work"][g] = None
            red["buf"][g][i].copy_(loss.detach())
            red["open"] = True
            if i == kEvery - 1:
                red["work"][g] = dist.all_reduce(red["buf"][g], op=dist.ReduceOp.SUM, group=group, async_op=True)
                red["open"] = False
            return red["buf"][g][i]
        return loss

    def finish_reduce():
        if red["open"]:                                  # a group that is not full yet: reduce what it holds, start afresh
            g = ((red["n"] - 1) // kEvery) % kDepth
            red["work"][g] = dist.all_reduce(red["buf"][g], op=dist.ReduceOp.SUM, group=group, async_op=True)
            red["n"] = (red["n"] + kEvery - 1) // kEvery * kEvery
            red["open"] = False
        for i in range(kDepth):
            if red["work"][i] is not None:
                red["work"][i].wait()
                red["work"][i] = None

    def step():
        x.grad = None
        loss = b200ctc.connectionist_temporal_classification(x, labels, 0, in_len, lab_len, reduce="mean", **kw)
        loss.backward()
        return reduce_loss(loss)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    finish_reduce()
    barrier()

    # ---- timed region: device time, CUDA events on the stream the kernels are launched on ----
    sampler = ClockSampler(local_rank)
    if rank == 0:                                    # one nvidia-smi poller per job, not per rank: at 8 ranks the host
        sampler.start()                              # cores are what the eager launch path is short of
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(args.steps)]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    h0 = time.perf_counter()
    e0.record()
    for k in range(args.steps):
        x.grad = None
        ev[k][0].record()
        loss = b200ctc.connectionist_temporal_classification(x, labels, 0, in_len, lab_len, reduce="mean", **kw)
        ev[k][1].record()
        loss.backward()
        ev[k][2].record()
        loss = reduce_loss(loss)
    finish_reduce()
    e1.record()
    host_ms = (time.perf_counter() - h0) * 1e3 / args.steps     # host time to ENQUEUE one step (no sync inside the loop)
    barrier()
    elapsed_ms = e0.elapsed_time(e1)
    fwd_ms = float(np.mean([ev[k][0].elapsed_time(ev[k][1]) for k in range(args.steps)]))
    bwd_ms = float(np.mean([ev[k][1].elapsed_time(ev[k][2]) for k in range(args.steps)]))
    t = torch.tensor([elapsed_ms, fwd_ms, bwd_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    elapsed_ms, fwd_ms, bwd_ms = [float(v) for v in t.tolist()]
    loss_value = float(loss.item())
    eager_outputs = sample_outputs(loss, x.grad) if args.dump_outputs else None

    # ---- the dominant kernel alone (gradient_ring_kernel): K launches of b200ctc_backward through the C ABI on the
    #      workspace of one forward, bracketed by CUDA events on the launching stream ----
    k3_ms = None
    try:
        if args.no_kernel_loop:
            raise RuntimeError("--no-kernel-loop")
        L = b200ctc._lib
        lib = L.load()
        xd = x.detach()
        Lmax = labels.shape[1]
        nbytes = L.workspace_bytes(L.KIND_CTC, B, T, V, Lmax)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        loss_b = torch.empty(B, dtype=torch.float32, device=dev)
        loss_r = torch.empty((), dtype=torch.float32, device=dev)
        gy = torch.ones((), dtype=torch.float32, device=dev)
        gbuf = torch.empty_like(xd)
        sp = torch.cuda.current_stream(dev).cuda_stream
        L.check(lib.b200ctc_forward(L.KIND_CTC, xd.data_ptr(), xd.stride(0), xd.stride(1), labels.data_ptr(), None,
                                    in_len.data_ptr(), lab_len.data_ptr(), 0, B, T, V, Lmax, loss_b.data_ptr(),
                                    loss_r.data_ptr(), 1.0 / B, None, ws.data_ptr(), nbytes, 0, sp))

        def k3():
            L.check(lib.b200ctc_backward(L.KIND_CTC, xd.data_ptr(), xd.stride(0), xd.stride(1), labels.data_ptr(), None, 0,
                                         B, T, V, Lmax, gy.data_ptr(), 0, 1.0 / B, gbuf.data_ptr(), gbuf.stride(0),
                                         gbuf.stride(1), ws.data_ptr(), nbytes, sp))
        for _ in range(args.warmup):
            k3()
        torch.cuda.synchronize()
        q0, q1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        q0.record()
        for _ in range(args.steps):
            k3()
        q1.record()
        torch.cuda.synchronize()
        k3_ms = q0.elapsed_time(q1) / args.steps
        del ws, gbuf
    except Exception as exc:
        sys.stderr.write("bench.py: kernel-only timing skipped (%s)\n" % exc)

    # ---- the same step captured once in a CUDA graph and replayed (single GPU): identical kernels on identical
    #      buffers, minus the host launch path and the launch/dependency gaps between the kernels ----
    graph_ms, graph_outputs = None, None
    # Several GPUs: the graph holds the rank-local part of the step (capturing the NCCL all-reduce hung on this image);
    # the all-reduce of the graph's loss output is issued eagerly behind the replays (reduce_loss), as in the eager step.
    # B200CTC_BENCH_GRAPH_MULTI=0 switches the multi-GPU replay off.
    multi = world > 1 and os.environ.get("B200CTC_BENCH_GRAPH_MULTI", "1") == "1"
    if (world == 1 or multi) and not args.no_graph:
        graph, gloss, captured = None, None, 1.0
        try:
            del loss                                    # drop the eager autograd graph (its AccumulateGrad node is bound to
            x.grad = None                               # the default stream, which would invalidate the capture)
            gkw = {"batch_global": world * B} if world > 1 else {}
            # the package's own helper (asr/loss/graphed.py): what a training loop with fixed shapes would use
            gstep = b200ctc.GraphedStep(
                lambda: b200ctc.connectionist_temporal_classification(x, labels, 0, in_len, lab_len, reduce="mean", **gkw),
                [x], warmup=1, capture_error_mode="thread_local" if world > 1 else None)
            graph, gloss = gstep.graph, gstep.loss
        except Exception as exc:                                   # capture unsupported: the eager number stands
            sys.stderr.write("bench.py: CUDA graph capture skipped (%s)\n" % exc)
            captured = 0.0
        if world > 1:                                              # every rank replays, or none does
            flag = torch.tensor([captured], device=dev, dtype=torch.float64)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            captured = float(flag.item())
        if captured == 1.0:
            def replay():
                graph.replay()
                return reduce_loss(gloss)
            try:
                for _ in range(args.warmup):
                    replay()
                finish_reduce()
                barrier()
                g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                g0.record()
                for _ in range(args.steps):
                    gl = replay()
                finish_reduce()
                g1.record()
                barrier()
                ok = abs(float(gl.item()) - loss_value) <= 1e-5 * abs(loss_value)
                gt = torch.tensor([g0.elapsed_time(g1) / args.steps, 0.0 if ok else 1.0], device=dev, dtype=torch.float64)
                if world > 1:
                    dist.all_reduce(gt, op=dist.ReduceOp.MAX)      # slowest rank; any rank's mismatch disables it
                if float(gt[1].item()) == 0.0:
                    graph_ms = float(gt[0].item())
                    graph_outputs = sample_outputs(gl, x.grad) if args.dump_outputs else None
            except Exception as exc:                               # the eager number stands
                sys.stderr.write("bench.py: CUDA graph replay skipped (%s)\n" % exc)

    # ---- end to end: host (pinned) buffers through the host-array entry point (asr/loss/host.py):
    #      activations H2D, loss + gradient, gradient and loss D2H, all inside the timed region ----
    x_host = torch.from_numpy(np.ascontiguousarray(prob["x"].transpose(1, 0, 2))).pin_memory()     # (B,T,V)
    g_host = torch.empty_like(x_host).pin_memory()

    def e2e_step():
        l, _ = b200ctc.ctc_host(x_host, labels, 0, in_len, lab_len, reduce="mean", grad_out=g_host)
        return l

    e2e_loss = e2e_step()
    barrier()
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s0.record()
    for _ in range(args.e2e_steps):
        e2e_loss = e2e_step()
    s1.record()
    barrier()
    clocks = sampler.stop() if rank == 0 else None   # sampled over both timed regions (device-resident and end-to-end steps)
    t2 = torch.tensor([s0.elapsed_time(s1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t2, op=dist.ReduceOp.MAX)
    e2e_ms = float(t2.item())

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peak, peak_kind = measured_peak()
    k1_bytes, k3_bytes = algorithmic_bytes(V, prob["input_length"], B, T)
    step_bytes = k1_bytes + k3_bytes
    eager_ms_per_step = elapsed_ms / args.steps
    ms_per_step = min(eager_ms_per_step, graph_ms) if graph_ms else eager_ms_per_step
    if args.dump_outputs:
        write_outputs(args.dump_outputs, graph_outputs if graph_ms and graph_ms < eager_ms_per_step else eager_outputs)
    value = world * B * T / (ms_per_step * 1e-3)
    k3_time_ms = k3_ms if k3_ms else bwd_ms
    achieved = k3_bytes / (k3_time_ms * 1e-3) / 1e9
    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_dict(world),
        "valid_frames_per_step": int(np.sum(prob["input_length"])), "loss": loss_value,
        "valid_frames_per_s": world * int(np.sum(prob["input_length"])) / (ms_per_step * 1e-3),
        "launch": (("CUDA graph replay of the public-API step (loss forward + backward captured once)" +
                    ("; the loss all-reduce issued eagerly, asynchronously, once per four replays" if world > 1 else ""))
                   if graph_ms and graph_ms < eager_ms_per_step else "eager calls of the public API"),
        "eager_ms_per_step": eager_ms_per_step, "graph_ms_per_step": graph_ms,
        "fwd_ms": fwd_ms, "bwd_ms": bwd_ms, "host_enqueue_ms_per_step": host_ms,
        "roofline": {"bound": "hbm", "kernel": "gradient_ring_kernel", "achieved": achieved, "peak": peak,
                     "unit": "GB/s", "frac": achieved / peak, "traffic": profiled_traffic("gradient_ring_kernel"),
                     "peak_source": peak_kind, "kernel_ms": k3_time_ms,
                     "timed": ("%d back-to-back launches through b200ctc_backward, CUDA events" % args.steps) if k3_ms
                              else "event pair around loss.backward()",
                     "algorithmic_bytes_per_launch": k3_bytes},
        "step_roofline": {"achieved": step_bytes / (ms_per_step * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                          "frac": step_bytes / (ms_per_step * 1e-3) / 1e9 / peak,
                          "algorithmic_bytes_per_step": step_bytes},
        "e2e": {"value": world * B * T * args.e2e_steps / (e2e_ms * 1e-3), "unit": UNIT,
                "h2d_bytes_per_step": int(np.sum(prob["input_length"])) * V * 4, "d2h_bytes_per_step": int(np.sum(prob["input_length"])) * V * 4 + 4,
                "ms_per_step": e2e_ms / args.e2e_steps, "loss": e2e_loss,
                "api": "b200ctc.ctc_host: 16 utterance groups, H2D / kernels / D2H on three streams, pinned host buffers; only valid "
                       "frames cross PCIe in either direction, the padded gradient rows (exact zeros) are written by host threads"},
        "gpu_launches": 4 * args.steps,          # per step: header reset, softmax/gather, lattice(+prep), gradient
        "clocks": clocks,
    }
    if world == 1 and not args.no_cpu_baseline:
        threads = host_threads()
        ref = ReferenceSample(prob)
        v, secs, reps = port_baseline(prob, threads)
        port = {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
                "sample": "oracle C port (oracle/ctc_oracle.c, banded restatement, float64, OpenMP x%d): %d passes over the "
                          "same 64-utterance workload, %.1f s of CPU work" % (threads, reps, secs)}
        if ref.ok:                                   # ~12 s: warm-up + 6 timed steps of the reference's own NumPy path
            ref.step()
            n, tot = 6, 0.0
            for _ in range(n):
                _, f, b = ref.step()
                tot += f + b
            out["cpu_baseline"] = {"value": ref.frames * n / tot, "unit": UNIT, "cores": ref.threads, "kind": "reference",
                                   "sample": ref.describe() + "; %d steps, %.1f s of CPU work; host has %d cores" % (n, tot, threads)}
            out["port_baseline"] = port
        else:
            out["cpu_baseline"] = port
    emit(out)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
