"""Forced alignment (csrc/viterbi.cu) on the bench workloads: device time by CUDA events, warmed up, activations
(614-717 MB) far larger than the 126 MB L2 and alternated between two copies, so no call finds its input in L2.

  cfg 2  CTC       B=64, T=800, V=3500, L<=80, variable lengths (bench.py's workload)
  cfg 3  Gram-CTC  B=32, T=600, V=8000, L<=60, variable lengths

Arms:
  align       b200ctc.ctc_forced_align / gram_ctc_forced_align (score, path, ids, frame_logp, spans)
  loss_fwd    the loss's forward pass alone at the same shape (reduce='no', no gradient), for scale
  torchaudio  cfg 2 only: torch.log_softmax over the batch, then torchaudio.functional.forced_align once per utterance
              (it takes one utterance per call), on the same GPU

    python tools/align_bench.py > profiles/r3_align.txt

--profile: in a run of its own, the per-kernel device time of one alignment call per workload (torch.profiler).
"""
import importlib
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
pkg = importlib.import_module("b200ctc")


def gpu_identity():
    """The card's name and power limit, read in the same run as the numbers."""
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit": q or "unavailable"}


def timed(fn, inputs, calls, warmup, rounds):
    """Median over `rounds` of the mean device time per call (ms); call i uses inputs[i % len(inputs)]."""
    for i in range(warmup):
        fn(inputs[i % len(inputs)])
    torch.cuda.synchronize()
    per = []
    for _ in range(rounds):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(calls):
            fn(inputs[i % len(inputs)])
        e1.record()
        torch.cuda.synchronize()
        per.append(e0.elapsed_time(e1) / calls)
    return {"ms_per_call_rounds": per, "ms_per_call": float(np.median(per))}


def problem(kind, B, T, V, L, seed):
    synth = pkg.synth
    dev = torch.device("cuda:0")
    if kind == "ctc":
        prob = synth.ctc_problem(B, T, V, L, seed=seed)
    else:
        prob = synth.gram_problem(B, T, V, L, seed=seed)
    xs = [torch.tensor(prob["x"], device=dev)]
    xs.append(xs[0].flip(2).contiguous())                 # a second input of the same statistics at other addresses
    lab = torch.tensor(prob["labels"], device=dev)
    big = torch.tensor(prob["bigrams"], device=dev) if kind == "gram" else None
    il = torch.tensor(prob["input_length"], device=dev)
    ll = torch.tensor(prob["label_length"], device=dev)
    return prob, xs, lab, big, il, ll


def measure(kind, B, T, V, L, calls, warmup, rounds, ta_calls):
    prob, xs, lab, big, il, ll = problem(kind, B, T, V, L, seed=0)
    out = {"shape": {"kind": kind, "B": B, "T": T, "V": V, "Lmax": L, "valid_frames": int(prob["input_length"].sum())}}
    if kind == "ctc":
        align = lambda x: pkg.ctc_forced_align(x, lab, 0, il, ll)
        loss = lambda x: pkg.ctc(x, lab, 0, il, ll, reduce="no")
    else:
        align = lambda x: pkg.gram_ctc_forced_align(x, lab, big, 0, il, ll)
        loss = lambda x: pkg.gram_ctc(x, lab, big, 0, il, ll, reduce="no")
    out["align"] = timed(align, xs, calls, warmup, rounds)
    with torch.no_grad():
        out["loss_fwd"] = timed(loss, xs, calls, warmup, rounds)
    a = align(xs[0])
    lo = loss(xs[0]).detach()
    out["align"]["score_minus_loss_mean"] = float((a.score - lo).mean())
    if kind == "ctc" and ta_calls:
        import torchaudio.functional as F
        Tb = [int(v) for v in prob["input_length"]]
        Lb = [int(v) for v in prob["label_length"]]
        lab32 = lab.to(torch.int32)

        def torchaudio_arm(x):
            lp = torch.log_softmax(x, dim=2).transpose(0, 1).contiguous()    # (B,T,V): forced_align wants contiguous rows
            ids = []
            for b in range(B):
                path, _ = F.forced_align(lp[b:b + 1, :Tb[b]], lab32[b:b + 1, :Lb[b]], blank=0)
                ids.append(path)
            return ids

        out["torchaudio"] = timed(torchaudio_arm, xs, ta_calls, 1, rounds)
        ids = torchaudio_arm(xs[0])
        same = sum(int(torch.equal(ids[b][0].to(torch.int64), a.ids[b, :Tb[b]])) for b in range(B))
        out["torchaudio"]["utterances_with_ids_equal_to_align"] = "%d/%d" % (same, B)
    return out


def profile():
    from torch.profiler import profile as tprof, ProfilerActivity
    for kind, shape in (("ctc", (64, 800, 3500, 80)), ("gram", (32, 600, 8000, 60))):
        _, xs, lab, big, il, ll = problem(kind, *shape, seed=0)
        call = ((lambda: pkg.ctc_forced_align(xs[0], lab, 0, il, ll)) if kind == "ctc"
                else (lambda: pkg.gram_ctc_forced_align(xs[0], lab, big, 0, il, ll)))
        for _ in range(3):
            call()
        torch.cuda.synchronize()
        with tprof(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(5):
                call()
            torch.cuda.synchronize()
        print("# %s %s: device time per call by kernel (mean of 5 calls)" % (kind, shape))
        for ev in sorted(prof.key_averages(), key=lambda e: -e.device_time_total):
            if ev.device_time_total > 0:
                print("#   %-60s %9.1f us" % (ev.key[:60], ev.device_time_total / 5))


def main():
    if "--profile" in sys.argv:
        print("# %s" % json.dumps(gpu_identity()))
        profile()
        return
    r = gpu_identity()
    r["timing"] = ("CUDA events; median of 3 rounds (align, loss_fwd: 20 calls; torchaudio: 3 calls) after warm-up; "
                   "two input copies alternated, each larger than L2")
    r["cfg2_ctc"] = measure("ctc", 64, 800, 3500, 80, calls=20, warmup=5, rounds=3, ta_calls=3)
    r["cfg3_gram"] = measure("gram", 32, 600, 8000, 60, calls=20, warmup=5, rounds=3, ta_calls=0)
    print(json.dumps(r))
    print("# %s, power limit %s" % (r["gpu"], r["nvidia_smi_name_power_limit"]))
    for cfg in ("cfg2_ctc", "cfg3_gram"):
        c = r[cfg]
        a = c["align"]["ms_per_call"]
        print("# %s %s" % (cfg, c["shape"]))
        for arm in ("align", "loss_fwd", "torchaudio"):
            if arm in c:
                print("#   %-10s %9.3f ms per call   %7.2fx the alignment call" % (arm, c[arm]["ms_per_call"], c[arm]["ms_per_call"] / a))
        if "torchaudio" in c:
            print("#   torchaudio ids equal to the alignment's on %s utterances" % c["torchaudio"]["utterances_with_ids_equal_to_align"])


if __name__ == "__main__":
    main()
