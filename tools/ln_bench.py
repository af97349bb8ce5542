"""LayerNormalization -> loss: the fused path (csrc/layernorm_loss.cu) against the unfused pipelines it replaces, on the
bench workload (B=64, T=800, V=3500, L<=80, variable lengths).  Device time, CUDA events, inputs resident in HBM.

  fused            b200ctc.layernorm_ctc(z, gamma, beta, ...): z (B,V,1,T) read in place, dz written in place
  reference-style  what the reference's model tail does, op by op (asr/nn/layernorm.py:33-46, asr/nn/nn.py:265,
                   asr/model/cnn.py:41-44) as torch ops, then b200ctc.ctc on the transposed copy
  torch-native     torch.nn.functional.layer_norm over a (B,T,V) view (one transposing copy + one fused LN kernel),
                   then b200ctc.ctc(batch_first=True)

    python tools/ln_bench.py > profiles/r2_layernorm_fusion.txt

--kind joint: the joint Gram-CTC + CTC objective (run/gram_ctc/cnn/train.py:196-198) on the Gram-CTC workload of BASELINE
configs[2] with V cut to the fused limit (B=32, T=600, V=4000, L<=60, variable lengths).  Arms:

  fused_joint      b200ctc.layernorm_gram_ctc(..., joint_ctc=True): forward and backward also timed separately
  fused_gram       b200ctc.layernorm_gram_ctc alone (the Gram-CTC loss only): its backward is the yardstick of the joint one
  fused_two_calls  b200ctc.layernorm_gram_ctc(...) + b200ctc.layernorm_ctc(...): the joint objective as two fused calls
  torch_native     torch.nn.functional.layer_norm over a (B,T,V) view, then b200ctc.gram_ctc(joint_ctc=True, batch_first=True)
  reference_style  the reference's model tail op by op, then b200ctc.gram_ctc(joint_ctc=True) on the transposed copy

    python tools/ln_bench.py --kind joint > profiles/r3_layernorm_joint.txt
"""
import argparse, importlib, json, os, subprocess, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import b200ctc
synth = importlib.import_module("chainer-speech-recognition_b200.synth")


def measure(B=64, T=800, V=3500, L=80, steps=10, warmup=3):
    dev = torch.device("cuda:0")
    rs = np.random.RandomState(0)
    in_len, lab_len = synth.make_lengths(rs, B, T, L)
    labels = synth.make_ctc_labels(rs, B, L, V, lab_len)
    g = torch.Generator(device=dev); g.manual_seed(0)
    z = (torch.randn((B, V, 1, T), device=dev, generator=g) * 1.7 + 0.3).requires_grad_(True)
    gamma = (1 + 0.2 * torch.randn(V, device=dev, generator=g)).requires_grad_(True)
    beta = (0.1 * torch.randn(V, device=dev, generator=g)).requires_grad_(True)
    lab = torch.tensor(labels, device=dev); il = torch.tensor(in_len, device=dev); ll = torch.tensor(lab_len, device=dev)

    def fused():
        return b200ctc.layernorm_ctc(z, gamma, beta, lab, 0, il, ll, reduce="mean")

    def reference_style():
        x = z
        mean = x.mean(dim=(1, 2), keepdim=True)
        diff = x - mean
        std = torch.sqrt((diff * diff).sum(dim=(1, 2), keepdim=True) / V)
        y = diff / std * gamma[None, :, None, None] + beta[None, :, None, None]
        out = y.swapaxes(1, 3).reshape(B, -1)                               # the transposed copy
        xs = out.view(B, T, V).transpose(0, 1)                                # split_axis: T views (B,V) = a (T,B,V) view
        return b200ctc.ctc(xs, lab, 0, il, ll, reduce="mean")

    def torch_native():
        y = torch.nn.functional.layer_norm(z.squeeze(2).transpose(1, 2), (V,), gamma, beta, eps=0.0)   # (B,T,V)
        return b200ctc.ctc(y, lab, 0, il, ll, reduce="mean", batch_first=True)

    out = {}
    for name, fn in (("fused", fused), ("reference_style", reference_style), ("torch_native", torch_native)):
        for _ in range(warmup):
            z.grad = gamma.grad = beta.grad = None
            fn().backward()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            z.grad = gamma.grad = beta.grad = None
            loss = fn()
            loss.backward()
        e1.record()
        torch.cuda.synchronize()
        out[name] = {"ms_per_step": e0.elapsed_time(e1) / steps, "loss": float(loss)}
        if name == "fused":                       # forward and backward separately
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            z.grad = gamma.grad = beta.grad = None
            ev[0].record(); loss = fn(); ev[1].record(); loss.backward(); ev[2].record()
            torch.cuda.synchronize()
            out[name]["fwd_ms"] = ev[0].elapsed_time(ev[1]); out[name]["bwd_ms"] = ev[1].elapsed_time(ev[2])
    valid = float(in_len.sum())
    # algorithmic bytes: fused = read z twice (valid frames) + write dz once; the unfused pipelines add LN forward
    # (read z, write y), the transposed copy (read + write), its backward (read + write) and LN backward (read g, read z, write dz)
    out["fused"]["algorithmic_bytes"] = 8 * V * valid + 4 * V * B * T
    out["reference_style"]["algorithmic_bytes"] = out["fused"]["algorithmic_bytes"] + 4 * V * B * T * (2 + 2 + 2 + 3)
    out["frames"] = B * T
    return out


def gpu_identity():
    """The card's name and power limit, read in the same run as the numbers."""
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit": q or "unavailable"}


def measure_joint(B=32, T=600, V=4000, L=60, steps=20, warmup=3, rounds=3):
    dev = torch.device("cuda:0")
    rs = np.random.RandomState(0)
    in_len, lab_len = synth.make_lengths(rs, B, T, L)
    in_len = np.maximum(in_len, np.minimum(T, 3 * lab_len + 1)).astype(np.int32)
    uni, big = synth.make_gram_labels(rs, B, L, V, lab_len, n_unigram=119)
    g = torch.Generator(device=dev); g.manual_seed(0)
    z = (torch.randn((B, V, 1, T), device=dev, generator=g) * 1.7 + 0.3).requires_grad_(True)
    gamma = (1 + 0.2 * torch.randn(V, device=dev, generator=g)).requires_grad_(True)
    beta = (0.1 * torch.randn(V, device=dev, generator=g)).requires_grad_(True)
    lab = torch.tensor(uni, device=dev); bg = torch.tensor(big, device=dev)
    il = torch.tensor(in_len, device=dev); ll = torch.tensor(lab_len, device=dev)

    def fused_joint():
        return b200ctc.layernorm_gram_ctc(z, gamma, beta, lab, bg, 0, il, ll, reduce="mean", joint_ctc=True)

    def fused_gram():
        return b200ctc.layernorm_gram_ctc(z, gamma, beta, lab, bg, 0, il, ll, reduce="mean")

    def fused_two_calls():
        return (b200ctc.layernorm_gram_ctc(z, gamma, beta, lab, bg, 0, il, ll, reduce="mean")
                + b200ctc.layernorm_ctc(z, gamma, beta, lab, 0, il, ll, reduce="mean"))

    def torch_native():
        y = torch.nn.functional.layer_norm(z.squeeze(2).transpose(1, 2), (V,), gamma, beta, eps=0.0)   # (B,T,V)
        return b200ctc.gram_ctc(y, lab, bg, 0, il, ll, reduce="mean", joint_ctc=True, batch_first=True)

    def reference_style():
        x = z
        mean = x.mean(dim=(1, 2), keepdim=True)
        diff = x - mean
        std = torch.sqrt((diff * diff).sum(dim=(1, 2), keepdim=True) / V)
        y = diff / std * gamma[None, :, None, None] + beta[None, :, None, None]
        out = y.swapaxes(1, 3).reshape(B, -1)                               # the transposed copy
        xs = out.view(B, T, V).transpose(0, 1)                                # split_axis: a (T,B,V) view
        return b200ctc.gram_ctc(xs, lab, bg, 0, il, ll, reduce="mean", joint_ctc=True)

    arms = (("fused_joint", fused_joint), ("fused_gram", fused_gram), ("fused_two_calls", fused_two_calls),
            ("torch_native", torch_native), ("reference_style", reference_style))
    out = {name: {"ms_per_step_rounds": []} for name, _ in arms}
    for name, fn in arms:
        for _ in range(warmup):
            z.grad = gamma.grad = beta.grad = None
            fn().backward()
    torch.cuda.synchronize()
    for _ in range(rounds):                       # the arms alternate: drift on a shared host hits all of them alike
        for name, fn in arms:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                z.grad = gamma.grad = beta.grad = None
                loss = fn()
                loss.backward()
            e1.record()
            torch.cuda.synchronize()
            out[name]["ms_per_step_rounds"].append(e0.elapsed_time(e1) / steps)
            out[name]["loss"] = float(loss)
    for name, fn in arms:
        out[name]["ms_per_step"] = float(np.median(out[name]["ms_per_step_rounds"]))
    for name, fn in (("fused_joint", fused_joint), ("fused_gram", fused_gram)):      # forward and backward separately
        fw, bw = [], []
        for _ in range(steps):
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            z.grad = gamma.grad = beta.grad = None
            ev[0].record(); loss = fn(); ev[1].record(); loss.backward(); ev[2].record()
            torch.cuda.synchronize()
            fw.append(ev[0].elapsed_time(ev[1])); bw.append(ev[1].elapsed_time(ev[2]))
        out[name]["fwd_ms"] = float(np.median(fw)); out[name]["bwd_ms"] = float(np.median(bw))
    out["shape"] = {"B": B, "T": T, "V": V, "Lmax": L, "frames": B * T, "valid_frames": int(in_len.sum())}
    out["timing"] = "CUDA events; median of %d rounds of %d steps after %d warm-up steps per arm; z (%.0f MB) in HBM" % (
        rounds, steps, warmup, 4.0 * B * V * T / 1e6)
    out.update(gpu_identity())
    return out


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--kind", choices=("ctc", "joint"), default="ctc")
    if ap.parse_args().kind == "joint":
        r = measure_joint()
        print(json.dumps(r))
        print("# %s, power limit %s" % (r["gpu"], r["nvidia_smi_name_power_limit"]))
        f = r["fused_joint"]["ms_per_step"]
        for k in ("fused_joint", "fused_gram", "fused_two_calls", "torch_native", "reference_style"):
            print("# %-16s %8.3f ms per step   %6.2fx the fused joint step   loss %.4f" % (k, r[k]["ms_per_step"], r[k]["ms_per_step"] / f,
                                                                                     r[k]["loss"]))
        for k in ("fused_joint", "fused_gram"):
            print("# %-16s forward %.3f ms   backward %.3f ms" % (k, r[k]["fwd_ms"], r[k]["bwd_ms"]))
        sys.exit(0)
    r = measure()
    print(json.dumps(r))
    f = r["fused"]["ms_per_step"]
    for k in ("fused", "reference_style", "torch_native"):
        print("# %-16s %8.3f ms per step   %6.2fx the fused path   loss %.4f" % (k, r[k]["ms_per_step"], r[k]["ms_per_step"] / f, r[k]["loss"]))
