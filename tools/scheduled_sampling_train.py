"""Training-step timing with scheduled sampling: the decoder-only step (forward, loss, BPTT, parameter gradients) at C2 dims
(B=256, T=20, D=512, A=128, E=256, H=512, L=196, bf16 tensor cores), teacher-forced (epsilon = 1) and with every step after
step 2 fed back (epsilon = 0), on the logits path (per-step [B, V] logits + row_argmax_kernel, whole [T*B, V] logits +
ce_rows_kernel) and on the fused path (per-tile statistics in the vocabulary GEMM's epilogue, no logits).

Cases: V = 10,000 teacher-forced, then epsilon = 0 unfused and epsilon = 0 fused (SAT_TRAIN_FUSED_SS=1) alternated; V = 60,000,
100,003 and 131,072 at epsilon = 0 (fused: the row kernel cannot hold a logits row).  Every case runs in a child process of its
own (SAT_TRAIN_FUSED_SS is read once per process).  Per case: ms per step from CUDA events after warm-up, the device time of the
sampled steps' extra work inside the time loop (sat_profile_begin(8): deep output, vocabulary GEMM with its epilogue or the
logits + arg-max, re-embedding and gate projection), peak device memory, and the card's name and power limit read in the same run.

    python tools/scheduled_sampling_train.py [--iters 10] [--warmup 3] [--rounds 2]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DIMS = dict(D=512, A=128, E=256, H=512, hw=(14, 14), B=256, T=20)


def child(args):
    import torch
    sys.path.insert(0, ROOT)
    from oracle import sat_oracle as O
    from sat_b200 import _lib, decoder
    from sat_b200.packing import PackedWeights
    c, V = DIMS, args.V
    W = O.random_weights(c["D"], c["A"], c["E"], c["H"], V, seed=1, sharpen=True)
    pw = PackedWeights(W, dtype=torch.bfloat16, device="cuda")
    g = torch.Generator().manual_seed(2)
    ann = torch.randn(c["B"], c["D"], *c["hw"], generator=g)
    bld = decoder.annotations_as_bld(ann.cuda(), torch.bfloat16)
    T = c["T"]
    caps = torch.randint(1, V - 3, (c["B"], T + 1), generator=g)
    caps[:, 0] = V - 2
    lens = torch.randint(T // 2, T + 1, (c["B"],), generator=g)
    caps, lens = caps.cuda(), lens.cuda()
    sampled = None if args.eps >= 1.0 else [0, 0, 0] + [1] * (T - 3)
    state = {}

    def run():
        state.pop("buf", None)                                # the previous step's buffers are freed first, as in training
        buf = decoder.train_forward(pw, bld, caps, lens, 0.0, 1.0, exact=False, use_tc=True, backward=True, sampled=sampled,
                                    fuse_ce=True)
        decoder.train_backward(pw, buf)
        state["buf"] = buf

    for _ in range(args.warmup):
        run()
    fused = state["buf"].fuse_ce
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    for _ in range(args.iters):
        run()
    ev[1].record()
    torch.cuda.synchronize()
    ms = ev[0].elapsed_time(ev[1]) / args.iters
    peak = torch.cuda.max_memory_allocated()
    _lib.profile_begin(8)
    for _ in range(2):
        run()
    loop_ms, loop_n = _lib.profile_end()
    smi = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit",
                          "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    print(json.dumps(dict(V=V, eps=args.eps, forced=os.environ.get("SAT_TRAIN_FUSED_SS") == "1", path="fused" if fused else "logits",
                          ms_per_step=ms, in_loop_ms_per_step=loop_ms / 2, sampled_steps=loop_n // 2, peak_mem_gb=peak / 1e9,
                          loss=float(state["buf"].t["out"][0]), device=torch.cuda.get_device_name(), nvidia_smi=smi)), flush=True)


def spawn(args, V, eps, force):
    env = dict(os.environ, PYTHONPATH=ROOT)
    env.pop("SAT_TRAIN_FUSED_SS", None)
    if force:
        env["SAT_TRAIN_FUSED_SS"] = "1"
    cmd = [sys.executable, os.path.abspath(__file__), "--child", "--V", str(V), "--eps", str(eps), "--iters", str(args.iters),
           "--warmup", str(args.warmup)]
    r = subprocess.run(cmd, env=env, cwd=ROOT, capture_output=True, text=True)
    if r.returncode != 0:
        raise SystemExit("case V=%d eps=%g failed:\n%s" % (V, eps, r.stderr[-3000:]))
    rec = json.loads(r.stdout.strip().splitlines()[-1])
    print(json.dumps(rec), flush=True)
    return rec


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=2, help="alternations of the V = 10,000 epsilon = 0 A/B")
    ap.add_argument("--child", action="store_true")
    ap.add_argument("--V", type=int)
    ap.add_argument("--eps", type=float, default=0.0)
    args = ap.parse_args()
    if args.child:
        return child(args)
    recs = [spawn(args, 10000, 1.0, False)]
    for _ in range(args.rounds):                                   # V = 10,000, epsilon = 0: logits path vs fused, alternated
        recs.append(spawn(args, 10000, 0.0, False))
        recs.append(spawn(args, 10000, 0.0, True))
    for V in (60000, 100003, 131072):
        recs.append(spawn(args, V, 0.0, False))
    print("\n%-8s %-4s %-7s %10s %14s %9s" % ("V", "eps", "path", "ms/step", "in-loop ms", "peak GB"))
    for r in recs:
        print("%-8d %-4g %-7s %10.2f %14.2f %9.2f" % (r["V"], r["eps"], r["path"], r["ms_per_step"], r["in_loop_ms_per_step"],
                                                     r["peak_mem_gb"]))
    print("device: %s | nvidia-smi name, power.limit: %s" % (recs[0]["device"], recs[0]["nvidia_smi"]))


if __name__ == "__main__":
    main()
