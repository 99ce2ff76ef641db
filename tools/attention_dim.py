"""Attention stage timing across attention_dim, pipelined kernels against the plain single-pass ones.

Workloads (bf16 tensor-core path):
  train  the decoder-only training step (forward, loss, BPTT, parameter gradients) at C2 dims: B = 256, T = 20, L = 196, D = 512,
         E = 256, H = 512, V = 10,000.  ms per step from CUDA events after warm-up; the attention forward and backward device
         time per step (sat_profile_begin(1) / (2): the attention-step launches inside the time loops);
  beam   beam-5 decode at C5 dims: 256 images, L = 256, D = 2048, E = 512, H = 1024, V = 10,000, 20 steps.  ms per call and the
         attention forward device time per call (sat_profile_begin(1)).
A in {128, 256, 384, 512, 768, 1024}; every (A, kernels) pair runs in a child process of its own, the pipelined kernels and
the plain ones (SAT_ATT_MODE=0 SAT_ATTB_MODE=0, read once per process) alternated.  Also: peak device memory, and the card's
name and power limit read in the same run.

    python tools/attention_dim.py [--A 128,256,384,512,768,1024] [--iters 5] [--warmup 2] [--rounds 1] [--json out.json]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TRAIN = dict(B=256, T=20, hw=(14, 14), D=512, E=256, H=512, V=10000)
BEAM = dict(n=256, hw=(16, 16), D=2048, E=512, H=1024, V=10000, k=5, S=20)


def child(args):
    import torch
    sys.path.insert(0, ROOT)
    from oracle import sat_oracle as O
    from sat_b200 import _lib, decode, decoder
    from sat_b200.packing import PackedWeights
    A, out = args.A, {}
    # training step
    c = TRAIN
    W = O.random_weights(c["D"], A, c["E"], c["H"], c["V"], seed=1, sharpen=True)
    pw = PackedWeights(W, dtype=torch.bfloat16, device="cuda")
    g = torch.Generator().manual_seed(2)
    bld = decoder.annotations_as_bld(torch.randn(c["B"], c["D"], *c["hw"], generator=g).cuda(), torch.bfloat16)
    caps = torch.randint(1, c["V"] - 3, (c["B"], c["T"] + 1), generator=g)
    caps[:, 0] = c["V"] - 2
    lens = torch.randint(c["T"] // 2, c["T"] + 1, (c["B"],), generator=g)
    caps, lens = caps.cuda(), lens.cuda()
    state = {}

    def step():
        state.pop("buf", None)                                # the previous step's buffers are freed first, as in training
        buf = decoder.train_forward(pw, bld, caps, lens, 0.0, 1.0, exact=False, use_tc=True, backward=True, fuse_ce=True)
        decoder.train_backward(pw, buf)
        state["buf"] = buf

    def timed(fn, iters, warmup):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        ev[0].record()
        for _ in range(iters):
            fn()
        ev[1].record()
        torch.cuda.synchronize()
        return ev[0].elapsed_time(ev[1]) / iters, torch.cuda.max_memory_allocated() / 1e9

    def stage(kind, fn, reps=2):
        _lib.profile_begin(kind)
        for _ in range(reps):
            fn()
        ms, _ = _lib.profile_end()
        return ms / reps

    ms, peak = timed(step, args.iters, args.warmup)
    out["train"] = dict(ms_per_step=ms, att_fwd_ms=stage(1, step), att_bwd_ms=stage(2, step), peak_mem_gb=peak,
                        loss=float(state["buf"].t["out"][0]))
    del state["buf"], pw, bld
    torch.cuda.empty_cache()
    # beam-5 decode
    c = BEAM
    W = O.random_weights(c["D"], A, c["E"], c["H"], c["V"], seed=3, sharpen=True)
    dw = decode.DecodeWeights(W, torch.bfloat16, torch.device("cuda"), False, True)
    bld = decoder.annotations_as_bld(torch.randn(c["n"], c["D"], *c["hw"], generator=g).cuda(), torch.bfloat16)
    vocab = dict(PAD=0, UNK=c["V"] - 3, START=c["V"] - 2, END=c["V"] - 1)

    def beam():
        t = decode.decode_annotations(dw, bld, c["k"], c["S"], 1.0, "LN", 0.5, vocab, early_out=False)
        state["t"] = t

    ms, peak = timed(beam, max(2, args.iters // 2), 1)
    out["beam"] = dict(ms_per_call=ms, att_fwd_ms=stage(1, beam), peak_mem_gb=peak)
    smi = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit",
                          "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    out.update(A=A, kernels="plain" if os.environ.get("SAT_ATT_MODE") == "0" else "pipelined",
               device=torch.cuda.get_device_name(), nvidia_smi=smi)
    print(json.dumps(out), flush=True)


def spawn(args, A, plain):
    env = dict(os.environ, PYTHONPATH=ROOT)
    for k in ("SAT_ATT_MODE", "SAT_ATTB_MODE"):
        env.pop(k, None)
    if plain:
        env.update(SAT_ATT_MODE="0", SAT_ATTB_MODE="0")
    cmd = [sys.executable, os.path.abspath(__file__), "--child", "--A", str(A), "--iters", str(args.iters), "--warmup", str(args.warmup)]
    r = subprocess.run(cmd, env=env, cwd=ROOT, capture_output=True, text=True)
    if r.returncode != 0:
        raise SystemExit("A=%d %s failed:\n%s" % (A, "plain" if plain else "pipelined", r.stderr[-3000:]))
    rec = json.loads(r.stdout.strip().splitlines()[-1])
    print(json.dumps(rec), flush=True)
    return rec


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--A", default="128,256,384,512,768,1024")
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--rounds", type=int, default=1, help="alternations of pipelined / plain per A")
    ap.add_argument("--json", default=None, help="also write every record to this file")
    ap.add_argument("--child", action="store_true")
    args = ap.parse_args()
    if args.child:
        args.A = int(args.A)
        return child(args)
    recs = []
    for A in [int(a) for a in args.A.split(",")]:
        for _ in range(args.rounds):
            recs.append(spawn(args, A, False))
            recs.append(spawn(args, A, True))
    if args.json:
        with open(args.json, "w") as f:
            json.dump(recs, f, indent=1)
    print("\n%5s %-9s | %9s %9s %9s %8s | %9s %9s %8s" % ("A", "kernels", "step ms", "att fwd", "att bwd", "peak GB",
                                                          "beam ms", "att fwd", "peak GB"))
    for r in recs:
        t, b = r["train"], r["beam"]
        print("%5d %-9s | %9.2f %9.2f %9.2f %8.2f | %9.2f %9.2f %8.2f" % (r["A"], r["kernels"], t["ms_per_step"], t["att_fwd_ms"],
                                                                          t["att_bwd_ms"], t["peak_mem_gb"], b["ms_per_call"],
                                                                          b["att_fwd_ms"], b["peak_mem_gb"]))
    print("device: %s | nvidia-smi name, power.limit: %s" % (recs[0]["device"], recs[0]["nvidia_smi"]))


if __name__ == "__main__":
    main()
