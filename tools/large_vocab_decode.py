"""Decode timing at large vocabularies: bf16 tensor-core beam search / sampling on the fused candidate path (per-tile candidate
lists from the vocabulary GEMM's epilogue) against the shared-memory row kernels, and greedy decode at the same sizes for scale.

bench.py's "beam" dimensions (wide_resnet101_2: L=256, D=2048, H=512, A=128, E=256; 256 images, k=5, max_gen_length=30), seeded
random weights and annotations; the encoder is left out, so the decoder is what is timed.  Every case runs in a child process of
its own (SAT_VOCAB_TOPK is read once per process); the V = 10,000 A/B alternates the two paths.  Per case: ms per decode and
captions/s from CUDA events after warm-up, the vocabulary stage's device time (sat_profile_begin(3): the GEMM with its epilogue
plus the finalize / row kernel), peak device memory, and the card's name and power limit read in the same run.

    python tools/large_vocab_decode.py [--iters 5] [--warmup 2] [--rounds 2]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DIMS = dict(D=2048, A=128, E=256, H=512, hw=(16, 16), B=256, k=5, S=30)


def child(args):
    import torch
    sys.path.insert(0, ROOT)
    from oracle import sat_oracle as O
    from sat_b200 import _lib, decode, decoder
    c, V, k, method = DIMS, args.V, args.k, args.method
    W = O.random_weights(c["D"], c["A"], c["E"], c["H"], V, seed=1, sharpen=True)
    dw = decode.DecodeWeights(W, torch.bfloat16, torch.device("cuda"), False, True)
    g = torch.Generator(device="cuda").manual_seed(2)
    ann = torch.randn(c["B"], c["D"], *c["hw"], generator=g, device="cuda")
    bld = decoder.annotations_as_bld(ann, torch.bfloat16)
    del ann
    voc = dict(PAD=0, UNK=V - 3, START=V - 2, END=V - 1)
    d = decoder.make_dims(c["B"] * k, c["B"], c["hw"][0] * c["hw"][1], dw.pw, c["S"] + 1, torch.bfloat16, False, True)
    path = _lib.lib().sat_decode_vocab_path(d, k, decode.SAMPLE[method], 3)
    run = lambda: decode.decode_annotations(dw, bld, k, c["S"], 1.0, "LN", 0.5, voc, sample_method=method, seed=3)
    for _ in range(args.warmup):
        run()
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
    _lib.profile_begin(3)
    for _ in range(2):
        run()
    voc_ms, voc_n = _lib.profile_end()
    smi = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit",
                          "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    print(json.dumps(dict(V=V, k=k, method=method, forced=os.environ.get("SAT_VOCAB_TOPK") == "1",
                          path={0: "rows", 1: "fused greedy", 2: "fused candidates"}[path], ms_per_decode=ms,
                          captions_per_s=c["B"] * 1000.0 / ms, vocab_stage_ms_per_decode=voc_ms / 2, vocab_stage_launches=voc_n // 2,
                          peak_mem_gb=peak / 1e9, device=torch.cuda.get_device_name(), nvidia_smi=smi)), flush=True)


def spawn(args, V, k, method, force):
    env = dict(os.environ, PYTHONPATH=ROOT)
    env.pop("SAT_VOCAB_TOPK", None)
    if force:
        env["SAT_VOCAB_TOPK"] = "1"
    cmd = [sys.executable, os.path.abspath(__file__), "--child", "--V", str(V), "--k", str(k), "--method", method,
           "--iters", str(args.iters), "--warmup", str(args.warmup)]
    r = subprocess.run(cmd, env=env, cwd=ROOT, capture_output=True, text=True)
    if r.returncode != 0:
        raise SystemExit("case V=%d k=%d %s failed:\n%s" % (V, k, method, r.stderr[-3000:]))
    rec = json.loads(r.stdout.strip().splitlines()[-1])
    print(json.dumps(rec), flush=True)
    return rec


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--rounds", type=int, default=2, help="alternations of the V = 10,000 A/B")
    ap.add_argument("--child", action="store_true")
    ap.add_argument("--V", type=int)
    ap.add_argument("--k", type=int)
    ap.add_argument("--method", default="beam")
    args = ap.parse_args()
    if args.child:
        return child(args)
    recs = []
    for _ in range(args.rounds):                                   # V = 10,000: row kernels vs fused candidates, alternated
        recs.append(spawn(args, 10000, DIMS["k"], "beam", False))
        recs.append(spawn(args, 10000, DIMS["k"], "beam", True))
    for V in (60000, 131072):
        recs.append(spawn(args, V, DIMS["k"], "beam", False))
        recs.append(spawn(args, V, 1, "beam", False))
    recs.append(spawn(args, 50000, DIMS["k"], "multinomial", False))
    print("\n%-8s %-2s %-12s %-17s %10s %11s %12s %9s" % ("V", "k", "method", "path", "ms/decode", "captions/s", "vocab ms", "peak GB"))
    for r in recs:
        print("%-8d %-2d %-12s %-17s %10.2f %11.0f %12.2f %9.2f" % (r["V"], r["k"], r["method"], r["path"], r["ms_per_decode"],
                                                                   r["captions_per_s"], r["vocab_stage_ms_per_decode"], r["peak_mem_gb"]))
    print("device: %s | nvidia-smi name, power.limit: %s" % (recs[0]["device"], recs[0]["nvidia_smi"]))


if __name__ == "__main__":
    main()
