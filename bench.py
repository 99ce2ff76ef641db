#!/usr/bin/env python
"""Benchmark of the SAT decoder hot path on B200 (BASELINE.json metric: captions/sec for the train step and greedy / beam
decode at 1/2/4/8 GPUs, step p50 ms).

    python bench.py --gpus N --steps K --warmup W [--workload all|train|c3|greedy|beam] [--impl reference] [--dump-outputs DIR]

The line's headline (`value`, `e2e`, `roofline`, `cpu_baseline`) is BASELINE.json configs[1]: SAT resnet50 encoder, L=196,
D=512, hidden 512, vocab 6400, batch 256 per GPU, bf16 training step (encoder fwd + decoder fwd + loss + full backward +
optimizer step).  With the default `--workload all` the same line carries one sub-record per remaining BASELINE config:
  "c3"     configs[2]  resnet101 encoder, D=2048, H=1024, batch 512 per GPU, DDP training step
  "greedy" configs[3]  greedy decode, resnet50 dims, max caplen 30, batch 1024 per GPU
  "beam"   configs[4]  beam search k=5, wide_resnet101_2 dims, L=256, V=10000, batch 256 per GPU
each with its own value / ms_per_step / e2e / roofline / config.  For N>1 launch with torch.distributed.run: every rank
keeps the per-GPU batch (weak scaling); training averages gradients with NCCL all-reduce overlapped with the backward,
decode shards by image with no collective.  Times are CUDA-event times, max over ranks.

`--impl reference` times the UNMODIFIED reference (model.py / util.py, copied into the git-ignored oracle/_ref/ by
__graft_entry__.build(); the oracle port when that copy is absent) on the host CPU on a bounded sample of each workload.
Prints ONE JSON line on rank 0.

`--dump-outputs DIR` (B200 arm, rank 0) writes what each workload's timed step computed in its last timed step to
DIR/<workload>.<output>.npy, float32 or float64, so that two builds run with the same arguments (hence the same seeded inputs)
can be compared output for output:
  train / c3     loss, aux (the 8 step statistics of fused_loss), grad.<parameter> for every decoder parameter and
                 grad.encoder (all encoder gradients, flattened and concatenated)
  greedy / beam  tokens [B, S+1] (-1 past the caption's end), lengths, scores, perplexities and alphas [B, S+1, L] (0 past the
                 end) of the returned caption of every image, as SAT.caption returns them
An output of more than DUMP_SAMPLE elements is stored as the DUMP_SAMPLE elements at fixed flat indices (drawn from a generator
seeded with 0, sorted); all files together stay under 64 MB.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time
import warnings

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "captions_per_sec"

# BASELINE.json configs (SURVEY.md §8d): decoder dims A=128, E=256 everywhere
CFG = {
    "train": dict(kind="train", arch="resnet50", D=512, size=14, L=196, H=512, A=128, E=256, V=6400, T=20, B=256),
    "c3": dict(kind="train", arch="resnet101", D=2048, size=14, L=196, H=1024, A=128, E=256, V=6400, T=20, B=512),
    "greedy": dict(kind="decode", arch="resnet50", D=512, size=14, L=196, H=512, A=128, E=256, V=6400, k=1, S=30, B=1024),
    "beam": dict(kind="decode", arch="wide_resnet101_2", D=2048, size=16, L=256, H=512, A=128, E=256, V=10000, k=5, S=30, B=256),
}
# bounded CPU samples of the same workloads (captions per timed step of the reference arm / cpu_baseline)
CPU_SAMPLE = {"train": 16, "c3": 8, "greedy": 8, "beam": 4}
DUMP_SAMPLE = 1 << 18
DUMP_MAX_BYTES = 64 << 20


def vocab(V):
    stoi = {"<PAD>": 0}
    for i in range(1, V - 3):
        stoi["w%d" % i] = i
    stoi["<UNK>"], stoi["<START>"], stoi["<END>"] = V - 3, V - 2, V - 1
    return stoi, {v: k for k, v in stoi.items()}


def hparams(c, precision="bf16", **over):
    stoi, itos = vocab(c["V"])
    hp = dict(encoder_arch=c["arch"], pretrained=False, input_size=224, encoder_dim=c["D"], encoder_size=c["size"],
              mean=[0.485, 0.456, 0.406], std=[0.229, 0.224, 0.225], embed_dim=c["E"], embed_norm=None,
              attention_dim=c["A"], decoder_dim=c["H"], decoder_layers=1, dropout=0.0, embedding_dropout=0.0,
              label_smoothing=0.0, weight_tying=False, deep_output=True, vocab_size=c["V"], vocab_stoi=stoi,
              vocab_itos=itos, pretrained_embedding=None, att_gamma=1.0, decoder_tf="always", precision=precision,
              opt="adam", decoder_lr=4e-4, embedding_lr=4e-4, encoder_lr=1e-4, weight_decay=0.0,
              encoder_finetune_after=-1)
    hp.update(over)
    return hp


def synth_batch(B, T, V, seed, device="cpu", pin=False):
    g = torch.Generator().manual_seed(seed)
    img = torch.rand(B, 3, 224, 224, generator=g)
    caps = torch.randint(1, V - 3, (B, 1, T + 1), generator=g)
    caps[:, :, 0] = V - 2
    caps[:, :, T] = V - 1
    lens = torch.full((B, 1), T, dtype=torch.long)
    if pin:
        img, caps, lens = img.pin_memory(), caps.pin_memory(), lens.pin_memory()
    if device != "cpu":
        img, caps, lens = img.to(device), caps.to(device), lens.to(device)
    return img, caps, lens


def workload_string(name, c, B):
    if c["kind"] == "train":
        return ("train_step: SAT %s encoder (pretrained=False, encoder_size=%d -> L=%d), D=%d, A=%d, E=%d, H=%d, V=%d, T=%d targets, "
                "batch %d per GPU, teacher-forced fwd+loss+bwd+Adam" % (c["arch"], c["size"], c["L"], c["D"], c["A"], c["E"], c["H"],
                                                                          c["V"], c["T"], B))
    return ("%s decode: %s encoder, L=%d, D=%d, H=%d, V=%d, beamk=%d, max_gen_length=%d, batch %d images per GPU"
            % (name, c["arch"], c["L"], c["D"], c["H"], c["V"], c["k"], c["S"], B))


def config_dict(name, c, B, gpus):
    s = 2
    if c["kind"] == "train":
        l2 = "working set > L2: encoder activations of a batch-%d %s step (GBs) are rewritten every step" % (B, c["arch"])
        par = "dp%d" % gpus
    else:
        l2 = ("annotations + P (%.0f MB) exceed or rival L2; logits / statistics [rows,V] are rewritten every step"
              % (B * c["L"] * (c["D"] + c["A"]) * s / 1e6))
        par = "independent shards x%d" % gpus
    return {"workload": workload_string(name, c, B), "global_batch": B * gpus, "parallelism": par, "l2": l2,
            **({"caption_len": c["T"]} if c["kind"] == "train" else {})}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                       "-lms", "100"], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(", ") for r in open(self.f.name) if r.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for n, v in zip(names, r[5:9]):
                    if v.strip().lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        busy = [s for s in sm if s > 0]
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def load_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


def load_traffic(workload):
    """DRAM bytes per launch of the named kernels from the committed `ncu --set full` captures of the same decoder workloads
    (profiles/r02_kernel_traffic.json, one entry per workload, written by tools/ncu_traffic.py from tools/profile_round2.sh's
    .ncu-rep files); {} when that workload has no capture (traffic: null)."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "r02_kernel_traffic.json")))
    except Exception:
        return {}
    if workload in d:
        return d[workload]
    return d if (workload == "train" and "attention_step_fwd_pipe_kernel" in d) else {}


# ------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the unmodified reference (SAT_REFERENCE_DIR or oracle/_ref) on the host cores
# ------------------------------------------------------------------------------------------------
def _reference_model(c):
    """(kind, SAT module) -- kind 'reference' = the unmodified reference's SAT driven through oracle/ref_harness, with the
    readme's own resize layer appended to its encoder (readme.md:118-121); 'port' = not available (oracle port is used)."""
    from oracle import ref_harness as rh
    if not rh.available():
        return "port", None
    from torch import nn
    model_mod, _ = rh.load_reference()
    stoi, itos = vocab(c["V"])
    hp = rh.default_hparams(encoder_arch=c["arch"], encoder_dim=c["D"], embed_dim=c["E"], attention_dim=c["A"], decoder_dim=c["H"],
                            vocab_size=c["V"], vocab_stoi=stoi, vocab_itos=itos, encoder_finetune_after=1)
    torch.manual_seed(0)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        m = model_mod.SAT(**hp)
    m.encoder = nn.Sequential(*m.encoder, nn.Upsample((c["size"], c["size"]), mode="bilinear", align_corners=False))
    return "reference", m


def cpu_train(name, steps, warmup):
    """reference train step (training_step: encoder fwd, decoder fwd, loss; backward; Adam) at a bounded batch, fp32, all cores."""
    c = CFG[name]
    sample_B = CPU_SAMPLE[name]
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    kind, m = _reference_model(c)
    img, caps, lens = synth_batch(sample_B, c["T"], c["V"], seed=1)
    if kind == "reference":
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            opt = m.configure_optimizers()
        m._optimizer = opt
        m.train()

        def step(i):
            opt.zero_grad(set_to_none=True)
            out = m.training_step((img.clone(), caps, lens), i)        # the reference normalises the images in place
            out["loss"].backward()
            opt.step()
    else:
        from oracle import sat_oracle as O
        torch.manual_seed(0)
        enc = O.build_encoder(c["arch"], c["D"], c["size"]).train()
        W = {k: v.requires_grad_(True) for k, v in O.random_weights(c["D"], c["A"], c["E"], c["H"], c["V"], seed=0).items()}
        opt = torch.optim.Adam(list(enc.parameters()) + list(W.values()), lr=1e-4)

        def step(i):
            opt.zero_grad(set_to_none=True)
            r = O.train_loss(W, enc(img.clone()), caps, lens, 0.0, 1.0)
            r["loss"].backward()
            opt.step()
    times = []
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for it in range(warmup + steps):
            t0 = time.perf_counter()
            step(it)
            if it >= warmup:
                times.append(time.perf_counter() - t0)
    tot = sum(times)
    what = ("unmodified reference SAT.training_step + backward + Adam" if kind == "reference" else "oracle port of the reference train step")
    return dict(value=sample_B * len(times) / tot, ms_per_step=1e3 * tot / len(times), p50_ms=1e3 * statistics.median(times), cores=cores,
                kind=kind, sample_B=sample_B,
                sample="%s (%s encoder fwd+bwd, decoder fwd+loss+bwd) on a bounded sample of %d captions per step of the batch-%d "
                       "workload, %d timed steps after %d warm-ups, fp32, torch CPU, %d threads" % (what, c["arch"], sample_B, c["B"],
                                                                                                  len(times), warmup, cores))


def cpu_decode(name, steps, warmup):
    """reference SAT.caption (encoder + per-image beam loop) on a bounded number of images."""
    c = CFG[name]
    n = CPU_SAMPLE[name]
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    kind, m = _reference_model(c)
    g = torch.Generator().manual_seed(1)
    img = torch.rand(n, 3, 224, 224, generator=g)
    if kind == "reference":
        def step():
            m.caption(img.clone(), beamk=c["k"], max_gen_length=c["S"])
    else:
        from oracle import sat_oracle as O
        W = O.random_weights(c["D"], c["A"], c["E"], c["H"], c["V"], seed=0)
        enc = O.build_encoder(c["arch"], c["D"], c["size"]).eval()
        voc = dict(PAD=0, UNK=c["V"] - 3, START=c["V"] - 2, END=c["V"] - 1)

        def step():
            O.caption(W, enc(img.clone()), voc, beamk=c["k"], max_gen_length=c["S"])
    times = []
    with torch.no_grad(), warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for it in range(warmup + steps):
            t0 = time.perf_counter()
            step()
            if it >= warmup:
                times.append(time.perf_counter() - t0)
    tot = sum(times)
    what = "unmodified reference SAT.caption" if kind == "reference" else "oracle port of SAT.caption"
    return dict(value=n * len(times) / tot, ms_per_step=1e3 * tot / len(times), p50_ms=1e3 * statistics.median(times), cores=cores, kind=kind,
                sample_B=n, sample="%s (%s encoder + per-image beam loop, beamk=%d, max_gen_length=%d) on a bounded sample of %d images per "
                                   "step of the batch-%d workload, %d timed steps after %d warm-ups, fp32, torch CPU, %d threads"
                                   % (what, c["arch"], c["k"], c["S"], n, c["B"], len(times), warmup, cores))


def cpu_workload(name, steps, warmup):
    return cpu_train(name, steps, warmup) if CFG[name]["kind"] == "train" else cpu_decode(name, steps, warmup)


def reference_record(name, r, args):
    c = CFG[name]
    cfg = config_dict(name, c, c["B"], args.gpus)
    cfg["workload"] += "; CPU reference arm timed on a bounded sample of %d captions per step" % r["sample_B"]
    cfg["device"] = "cpu"
    return {
        "impl": "reference", "metric": METRIC, "value": r["value"], "unit": "captions/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "step_p50_ms": r["p50_ms"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
        "cpu_baseline": {"value": r["value"], "unit": "captions/s", "cores": r["cores"], "kind": r["kind"], "sample": r["sample"]},
        "e2e": {"value": r["value"], "unit": "captions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    names = ["train", "c3", "greedy", "beam"] if args.workload == "all" else [args.workload]
    head = names[0]
    line = reference_record(head, cpu_workload(head, args.steps, args.warmup), args)
    for n in names[1:]:
        sub_steps = max(1, min(args.steps, 3))               # bounded: the whole arm ends within a few minutes
        rec = reference_record(n, cpu_workload(n, sub_steps, min(args.warmup, 1)), args)
        rec["steps"], rec["warmup"] = sub_steps, min(args.warmup, 1)
        for k in ("impl", "metric", "n_gpus", "higher_is_better", "scaling", "vs_baseline", "data"):
            rec.pop(k, None)
        line[n] = rec
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------------
class Dist:
    def __init__(self):
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=self.dev)

    def barrier(self):
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def max_ms(self, ms):
        if self.world > 1:
            import torch.distributed as dist
            t = torch.tensor([ms], device=self.dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return ms

    def close(self):
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()
            dist.destroy_process_group()


def timed(D, fn, steps, warmup, drain=None):
    """W untimed warm-ups, then exactly `steps` steps between barrier + synchronize on both sides; CUDA-event time, max over ranks"""
    for _ in range(warmup):
        fn()
    if drain is not None:
        drain()
    D.barrier()
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
    evs[0].record()
    for i in range(steps):
        fn()
        if drain is not None and i == steps - 1:
            drain()
        evs[i + 1].record()
    D.barrier()
    per = [evs[i].elapsed_time(evs[i + 1]) for i in range(steps)]
    return D.max_ms(evs[0].elapsed_time(evs[steps])), per


def dump_array(x):
    """host float32 / float64 copy of an output; above DUMP_SAMPLE elements, the fixed seeded sample of its flattened elements"""
    x = x.detach()
    if x.numel() > DUMP_SAMPLE:
        idx = torch.randint(0, x.numel(), (DUMP_SAMPLE,), generator=torch.Generator().manual_seed(0)).sort().values
        x = x.reshape(-1)[idx.to(x.device)]
    x = x.cpu()
    return (x if x.dtype == torch.float64 else x.float()).numpy()


def train_outputs(model, loss, aux):
    """what the last timed train step computed: its loss and statistics, and the parameter gradients it left"""
    out = {"loss": dump_array(loss), "aux": dump_array(aux)}
    enc = []
    for n, p in model.named_parameters():
        if p.grad is None:
            continue
        if n.startswith("encoder."):
            enc.append(p.grad.reshape(-1).float())
        else:
            out["grad." + n] = dump_array(p.grad)
    if enc:
        out["grad.encoder"] = dump_array(torch.cat(enc))
    return out


def decode_outputs(t, c):
    """the returned caption of every image of the last timed decode (decode.assemble, as SAT.caption returns them), padded to
    arrays"""
    import numpy as np
    from sat_b200 import decode
    caps, scores, alphas, ppls = decode.assemble(t, (c["size"], c["size"]))
    B, W = len(caps), c["S"] + 1
    tokens = torch.full((B, W), -1.0)
    alpha = torch.zeros(B, W, c["L"])
    for i, (cap, a) in enumerate(zip(caps, alphas)):
        tokens[i, :len(cap)] = torch.tensor(cap, dtype=torch.float32)
        alpha[i, :a.shape[0]] = a.reshape(a.shape[0], c["L"])
    return {"tokens": dump_array(tokens), "lengths": np.array([len(x) for x in caps], dtype=np.float32),
            "scores": np.array(scores, dtype=np.float64), "perplexities": np.array(ppls, dtype=np.float64),
            "alphas": dump_array(alpha)}


def write_outputs(path, outputs):
    import numpy as np
    arrays = {"%s.%s" % (w, k): v for w, o in outputs.items() for k, v in o.items()}
    total = sum(v.nbytes for v in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise RuntimeError("--dump-outputs: %d bytes exceed the %d-byte budget" % (total, DUMP_MAX_BYTES))
    os.makedirs(path, exist_ok=True)
    for name, v in arrays.items():
        np.save(os.path.join(path, name + ".npy"), v)


def roof_entry(kernel, bound, work, ms, n, peak, unit, traffic, traffic_keys=None, **extra):
    """`traffic`: the committed ncu capture of THIS workload ({} = none: traffic null); traffic_keys: entries of it to sum
    (default: the kernel's own name)"""
    per_launch_s = ms / max(n, 1) * 1e-3
    scale = 1e9 if unit == "GB/s" else 1e12
    achieved = work / per_launch_s / scale if n else None
    tr = None
    if isinstance(traffic, dict) and traffic:
        # every key is a substring of exactly one captured kernel name (template arguments included)
        hits = [[v for k, v in traffic.items() if sub in k] for sub in (traffic_keys or [kernel])]
        if all(len(h) == 1 for h in hits):
            tr = sum(h[0]["dram_bytes_per_launch"] for h in hits)
    e = {"kernel": kernel, "bound": bound, "achieved": achieved, "peak": peak, "unit": unit, "frac": (achieved / peak) if achieved else None,
         "traffic": tr, "launches_timed": n, "avg_launch_us": 1e6 * per_launch_s}
    e["algorithmic_%s_per_launch" % ("bytes" if bound == "hbm" else "flops")] = work
    e.update(extra)
    return e


def run_train(args, D, name, outputs=None):
    from sat_b200 import _lib, decoder
    from sat_b200.dist import OverlappedGradReducer
    from sat_b200.model import SAT
    from sat_b200.packing import PARAM_NAMES, PackedWeights

    c = CFG[name]
    world, rank, dev = D.world, D.rank, D.dev
    B = args.batch if (args.batch and name == "train") else c["B"]
    T, V = c["T"], c["V"]
    torch.manual_seed(0)                       # identical replicas
    model = SAT(**hparams(c, precision=args.precision)).to(dev)
    if args.precision == "bf16":
        model.encoder.to(memory_format=torch.channels_last)
    model.train()
    opt = model.configure_optimizers()
    enc_params = [p for p in model.encoder.parameters() if p.requires_grad]
    dec_params = [p for n, p in model.named_parameters() if not n.startswith("encoder.") and p.requires_grad]
    # SAT_BENCH_NO_REDUCE=1: diagnosis only (replicas without the gradient exchange, to separate communication cost from
    # two-process effects); the record is marked and is not a valid data-parallel number
    no_reduce = world > 1 and os.environ.get("SAT_BENCH_NO_REDUCE", "0") == "1"
    reducer = OverlappedGradReducer(dec_params, enc_params) if (world > 1 and not no_reduce) else None
    img_d, caps_d, lens_d = synth_batch(B, T, V, seed=100 + rank, device=dev)
    img_h, caps_h, lens_h = synth_batch(B, T, V, seed=100 + rank, pin=True)

    def backward_and_step(loss):
        if reducer is not None:
            reducer.prepare()                  # bucket views zeroed, hooks armed: all-reduces start inside backward()
        else:
            opt.zero_grad(set_to_none=True)
        loss.backward()
        if reducer is not None:
            reducer.finish()
        opt.step()

    last = {}

    def step_device():
        loss, aux = model.fused_loss((img_d.clone(), caps_d, lens_d))
        backward_and_step(loss)
        last["loss"], last["aux"] = loss, aux
        return loss

    # End-to-end step = what a training loop around the public API does: the NEXT batch's host->device copy is issued on a
    # copy stream while the current step computes (input prefetch), and each step's loss is read back through a pinned
    # buffer one step late, so neither copy stalls the launch queue.  Every timed step still issues one H2D copy of a
    # full batch and one D2H read of a loss; the last loss is drained before the closing event.
    copy_stream = torch.cuda.Stream()
    pending = {}
    loss_pin = [torch.zeros(1, dtype=torch.float32).pin_memory() for _ in range(2)]
    loss_ev = [torch.cuda.Event() for _ in range(2)]
    e2e_state = {"i": 0, "last": None}

    def prefetch():
        with torch.cuda.stream(copy_stream):
            pending["batch"] = (img_h.to(dev, non_blocking=True), caps_h.to(dev, non_blocking=True), lens_h.to(dev, non_blocking=True))
            pending["ev"] = torch.cuda.Event()
            pending["ev"].record(copy_stream)

    def step_e2e():
        if "batch" not in pending:
            prefetch()
        cur = torch.cuda.current_stream()
        cur.wait_event(pending["ev"])
        img, caps, lens = pending.pop("batch")
        for x in (img, caps, lens):
            x.record_stream(cur)
        prefetch()                                  # next batch's H2D overlaps this step's compute
        m = model.training_step((img, caps, lens), 0)
        backward_and_step(m["loss"])
        i = e2e_state["i"]
        loss_pin[i & 1].copy_(m["loss"].detach().reshape(1).float(), non_blocking=True)     # device -> host read of the step's result
        loss_ev[i & 1].record()
        if i > 0:
            loss_ev[(i - 1) & 1].synchronize()
            e2e_state["last"] = float(loss_pin[(i - 1) & 1][0])
        e2e_state["i"] = i + 1
        return e2e_state["last"]

    def drain_e2e():
        i = e2e_state["i"]
        if i > 0:
            loss_ev[(i - 1) & 1].synchronize()
            e2e_state["last"] = float(loss_pin[(i - 1) & 1][0])

    clocks = ClockSampler(D.local)
    l0 = _lib.launch_count()
    clocks.start()
    tot_ms, per = timed(D, step_device, args.steps, args.warmup)
    clk = clocks.stop()
    if outputs is not None:
        outputs[name] = train_outputs(model, last["loss"], last["aux"])
    launches = (_lib.launch_count() - l0) * args.steps // (args.steps + args.warmup)
    value = B * world * args.steps / (tot_ms * 1e-3)
    e2e_ms, _ = timed(D, step_e2e, args.steps, args.warmup, drain=drain_e2e)
    e2e_value = B * world * args.steps / (e2e_ms * 1e-3)
    h2d = img_h.numel() * 4 + caps_h.numel() * 8 + lens_h.numel() * 8

    # decoder-only (annotations resident): weight pack + fwd + loss + BPTT + parameter gradients, all inside the library
    with torch.no_grad():
        ann = model.encode(img_d.clone())
    cfg = model._cfg()
    W = {n: p for n, p in zip(PARAM_NAMES, model.decoder_weights()) if p is not None}
    bld = decoder.annotations_as_bld(ann, cfg["dtype"])
    pw = PackedWeights(W, dtype=cfg["dtype"], device=dev, backward=True)

    def dec_step():
        pw.repack(W)
        buf = decoder.train_forward(pw, bld, caps_d, lens_d, 0.0, 1.0, exact=cfg["exact"], use_tc=cfg["use_tc"], backward=True, fuse_ce=True)
        decoder.train_backward(pw, buf)

    dec_ms, dec_per = timed(D, dec_step, args.steps, args.warmup)

    # rooflines: in-situ device time of the named kernels' launches (CUDA events around every launch inside the decoder step)
    peaks, traffic = load_peaks(), (load_traffic(name) if B == c["B"] else {})
    hbm = float(peaks.get("hbm_gbs", 6650.0))
    tfl = float(peaks.get("bf16_tflops", 1590.0))
    src = "MEASURED_PEAKS.json (hbm_gbs, bf16_tflops burst)" if peaks else "fallback 6650 GB/s / 1590 TFLOP/s"
    s = 2 if cfg["dtype"] == torch.bfloat16 else 4
    L, Dd, A, E, H = c["L"], c["D"], c["A"], c["E"], c["H"]
    M = T * B

    def prof(kind):
        _lib.profile_begin(kind)
        for _ in range(3):
            dec_step()
        return _lib.profile_end()

    att_ms, att_n = prof(1)
    roof = roof_entry("attention_step_fwd_pipe_kernel", "hbm", B * (L * (A + Dd) * s + (H + 2 * Dd) * s + 4 * L), att_ms, att_n, hbm, "GB/s",
                      traffic, peak_source=src)
    attb_ms, attb_n = prof(2)
    voc_ms, voc_n = prof(3)
    gate_ms, gate_n = prof(4)
    roof["other_kernels"] = [
        roof_entry("attention_step_bwd_pipe_kernel", "hbm", B * (L * (A + Dd) * s + 2 * Dd * s + 8 * L), attb_ms, attb_n, hbm, "GB/s", traffic),
        roof_entry("gemm_tn_tc_kernel<EpiVocab> x2 + ce_finalize_kernel (fused vocabulary projection + cross entropy)", "tensor",
                   2 * 2.0 * M * V * E, voc_ms, voc_n, tfl, "TFLOP/s", traffic,
                   traffic_keys=["EpiVocab<0>", "EpiVocab<1>"],
                   note="one launch group = statistics pass + row finalize + dlogits pass (the logits are computed twice, never stored)"),
        roof_entry("gemm_tn_tc_kernel<EpiLstm> (gate GEMM + LSTM cell)", "tensor", 2.0 * B * Dd * 4 * H, gate_ms, gate_n, tfl, "TFLOP/s", traffic,
                   traffic_keys=["EpiLstm"], note="M = batch rows only: launch / latency bound, see DESIGN.md"),
    ]
    rec = {
        "value": value, "unit": "captions/s", "steps": args.steps, "warmup": args.warmup, "ms_per_step": tot_ms / args.steps,
        "step_p50_ms": statistics.median(per), "steps_ms": [round(x, 3) for x in per], "dtype": "bf16" if args.precision == "bf16" else "f32",
        "config": dict(config_dict(name, c, B, world), **({"INVALID_no_gradient_exchange": True} if no_reduce else {})), "clocks": clk,
        "e2e": {"value": e2e_value, "unit": "captions/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                "ms_per_step": e2e_ms / args.steps},
        "gpu_launches": int(launches),
        "decoder_only": {"value": B * world * args.steps / (dec_ms * 1e-3), "unit": "captions/s", "ms_per_step": dec_ms / args.steps,
                         "p50_ms": statistics.median(dec_per),
                         "what": "weight pack + decoder fwd + loss + BPTT + parameter gradients (all libsat_b200 kernels), annotations resident"},
        "roofline": roof,
    }
    if reducer is not None:
        # self-check of the data-parallel path (untimed): after one step's exchange every rank must hold the same gradients,
        # and they must differ from the rank's own local gradients (the ranks see different data)
        import torch.distributed as dist
        probe = [p for p in dec_params[:3] + enc_params[:2] + enc_params[-2:]]
        loss, _ = model.fused_loss((img_d.clone(), caps_d, lens_d))
        opt.zero_grad(set_to_none=True)
        loss.backward()
        local = torch.stack([p.grad.double().sum() for p in probe])
        loss, _ = model.fused_loss((img_d.clone(), caps_d, lens_d))
        reducer.prepare()
        loss.backward()
        reducer.finish()
        mine = torch.stack([p.grad.double().sum() for p in probe])
        both = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(both, mine)
        assert all(torch.equal(both[0], b) for b in both), "gradients differ across ranks after the all-reduce"
        assert not torch.allclose(mine, local, rtol=1e-6, atol=0), "all-reduce left the local gradients unchanged"
        opt.zero_grad(set_to_none=True)
    if reducer is not None:
        reducer.close()
    del model, opt, reducer
    torch.cuda.empty_cache()
    return rec


def run_decode(args, D, name, outputs=None):
    from sat_b200 import _lib, decode, decoder
    from sat_b200.model import SAT
    c = CFG[name]
    world, rank, dev = D.world, D.rank, D.dev
    torch.manual_seed(0)
    model = SAT(**hparams(c, precision=args.precision)).to(dev).eval()
    if args.precision == "bf16":
        model.encoder.to(memory_format=torch.channels_last)
    B = c["B"]
    g = torch.Generator().manual_seed(100 + rank)
    img_h = torch.rand(B, 3, 224, 224, generator=g).pin_memory()
    dw = decode.inference_weights(model)
    with torch.no_grad():
        ann = torch.cat([model.encode(img_h[i:i + 128].to(dev)) for i in range(0, B, 128)], 0)
    bld = decoder.annotations_as_bld(ann, dw.pw.dtype)
    voc = dict(PAD=0, UNK=c["V"] - 3, START=c["V"] - 2, END=c["V"] - 1)

    last = {}

    def step_device():
        last["t"] = decode.decode_annotations(dw, bld, c["k"], c["S"], 1.0, None, 0.5, voc)
        return last["t"]

    def step_e2e():
        # public bulk-captioning call: pinned host images in chunks of 256 (encoder activation memory); copies, kernels
        # and the host-side list assembly of consecutive chunks overlap inside caption_stream
        chunks = (img_h[i:i + 256] for i in range(0, B, 256))
        return list(model.caption_stream(chunks, beamk=c["k"], max_gen_length=c["S"]))

    clocks = ClockSampler(D.local)
    l0 = _lib.launch_count()
    clocks.start()
    tot_ms, per = timed(D, step_device, args.steps, args.warmup)
    clk = clocks.stop()
    if outputs is not None:
        outputs[name] = decode_outputs(last["t"], c)
    launches = (_lib.launch_count() - l0) * args.steps // (args.steps + args.warmup)
    value = B * world * args.steps / (tot_ms * 1e-3)
    e2e_ms, _ = timed(D, step_e2e, args.steps, 1)
    e2e_value = B * world * args.steps / (e2e_ms * 1e-3)

    _lib.profile_begin(1)
    for _ in range(2):
        step_device()
    att_ms, att_n = _lib.profile_end()
    _lib.profile_begin(3)
    for _ in range(2):
        step_device()
    voc_ms, voc_n = _lib.profile_end()
    s = 2 if dw.pw.dtype == torch.bfloat16 else 4
    R = B * c["k"]
    peaks, traffic = load_peaks(), load_traffic(name)
    hbm = float(peaks.get("hbm_gbs", 6650.0))
    tfl = float(peaks.get("bf16_tflops", 1590.0))
    att_bytes = B * c["L"] * (c["A"] + c["D"]) * s + R * ((c["H"] + 2 * c["D"]) * s + 4 * c["L"])   # per image-step + per row
    kname = "attention_step_fwd_group_tcr_kernel" if c["k"] > 1 else "attention_step_fwd_pipe_kernel"
    roof = roof_entry(kname, "hbm", att_bytes, att_ms, att_n, hbm, "GB/s", traffic,
                      peak_source="MEASURED_PEAKS.json (hbm_gbs, bf16_tflops burst)" if peaks else "fallback 6650 GB/s / 1590 TFLOP/s")
    roof["other_kernels"] = [roof_entry("vocabulary GEMM (gemm_tn_tc_kernel, M = live rows)", "tensor", 2.0 * R * c["V"] * c["E"], voc_ms, voc_n,
                                        tfl, "TFLOP/s", traffic, traffic_keys=["EpiVocab<2>" if c["k"] == 1 else "gemm_tn_tc_kernel<128, EpiStore"])]
    rec = {
        "value": value, "unit": "captions/s", "steps": args.steps, "warmup": args.warmup, "ms_per_step": tot_ms / args.steps,
        "step_p50_ms": statistics.median(per), "dtype": "bf16" if args.precision == "bf16" else "f32",
        "config": config_dict(name, c, B, world), "clocks": clk,
        "e2e": {"value": e2e_value, "unit": "captions/s", "h2d_bytes_per_step": img_h.numel() * 4,
                "d2h_bytes_per_step": int(B * (c["S"] + 1) * 4 * 2 + B * c["S"] * c["L"] * 4), "ms_per_step": e2e_ms / args.steps,
                "steps": args.steps},
        "gpu_launches": int(launches), "roofline": roof,
    }
    del model, dw, bld, ann
    torch.cuda.empty_cache()
    return rec


def run_b200(args):
    D = Dist()
    names = ["train", "c3", "greedy", "beam"] if args.workload == "all" else [args.workload]
    recs = {}
    outputs = {} if (args.dump_outputs and D.rank == 0) else None
    for n in names:
        recs[n] = run_train(args, D, n, outputs) if CFG[n]["kind"] == "train" else run_decode(args, D, n, outputs)
    if outputs is not None:
        write_outputs(args.dump_outputs, outputs)
    head = names[0]
    line = {"metric": METRIC, "n_gpus": D.world, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "data": "synthetic"}
    line.update(recs[head])
    for n in names[1:]:
        line[n] = recs[n]
    if D.world > 1:
        import torch.distributed as dist
        dist.barrier()
    if D.rank == 0:
        if D.world == 1 and not args.no_cpu_baseline:
            for n in names:
                r = cpu_workload(n, steps=5 if n == "train" else 3, warmup=1)       # ≈20 s of host time in total
                cb = {"value": r["value"], "unit": "captions/s", "cores": r["cores"], "kind": r["kind"], "sample": r["sample"]}
                if n == head:
                    line["cpu_baseline"] = cb
                else:
                    line[n]["cpu_baseline"] = cb
        print(json.dumps(line), flush=True)
    D.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="all", choices=["all", "train", "c3", "greedy", "beam"])
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch of the train workload (default: the BASELINE config's)")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--no-cpu-baseline", dest="no_cpu_baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what each workload's last timed step computed to DIR/<workload>.<output>.npy (B200 arm)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the B200 arm")
    if args.impl == "reference":
        return run_reference(args)
    args.warmup = max(args.warmup, 3)
    return run_b200(args)


if __name__ == "__main__":
    main()
