"""Apply-kernel bandwidth per optimizer (1 GPU): SGD and Adam as controls beside
Momentum, Adagrad and RMSProp, in one process.

For each workload -- the 2.0e8-element NMF W set and the 25 557 032-element
ResNet-50 bucket (BASELINE configs) -- and each optimizer it times
  * apply: psx_apply of ONE f32 landing slot (k_apply<OPT, SUM, SlotSrc<f32>>)
  * round: the N = 1 one-kernel psx_round (k_apply<OPT, SUM, SCATTER, PeerSrc<f32>>)
with CUDA events around the kernel launch only.  Every step first rewrites the
gradient (negates the worker's buffer; for `apply` the push copies it into the
slot), outside the timed window; every array is larger than the 126 MB L2.
Algorithmic bytes per element: state (SGD 8, Momentum/Adagrad 16, Adam/RMSProp
24, var and state read + written) + 4 per gradient read (+ 4 per parameter
written by the round).  The share of HBM peak uses bench.py's peak source.
After the timed steps one more step is checked against the CPU restatements on
a strided sample of contiguous chunks (var, state and, for the round, the pulled
parameters), bit for bit.

    python tools/bench_optimizers.py --out DIR [--steps K] [--warmup W]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from oracle import ps_oracle as o  # noqa: E402
from tests import optimizer_oracle as oo  # noqa: E402
from tfmesos_b200 import engine, psx  # noqa: E402

F = np.float32
WORKLOADS = [("nmf_2e8", 200_000_000), ("resnet50_bucket", 25_557_032)]
OPTIMIZERS = [  # name, optimizer, state bytes per element (read + write)
    ("sgd", lambda: engine.GradientDescentOptimizer(0.01), 8),
    ("adam", lambda: engine.AdamOptimizer(0.001), 24),
    ("momentum", lambda: engine.MomentumOptimizer(0.01, 0.9), 16),
    ("adagrad", lambda: engine.AdagradOptimizer(0.01, 0.1), 16),
    ("rmsprop", lambda: engine.RMSPropOptimizer(0.01, 0.9, 0.0, 1e-10), 24),
]
CHUNK, N_CHUNKS = 4096, 64


def hbm_peak():
    """bench.py's source: MEASURED_PEAKS.json if the tree has one, else its fallback."""
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]), \
            "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def card():
    return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()


def chunks(n):
    offs = np.linspace(0, n - CHUNK, N_CHUNKS).astype(np.int64) // 4 * 4
    return [int(x) for x in offs]


def sample(shard, which, n):
    return [shard.get_values(which, off, CHUNK) for off in chunks(n)]


def reference_step(opt_obj, var, m, v, g, state):
    """One update of the sampled elements by the CPU restatements."""
    h = opt_obj.hyper
    if opt_obj.opt == psx.OPT_SGD:
        o.sgd_apply(var, g, h[0])
    elif opt_obj.opt == psx.OPT_ADAM:
        o.adam_apply(var, m, v, g, h[0], h[1], h[2], h[3], state["beta1_power"],
                     state["beta2_power"])
    else:
        oo.apply(opt_obj.opt, var, m, v, g, h)


def n_state(opt_obj):
    return psx.OPT_STATE_ARRAYS[opt_obj.opt]


def run_one(path, n, make_opt, steps, warmup):
    opt_obj = make_opt()
    st = torch.cuda.current_stream()
    sp = st.cuda_stream
    init = torch.randn(n, device="cuda")
    if path == "apply":
        shard = psx.Shard(0, n, opt_obj.opt, *opt_obj.hyper, n_slots=1)
        client = psx.Client(shard.export(), 0, 0)
        grad = torch.randn(n, device="cuda") * 0.01
        cl = None
    else:
        cl = engine.LocalCluster([("w", (n,))], 1, 1, opt_obj, fused=True)
        shard = cl.servers[(0, 0)].shard
        worker = cl.workers[0]
        grad = worker.grad_flat[0][:n]
        grad.copy_(torch.randn(n, device="cuda") * 0.01)
    torch.cuda.synchronize()
    shard.set_values(psx.VAR, init.cpu().numpy())
    del init
    seq = [0]

    def step(e0=None, e1=None):
        grad.neg_()                                    # per-step gradient rewrite
        seq[0] += 1
        if cl is None:
            client.push(grad.data_ptr(), n, seq=seq[0], stream=sp)
            if e0 is not None:
                e0.record(st)
            shard.apply(psx.MODE_SUM, 0, 1, wait_seq=seq[0], stream=sp)
        else:
            worker.signal(seq[0], sp)
            if e0 is not None:
                e0.record(st)
            shard.round(psx.MODE_SUM, 0, 1, seq[0], sp)
        if e1 is not None:
            e1.record(st)
        if cl is not None:
            worker.wait_applied(seq[0], sp)

    for _ in range(warmup):
        step()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
          for _ in range(steps)]
    for e0, e1 in ev:
        step(e0, e1)
    torch.cuda.synchronize()
    ms = [e0.elapsed_time(e1) for e0, e1 in ev]

    # verification: one more step on a strided sample
    k = n_state(opt_obj)
    var = sample(shard, psx.VAR, n)
    m = sample(shard, psx.M, n) if k >= 1 else [np.zeros(CHUNK, F)] * N_CHUNKS
    v = sample(shard, psx.V, n) if k >= 2 else [np.zeros(CHUNK, F)] * N_CHUNKS
    state = shard.state()
    step()
    torch.cuda.synchronize()
    gh = grad.cpu().numpy()
    ok = True
    got_var = sample(shard, psx.VAR, n)
    got_m = sample(shard, psx.M, n) if k >= 1 else None
    got_v = sample(shard, psx.V, n) if k >= 2 else None
    pulled = cl.workers[0].param_flat[0][:n].cpu().numpy() if cl is not None else None
    for c, off in enumerate(chunks(n)):
        x, mm, vv = var[c].copy(), m[c].copy(), v[c].copy()
        reference_step(opt_obj, x, mm, vv, gh[off:off + CHUNK].copy(), state)
        ok &= np.array_equal(x.view(np.uint32), got_var[c].view(np.uint32))
        if k >= 1:
            ok &= np.array_equal(mm.view(np.uint32), got_m[c].view(np.uint32))
        if k >= 2:
            ok &= np.array_equal(vv.view(np.uint32), got_v[c].view(np.uint32))
        if pulled is not None:
            ok &= np.array_equal(x.view(np.uint32), pulled[off:off + CHUNK].view(np.uint32))
    if cl is None:
        client.close()
        shard.destroy()
    else:
        cl.close()
    del grad
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    return ms, bool(ok)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    args = ap.parse_args()
    assert args.warmup >= 3
    assert torch.cuda.is_available(), "needs a CUDA device: no CPU timing is reported"
    os.makedirs(args.out, exist_ok=True)
    psx.init(0)
    peak, peak_src = hbm_peak()
    head = {"card": card(), "hbm_peak_gbs": peak, "peak_source": peak_src,
            "steps": args.steps, "warmup": args.warmup,
            "timed": "CUDA events around the apply / round launch, gradient rewritten per step"}
    lines = [head]
    print(json.dumps(head), flush=True)
    for wname, n in WORKLOADS:
        for path in ("apply", "round"):
            for oname, make_opt, state_bytes in OPTIMIZERS:
                ms, ok = run_one(path, n, make_opt, args.steps, args.warmup)
                n_pad = (n + 1023) // 1024 * 1024
                per_elem = state_bytes + 4 + (4 if path == "round" else 0)
                med = float(np.median(ms))
                gbs = per_elem * n_pad / (med * 1e-3) / 1e9
                rec = {"workload": wname, "nelem": n, "path": path, "opt": oname,
                       "bytes_per_elem": per_elem, "median_ms": med, "min_ms": float(min(ms)),
                       "max_ms": float(max(ms)), "achieved_gbs": gbs, "frac_hbm_peak": gbs / peak,
                       "verified_sample": ok}
                lines.append(rec)
                print(json.dumps(rec), flush=True)
    with open(os.path.join(args.out, "bench_optimizers.jsonl"), "w") as f:
        for rec in lines:
            f.write(json.dumps(rec) + "\n")
    if not all(r.get("verified_sample", True) for r in lines):
        sys.exit("a sampled result differs from the CPU restatement")


if __name__ == "__main__":
    main()
