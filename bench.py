#!/usr/bin/env python
"""bench.py — explanations/sec of the transformer-attribution hot path on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this engine
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU implementation, same metric

A "step" is one pass of the hot path (forward -> class gradient of every attention map -> LRP relprop through
every block -> relu(grad*cam) head-mean -> +I -> rollout) over one batch of synthetic 224x224 images:
BASELINE.json configs[1], ViT-B/16, batch 256 per GPU, random-init weights, start_layer 0.
N > 1: launched by torchrun, one rank per GPU, the batch of every rank is independent ("weak" scaling, no
collective on the data path; the frozen weights are NCCL-broadcast once from rank 0 before the timed region).

One JSON line on stdout (rank 0).  `value` = whole-job expl/s with inputs resident in HBM; `e2e` = the same
metric through the public API (LRP.generate_LRP_batched) with pinned-host inputs and a D2H read of the maps in
every step; `roofline` = the dominant kernel (the z+ Linear-rule contraction) timed alone with CUDA events;
`cpu_baseline` = the CPU oracle/reference timed on this box's host cores on a bounded sample.

--dump-outputs DIR writes what the timed path returned in its last timed step (rank 0) as DIR/<name>.npy, float32 or
float64: the inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch                                                     # noqa: E402
import torch.distributed as dist                                 # noqa: E402

WORKLOADS = {
    "vit_base": dict(kind="vit", factory="vit_base_patch16_224", oracle="vit_base_patch16_224", batch=256, tokens=197,
                     dim=768, depth=12, heads=12, mlp=3072,
                     label="ViT-B/16 transformer_attribution, batch 256, 224x224, start_layer 0"),
    "vit_large": dict(kind="vit", factory="vit_large_patch16_224", oracle="vit_large_patch16_224", batch=128, tokens=197,
                      dim=1024, depth=24, heads=16, mlp=4096,
                      label="ViT-L/16 transformer_attribution, batch 128, 224x224, start_layer 0"),
    "deit_base": dict(kind="vit", factory="deit_base_patch16_224", oracle="deit_base_patch16_224", batch=256, tokens=197,
                      dim=768, depth=12, heads=12, mlp=3072,
                      label="DeiT-B/16 (reference 197-token model) transformer_attribution, batch 256, start_layer 0"),
    "deit_base_distilled": dict(kind="vit", factory="deit_base_distilled_patch16_224",
                                oracle="deit_base_distilled_patch16_224", batch=256, tokens=198, dim=768, depth=12,
                                heads=12, mlp=3072,
                                label="DeiT-B distilled (198 tokens) transformer_attribution, batch 256, start_layer 0"),
    "bert_base": dict(kind="bert", batch=64, tokens=512, dim=768, depth=12, heads=12, mlp=3072,
                      label="BERT-base seq_len 512 Generator.generate_LRP, batch 64, start_layer 0"),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="vit_base", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch (default: the BASELINE config's)")
    ap.add_argument("--flags", type=int, default=-1, help="engine flags (default: best validated path)")
    ap.add_argument("--cpu-samples", type=int, default=12, help="explanations timed for cpu_baseline")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-roofline", action="store_true")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: the BASELINE batch PER GPU (default, what the driver's scaling run uses); strong: the "
                         "BASELINE batch as the GLOBAL batch, sharded over the GPUs (SURVEY 8e: 256 -> 32 per GPU at 8). "
                         "With N > 1 the weak run also reports the strong-scaling numbers under the key 'strong'.")
    ap.add_argument("--no-graph", action="store_true", help="strong-scaling line without CUDA-graph replay")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(path, arrays):
    """Write each tensor of `arrays` (name -> tensor, leading dim = sample) as path/<name>.npy: floating outputs in
    float32, integer ones (class indices) as float64.  When they exceed DUMP_LIMIT_BYTES together, the same fixed,
    seeded sample of rows is taken from each and its row numbers are written as rows.npy."""
    import numpy as np
    arrays = {k: (v.float() if v.is_floating_point() else v.double()).detach().cpu() for k, v in arrays.items()}
    n = next(iter(arrays.values())).shape[0]
    row_bytes = sum(v[:1].numel() * v.element_size() for v in arrays.values())
    if n * row_bytes > DUMP_LIMIT_BYTES:
        keep = max(1, (DUMP_LIMIT_BYTES - 4096) // (row_bytes + 8))         # + 8 bytes per row of rows.npy, headers
        rows = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:keep].sort().values
        arrays = {k: v[rows] for k, v in arrays.items()}
        arrays["rows"] = rows.double()
    os.makedirs(path, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(path, k + ".npy"), v.numpy())


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return dict(hbm_gbs=d["hbm_gbs"], bf16_tflops=d["bf16_tflops"], bf16_sustained=d.get("bf16_tflops_sustained"),
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_sustained=1400.0, source="fallback (B200_PROFILING.md)")


def measured_traffic(key, units=None):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch (group) from the committed ncu --set full capture of the
    same kernel at the same shape (profiles/ncu_traffic.json), or None.  Entries captured at another batch carry
    `bytes_per_unit` (bytes per explanation) and are scaled by `units`."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            e = json.load(f).get(key, {})
        if units is not None and e.get("bytes_per_unit") is not None:
            return int(e["bytes_per_unit"] * units)
        return e.get("bytes")
    except (OSError, ValueError):
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 9:
                    continue
                try:
                    sm.append(float(f[1]))
                    mx.append(float(f[2]))
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))
        return out


def make_model(w, device):
    torch.manual_seed(0)
    if w["kind"] == "bert":
        from transformers import BertConfig
        from transformer_explainability_b200.BERT_explainability.modules.BERT.BertForSequenceClassification import \
            BertForSequenceClassification
        model = BertForSequenceClassification(BertConfig(num_labels=2))
    else:
        from transformer_explainability_b200.baselines.ViT import ViT_LRP
        model = getattr(ViT_LRP, w["factory"])(pretrained=False)
    return model.to(device).eval()


def synthetic_images(batch, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(batch, 3, 224, 224, generator=g)


def synthetic_inputs(w, batch, seed):
    """ViT: randn images.  BERT: ids ~ U{1000..4999}, [CLS]=101 first, [SEP]=102 last, mask all ones (movies documents
    are truncated to 512 and unpadded, bert_pipeline.py:262-271)."""
    if w["kind"] == "bert":
        g = torch.Generator().manual_seed(seed)
        ids = torch.randint(1000, 5000, (batch, w["tokens"]), generator=g)
        ids[:, 0], ids[:, -1] = 101, 102
        return ids
    return synthetic_images(batch, seed)


def explain_call(w, eng, x, batch):
    if w["kind"] == "bert":
        return eng.explain(x, None, start_layer=0, chunk=batch)
    return eng.explain(x, chunk=batch)


def timed_steps(fn, steps, warmup, world):
    """W warm-up steps, then exactly K steps bracketed by barrier + synchronize; CUDA events; max over ranks."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms.item())


def roofline_zplus(w, batch, flags, pk):
    """Dominant kernel: the z+ Linear-rule contraction (fc1/fc2 shapes), timed alone with CUDA events.
    Algorithmic flops per call = 8*rows*in*out (Z = x+W+^T + x-W-^T and S W+, S W-; SURVEY.md §8a)."""
    from transformer_explainability_b200 import ops, _lib
    rows = batch * w["tokens"]
    inf, outf = w["mlp"], w["dim"]                     # fc2 rule: x = gelu(h) [rows, mlp], W [dim, mlp]
    g = torch.Generator(device="cuda").manual_seed(1)
    x = torch.randn(rows, inf, device="cuda", generator=g)
    wt = torch.randn(outf, inf, device="cuda", generator=g) * 0.02
    r = torch.rand(rows, outf, device="cuda", generator=g)
    tc = bool(flags & _lib.FLAG_ZPLUS_TENSOR_CORES)
    bias = torch.randn(outf, device="cuda", generator=g) * 0.02
    y = ops.linear_forward(x, wt, bias) if tc else None          # the engine hands the saved forward output to the rule
    for _ in range(2):
        ops.linear_relprop(x, wt, r, tensor_cores=tc, y=y, bias=bias if tc else None)
    torch.cuda.synchronize()
    reps = 5
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        ops.linear_relprop(x, wt, r, tensor_cores=tc, y=y, bias=bias if tc else None)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    flops = 8.0 * rows * inf * outf
    achieved = flops / (ms * 1e-3) / 1e12
    # TF32 dense peak = half the measured bf16 peak (nominal 1.1 vs 2.25 PF); the fp32 SIMT path is judged
    # against the same tensor roof: it is the baseline the tcgen05 path replaces.
    peak = pk["bf16_tflops"] / 2.0
    traffic = measured_traffic("zplus_tc" if tc else "zplus_simt")
    return {"kernel": "zplus_linear_relprop[%s] rows=%d in=%d out=%d" % ("tcgen05-tf32" if tc else "simt-fp32", rows, inf, outf),
            "bound": "tensor", "achieved": round(achieved, 2), "peak": round(peak, 1), "unit": "TFLOP/s",
            "frac": round(achieved / peak, 4), "traffic": traffic, "ms_per_launch_group": round(ms, 3),
            "algorithmic_flops": flops,
            "executed_flops": (6.0 if tc else 8.0) * rows * inf * outf,
            "note": ("algorithmic = 8*rows*in*out (SURVEY 8a); the tcgen05 path executes 6*rows*in*out: the denominator is "
                     "formed in one pass from the saved forward output, ((y-b) + |x||W|^T)/2; each launch also derives "
                     "the TF32 weight copies (prepare kernel, <1% of the time)") if tc else "fp32 SIMT reference path",
            "peak_source": pk["source"] + "; TF32 dense taken as bf16/2 (tf32_matmul_measured_tflops: cuBLAS TF32 8192^3 on this box)"}


def _time_ms(fn, reps=5, warm=2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def measured_tf32_peak():
    """cuBLAS TF32 matmul 8192^3 (torch.matmul with TF32 allowed), best of 5 — printed beside the bf16/2 convention."""
    try:
        prev = torch.backends.cuda.matmul.allow_tf32
        torch.backends.cuda.matmul.allow_tf32 = True
        a = torch.randn(8192, 8192, device="cuda")
        b = torch.randn(8192, 8192, device="cuda")
        best = min(_time_ms(lambda: torch.matmul(a, b), reps=3, warm=1) for _ in range(5))
        torch.backends.cuda.matmul.allow_tf32 = prev
        return round(2.0 * 8192 ** 3 / (best * 1e-3) / 1e12, 1)
    except Exception:
        return None


def roofline_linear(w, batch, flags, pk):
    """The two Linear GEMM families of the forward / activation-gradient backward at the fc1 shape: 3xTF32 (fp32-grade)
    forward and — with TE_FLAG_BACKWARD_TF32 — the single-pass TF32 backward on the persistent pair kernel."""
    from transformer_explainability_b200 import ops, _lib
    rows, inf, outf = batch * w["tokens"], w["dim"], w["mlp"]
    g = torch.Generator(device="cuda").manual_seed(3)
    x = torch.randn(rows, inf, device="cuda", generator=g)
    wt = torch.randn(outf, inf, device="cuda", generator=g) * 0.02
    bias = torch.randn(outf, device="cuda", generator=g) * 0.02
    dy = torch.randn(rows, outf, device="cuda", generator=g)
    flops = 2.0 * rows * inf * outf
    peak = pk["bf16_tflops"] / 2.0
    out = {}
    tc = bool(flags & _lib.FLAG_LINEAR_TENSOR_CORES)
    f16 = tc and bool(flags & _lib.FLAG_LINEAR_F16_SPLIT)
    ms = _time_ms(lambda: ops.linear_forward(x, wt, bias, tensor_cores=tc, f16_split=f16))
    if f16:
        # fp16 (hi, lo) split: 3 fp16 MMAs per product against the measured bf16/fp16 MMA peak; the timed call includes the
        # weight split (once per model in the engine) and the activation pre-pass (fused into LayerNorm in the engine)
        fpeak = pk["bf16_tflops"]
        out["forward"] = {"kernel": "linear_forward[tcgen05-fp16 split, weight split + block-split pre-pass + GEMM] rows=%d in=%d out=%d" % (rows, inf, outf),
                          "bound": "tensor", "achieved": round(flops / ms / 1e9, 2), "peak": round(fpeak, 1), "unit": "TFLOP/s",
                          "frac": round(flops / ms / 1e9 / fpeak, 4), "ms": round(ms, 3),
                          "note": "fp32-grade: 3 fp16 MMAs per product (issue rate = 3x achieved); peak = measured bf16"}
    else:
        out["forward"] = {"kernel": "linear_forward[%s] rows=%d in=%d out=%d" % ("tcgen05-3xTF32" if tc else "simt-fp32", rows, inf, outf),
                          "bound": "tensor", "achieved": round(flops / ms / 1e9, 2), "peak": round(peak, 1), "unit": "TFLOP/s",
                          "frac": round(flops / ms / 1e9 / peak, 4), "ms": round(ms, 3),
                          "note": "fp32-grade: 3 TF32 MMAs per product (issue rate = 3x achieved)"}
    if tc and (flags & _lib.FLAG_BACKWARD_TF32):
        ms = _time_ms(lambda: ops.linear_backward_tf32(dy, wt))
        what = "tcgen05-TF32 persistent pair"
    else:
        ms = _time_ms(lambda: ops.linear_backward(dy, wt, tensor_cores=tc))
        what = "tcgen05-3xTF32" if tc else "simt-fp32"
    out["backward"] = {"kernel": "linear_backward[%s] rows=%d in=%d out=%d" % (what, rows, inf, outf), "bound": "tensor",
                       "achieved": round(flops / ms / 1e9, 2), "peak": round(peak, 1), "unit": "TFLOP/s",
                       "frac": round(flops / ms / 1e9 / peak, 4), "ms": round(ms, 3)}
    return out


def roofline_rollout(w, flags, pk, B=32, dense=False):
    """The fused-rollout target of the north star: aggregation + rollout over resident G/cam, HBM-bound.
    Algorithmic bytes per explanation = 2*L*H*N^2*4 (+ 4N out; + 4N^2 when the dense joint is returned)  (SURVEY.md §8d).
    dense: the [B,N,N] joint through the aggregation kernel + the N x N x N chain on tcgen05 (compute_rollout_attention's
    consumers); otherwise row 0 only (all generate_LRP reads) through the single fused kernel."""
    from transformer_explainability_b200 import ops, _lib
    L, H, N = w["depth"], w["heads"], w["tokens"]
    ld = (N + 3) // 4 * 4
    g = torch.Generator(device="cuda").manual_seed(2)
    grad = torch.randn(L, B, H, N, ld, device="cuda", generator=g) * 0.05
    cam = torch.randn(L, B, H, N, ld, device="cuda", generator=g) * 0.05
    fused = bool(flags & _lib.FLAG_ROLLOUT_FUSED)
    norm = w["kind"] == "bert"
    ms = _time_ms(lambda: ops.attribution_rollout(grad, cam, normalize=norm, fused=fused, want_joint=dense))
    nbytes = B * (2.0 * L * H * N * N * 4 + 4 * N + (4.0 * N * N if dense else 0.0))
    achieved = nbytes / (ms * 1e-3) / 1e9
    return {"kernel": "attribution_rollout[%s] L=%d B=%d H=%d N=%d" % (
                ("aggregate + tcgen05 N^3 chain, dense joint" if dense else "fused row-only") if fused else "aggregate+bmm", L, B, H, N),
            "bound": "hbm", "achieved": round(achieved, 1), "peak": pk["hbm_gbs"], "unit": "GB/s",
            "frac": round(achieved / pk["hbm_gbs"], 4),
            "traffic": None if dense else measured_traffic("rollout_fused" if fused else "rollout", units=B),
            "algorithmic_bytes": nbytes, "ms": round(ms, 3), "peak_source": pk["source"]}


def cpu_baseline(w, state_dict, n_samples):
    """The reference's CPU path on this box's host cores, B=1 loop (the only mode in which the reference is
    correct).  The real reference when /root/reference is present, else the bit-equal oracle port."""
    from oracle import ref_harness
    from oracle import vit as ovit
    from oracle import cpu as ocpu
    ocpu.set_torch_threads(cap=256)
    xs = synthetic_inputs(w, n_samples + 2, seed=1234)
    sd = {k: v.detach().float().cpu() for k, v in state_dict.items()}
    if w["kind"] == "bert":
        from oracle import bert as obert
        sd = {k: v for k, v in sd.items() if "position_ids" not in k}
        ones = torch.ones(1, w["tokens"], dtype=torch.long)
        if ref_harness.available():
            kind = "reference"
            model = ref_harness.build_bert(state_dict=sd)
            run = lambda x: ref_harness.bert_generate_lrp(model, x, ones, start_layer=0)["map"]      # noqa: E731
        else:
            kind = "port"
            run = lambda x: obert.explain(sd, x, ones, w["heads"], start_layer=0)[0]      # noqa: E731
    elif ref_harness.available():
        kind = "reference"
        model = ref_harness.build_vit(w["oracle"], state_dict=sd)
        run = lambda x: ref_harness.vit_generate_lrp(model, x)["map"]      # noqa: E731
    else:
        kind = "port"
        run = lambda x: ovit.explain(sd, x, w["heads"])[0]                 # noqa: E731
    for i in range(2):
        run(xs[i:i + 1])
    t0 = time.perf_counter()
    for i in range(2, n_samples + 2):
        run(xs[i:i + 1])
    dt = time.perf_counter() - t0
    return {"value": round(n_samples / dt, 4), "unit": "expl/s", "cores": torch.get_num_threads(), "kind": kind,
            "source": ("the reference's own files (%s)" % ("oracle/_ref mirror" if ref_harness.is_mirror() else ref_harness.REF))
            if kind == "reference" else "oracle port (bit-equal to the reference, tests/test_oracle_golden.py)",
            "sample": "%d B=1 explanations of the same workload (2 warm-up), %.1f s" % (n_samples, dt)}


def run_reference_arm(args, w):
    """--impl reference: the reference's own CPU implementation of the path, all host threads, bounded sample."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    model = make_model(w, "cpu")
    per_step = 2
    from oracle import ref_harness
    from oracle import vit as ovit
    from oracle import cpu as ocpu
    ocpu.set_torch_threads(cap=256)
    sd = {k: v.detach().float() for k, v in model.state_dict().items() if "position_ids" not in k}
    if w["kind"] == "bert":
        from oracle import bert as obert
        ones = torch.ones(1, w["tokens"], dtype=torch.long)
        if ref_harness.available():
            kind = "reference"
            ref = ref_harness.build_bert(state_dict=sd)
            run = lambda x: ref_harness.bert_generate_lrp(ref, x, ones, start_layer=0)["map"]      # noqa: E731
        else:
            kind = "port"
            run = lambda x: obert.explain(sd, x, ones, w["heads"], start_layer=0)[0]               # noqa: E731
    elif ref_harness.available():
        kind = "reference"
        ref = ref_harness.build_vit(w["oracle"], state_dict=sd)
        run = lambda x: ref_harness.vit_generate_lrp(ref, x)["map"]        # noqa: E731
    else:
        kind = "port"
        run = lambda x: ovit.explain(sd, x, w["heads"])[0]                 # noqa: E731
    xs = synthetic_inputs(w, per_step * (args.steps + args.warmup), seed=1234)
    i = 0
    for _ in range(args.warmup):
        for _ in range(per_step):
            run(xs[i:i + 1]); i += 1
    t0 = time.perf_counter()
    for _ in range(args.steps):
        maps = []
        for _ in range(per_step):
            maps.append(run(xs[i:i + 1])); i += 1
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"maps": torch.cat(maps)})
    val = per_step * args.steps / dt
    sample = "%d B=1 explanations per step on %d host threads" % (per_step, torch.get_num_threads())
    line = {"impl": "reference", "metric": "explanations_per_sec", "value": round(val, 4), "unit": "expl/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(dt / args.steps * 1e3, 2), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": w["label"], "per_step": sample},
            "cpu_baseline": {"value": round(val, 4), "unit": "expl/s", "cores": torch.get_num_threads(), "kind": kind,
                             "source": ("oracle/_ref mirror of the reference's own files" if ref_harness.is_mirror() else
                                        ref_harness.REF) if kind == "reference" else "oracle port", "sample": sample},
            "e2e": {"value": round(val, 4), "unit": "expl/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def main():
    args = parse()
    w = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference_arm(args, w)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the engine has no CPU fallback")
    from transformer_explainability_b200 import _lib, parallel
    from transformer_explainability_b200.baselines.ViT.ViT_explanation_generator import LRP
    rank, world, local = parallel.init_from_env("nccl")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    lib = _lib.load()
    batch = args.batch or w["batch"]
    flags = args.flags if args.flags >= 0 else default_flags()

    model = make_model(w, dev)
    model.engine_flags = flags
    eng = model.engine()
    if world > 1:
        if rank != 0:
            eng.weights.zero_()
        parallel.broadcast_flat_weights(eng.weights, src=0)          # the one collective of the path
    if w["kind"] == "bert":
        from transformer_explainability_b200.BERT_explainability.modules.BERT.ExplanationGenerator import Generator
        gen = Generator(model)
        public_call = lambda xd: gen.generate_LRP_batched(xd, None, start_layer=0, chunk=batch)      # noqa: E731
    else:
        lrp = LRP(model)
        public_call = lambda xd: lrp.generate_LRP_batched(xd, chunk=batch)                           # noqa: E731

    host = synthetic_inputs(w, batch, seed=100 + rank).pin_memory()
    x_dev = host.to(dev)
    explain_call(w, eng, x_dev[:min(batch, 8)], min(batch, 8))       # allocator / module warm-up (untimed)
    torch.cuda.synchronize()

    last = {}

    def step():
        last["out"] = explain_call(w, eng, x_dev, batch)

    sampler = ClockSampler(local)
    l0 = lib.te_kernel_launch_count()
    sampler.start()
    ms = timed_steps(step, args.steps, args.warmup, world)
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        maps, idx = last["out"]
        dump_outputs(args.dump_outputs, {"maps": maps, "index": idx})
    del last
    launches = (lib.te_kernel_launch_count() - l0) // max(1, (args.steps + args.warmup)) * args.steps
    value = world * batch * args.steps / (ms * 1e-3)

    sink = {}

    def e2e_step():
        xd = host.to(dev, non_blocking=True)                          # H2D of this step's inputs (pinned)
        maps = public_call(xd)                                        # public API
        sink["maps"] = maps.cpu()                                     # D2H read of the step's result

    ms_e2e = timed_steps(e2e_step, args.steps, 1, world)
    e2e = world * batch * args.steps / (ms_e2e * 1e-3)
    finite = bool(torch.isfinite(sink["maps"]).all())

    # ---- strong scaling: the BASELINE batch as the GLOBAL batch, contiguous shards (parallel.shard_range), no collective
    strong = None
    if world > 1 or args.scaling == "strong":
        gb = args.batch or w["batch"]
        lo, hi = parallel.shard_range(gb, rank, world)
        xs = x_dev[:hi - lo]
        strong = {"global_batch": gb, "per_gpu_batch": hi - lo, "unit": "expl/s"}
        variants = [("launches", lambda: explain_call(w, eng, xs, hi - lo))]
        if w["kind"] == "vit" and not args.no_graph:
            variants.append(("cuda_graph", lambda: eng.explain_graphed(xs)))
        for name, fn in variants:
            try:
                ms_s = timed_steps(fn, args.steps, args.warmup, world)
                strong[name] = {"value": round(gb * args.steps / (ms_s * 1e-3), 2), "ms_per_step": round(ms_s / args.steps, 3)}
            except Exception as exc:                                  # the weak line must survive a failure of the extra line
                if name == "launches" or world == 1:
                    raise
                strong[name] = {"error": str(exc)[:200]}
        best = max(v["value"] for k, v in strong.items() if isinstance(v, dict) and "value" in v)
        strong["value"] = best
        strong["note"] = ("global batch %d sharded contiguously over %d GPU(s); limited by tile quantisation of %d token rows "
                          "per GPU, not by launch gaps" % (gb, world, (hi - lo) * w["tokens"]))
        if args.scaling == "strong":
            value, ms = best, gb * args.steps / best * 1e3

    line = {"metric": "explanations_per_sec", "value": round(value, 2), "unit": "expl/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms / args.steps, 3),
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": w["label"], "per_gpu_batch": batch if args.scaling == "weak" else strong["per_gpu_batch"],
                       "global_batch": batch * world if args.scaling == "weak" else strong["global_batch"],
                       "weights": "random-init (reference constructor distributions)", "engine_flags": flags,
                       "l2": "working set exceeds L2 by orders of magnitude: >50 GB of saved activations are written and "
                             "re-read every step (126 MB L2)",
                       "outputs_finite": finite},
            "clocks": clocks,
            "e2e": {"value": round(e2e, 2), "unit": "expl/s", "h2d_bytes_per_step": host.numel() * host.element_size(),
                    "d2h_bytes_per_step": sink["maps"].numel() * 4, "ms_per_step": round(ms_e2e / args.steps, 3)},
            "gpu_launches": int(launches)}
    if strong is not None:
        line["strong"] = strong
    if rank == 0:
        pk = peaks()
        if not args.no_roofline:
            del x_dev
            eng._ws = None
            eng._graphs = {}
            torch.cuda.empty_cache()
            line["roofline"] = roofline_zplus(w, batch, flags, pk)
            line["roofline"]["tf32_matmul_measured_tflops"] = measured_tf32_peak()
            line["roofline_linear"] = roofline_linear(w, batch, flags, pk)
            rb = min(batch, 256 if w["tokens"] <= 256 else 32)
            line["roofline_rollout"] = roofline_rollout(w, flags, pk, B=rb)
            line["roofline_rollout_dense"] = roofline_rollout(w, flags, pk, B=rb, dense=True)       # same batch as the row-only line
        if world == 1 and not args.no_cpu_baseline:
            del eng._ws
            eng._ws = None
            line["cpu_baseline"] = cpu_baseline(w, model.state_dict(), args.cpu_samples)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def default_flags():
    """Best validated kernel selection (see DESIGN.md): updated as faster paths pass parity."""
    from transformer_explainability_b200 import _lib
    # 51 = tcgen05 z+ rule (1) + fused row-only rollout (2) + tcgen05 Linears (16) + attention contractions (32);
    # + 256 single-pass TF32 backward + 1024 single-pass TF32 relevance-side attention products + 2048 bf16 z+ denominator term
    # + 4096 forward Linears as the block-scaled fp16 split  = 7475
    return _lib.FLAG_BENCH_DEFAULT


if __name__ == "__main__":
    main()
