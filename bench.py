"""Headline benchmark: volumes/sec at 512x512x320 (BASELINE.json: "MIM train step + embedding inference, 1/2/4/8 B200").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

ONE JSON line.  The headline (`value`, `e2e`, `roofline`) is the workload that has a collective and that the north star
sets its scaling target on — BASELINE configs[2], the smb-vision-base MIM pre-training step (forward + norm-pix MSE loss +
backward + bf16 gradient all-reduce over NCCL overlapped with backward + global-norm clip + AdamW), one 512x512x320 volume
per GPU per step — at EVERY N, so that the driver's v_N / (N * v_1) is computed on one and the same workload (round 1
head-lined the collective-free inference pass and the MIM curve sat in a side key the driver does not read).  BASELINE
configs[1], embedding inference (`model.videomae(x)`, volume-sharded, no collective), is the `inference` block of the same
line with its own value / e2e / roofline; configs[3] (classification fine-tune, batch 4/GPU) and configs[4] (V-JEPA step)
are the `classification` and `vjepa_step` blocks.

`--impl reference` times the reference's own CPU path — upstream `transformers.VideoMAEForPreTraining` / `VideoMAEModel`,
the classes the reference imports (src/run_mim.py:19-20, src/run_inference.py:12), UNMODIFIED and at full depth (12 + 4
layers), fp32, sdpa backend, all host threads — on the same synthetic volume: real steps, no extrapolation; the number of
steps actually run is what the line's `steps` says (bounded by a time budget, `steps_requested` keeps the driver's K).

`--dump-outputs DIR` writes what each timed block returned in its last timed step as DIR/<name>.npy (fp32, rank 0; the
large arrays as the same seeded sample of rows in every run, < 64 MB in all).  The inputs and weights are seeded, so two
builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import contextlib
import gc
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "volumes/sec at 512x512x320: MIM train step (embedding inference reported beside it)"
UNIT = "volumes/s"
WORKLOAD = ("smb-vision-base MIM pre-training step (BASELINE configs[2]): 512x512x320 volume = 20480 tokens, 65 % masked, batch 1 volume/GPU, "
            "forward + norm-pix MSE + backward + gradient all-reduce + clip 1.0 + AdamW; bf16 tensor-core operands, fp32 accumulate / master weights")
INFER_WORKLOAD = "smb-vision-base embedding inference (BASELINE configs[1]): model.videomae(x) on one 512x512x320 volume (20480 tokens) per GPU per step"
BASE = {}  # OracleConfig defaults == smb-vision-base at 512x512x320

# algorithmic FLOPs (SURVEY.md §8d)
N_TOK, N_VIS, N_MSK, D, HEADS, LAYERS, MLP = 20480, 7168, 13312, 768, 12, 12, 3072
ATTN_FWD_FLOPS = 4.0 * N_TOK * N_TOK * 64 * HEADS  # 1.2885 TFLOP per launch at the inference shape
EMBED_FLOPS = 2.0 * N_TOK * 4096 * D + LAYERS * (2.0 * N_TOK * D * (3 * D + D + 2 * MLP) + ATTN_FWD_FLOPS)  # 19.07 TFLOP
TRAIN_FLOPS = 18.461e12  # 3 x 6.154 TFLOP forward, no recompute


def attn_bwd_dkdv_flops(H, N):
    """algorithmic work of the dK/dV kernel: dP = dO V^T, dV = P^T dO, dK = dS^T Q (3 x 2 N^2 64 per head); its recomputation
    of S = Q K^T is NOT counted (SURVEY.md §8d: no recompute)."""
    return 6.0 * N * N * 64 * H


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        j = json.load(open(p))
        return dict(hbm=j["hbm_gbs"], tf_burst=j["bf16_tflops"], tf_sust=j.get("bf16_tflops_sustained", j["bf16_tflops"]), src="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, src="fallback (B200_PROFILING.md)")


def ncu_traffic(kernel_key):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of one `ncu --set full` capture, from the newest
    profiles/r*_ncu_traffic.json (written by tools/summarize_ncu.py from the .ncu-rep); (bytes or None, source)."""
    import glob

    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_ncu_traffic.json")), reverse=True):
        try:
            j = json.load(open(path))
        except Exception:
            continue
        for name, rec in j.get("kernels", {}).items():
            if kernel_key in name:
                return rec.get("dram_bytes_per_launch"), f"{os.path.relpath(path, ROOT)}: {name} ({rec.get('shape', '')})"
    return None, "no ncu --set full capture of this kernel under profiles/"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx, self.proc, self.lines = gpu_index, None, []

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=lambda: self.lines.extend(self.proc.stdout), daemon=True)
            self.th.start()
        except Exception:
            self.proc = None
        return self

    def __exit__(self, *a):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=3)
            except Exception:
                self.proc.kill()
            self.th.join(timeout=2)

    def summary(self):
        sm, mx, reasons = [], 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = max(mx, float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=[], samples=0)
        busy = [v for v in sm if v > 0.5 * max(sm)] or sm
        return dict(sm_mhz=statistics.median(busy), sm_max_mhz=mx, reasons=sorted(reasons), samples=len(sm))


# ------------------------------------------------------------------------------------------
# --dump-outputs
# ------------------------------------------------------------------------------------------
DUMP_LIMIT = 64 << 20


def host(t):
    """fp32 host copy of a device tensor."""
    return t.detach().float().cpu().numpy()


def sample_rows(t, rows):
    """fp32 host copy of `rows` rows of t [..., C] (leading dims flattened), chosen by a fixed seed and kept in order, so
    every run samples the same rows; all of them when there are no more than `rows`."""
    import torch

    t = t.detach().reshape(-1, t.shape[-1])
    if t.shape[0] > rows:
        idx = torch.randperm(t.shape[0], generator=torch.Generator().manual_seed(0))[:rows].sort().values
        t = t[idx.to(t.device)]
    return host(t)


def write_dump(out_dir, arrays):
    import numpy as np

    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_LIMIT, f"--dump-outputs: {total} bytes exceed {DUMP_LIMIT}"
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


# ------------------------------------------------------------------------------------------
# CPU legs (rank 0 only; the two places bench.py may execute oracle/ or the upstream classes)
# ------------------------------------------------------------------------------------------
def cpu_baseline_mim():
    """`cpu_baseline` of the GPU arm: the ORACLE PORT (oracle/videomae_oracle.py: fp32 torch restatement of modeling_videomae.py,
    sdpa attention) doing ONE full MIM forward + backward — all 12 + 4 layers, the whole 512x512x320 volume, the seed-0 mask —
    on all host threads.  No extrapolation: the sample IS one step of the workload (≈ 15-25 s)."""
    import numpy as np
    import torch

    from oracle import videomae_oracle as vo
    from oracle.mim_mask import OracleMaskGenerator

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    old, vo.ATTN_IMPL = vo.ATTN_IMPL, "sdpa"
    try:
        cfg = vo.OracleConfig(**BASE)
        sd = {k: v.requires_grad_(True) for k, v in vo.synthetic_state_dict(cfg, 1234).items()}
        x = vo.synthetic_volume(cfg, 1, 7)
        np.random.seed(0)
        mask = torch.from_numpy(OracleMaskGenerator(512, 320, 32, 16, 0.65)()).unsqueeze(0)
        t0 = time.perf_counter()
        loss, _, _ = vo.pretrain_forward(sd, cfg, x, mask)
        loss.backward()
        t = time.perf_counter() - t0
    finally:
        vo.ATTN_IMPL = old
    return {"value": 1.0 / t, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"oracle port (fp32, sdpa): ONE full MIM forward + backward, 12 + 4 layers, whole 512x512x320 volume, 65 % masked: {t:.1f} s "
                      f"(no optimiser step, no extrapolation); loss {float(loss):.6f}"}


def run_reference(args, rank):
    """`--impl reference`: the reference's OWN classes, unmodified, full depth, on the host cores (rank 0 only).
    Headline = MIM training step: `model(x, mask).loss.backward()` + `clip_grad_norm_(1.0)` + `torch.optim.AdamW.step()` of
    `transformers.VideoMAEForPreTraining` (what HF Trainer runs at src/run_mim.py:445 with scripts/training/run_mim.sh:17-21).
    Beside it: `model.videomae(x).last_hidden_state` under no_grad (src/run_inference.py:78-86).  Every timed step is a real,
    complete step; the step count is cut to a time budget and REPORTED (`steps`)."""
    if rank != 0:
        return
    import numpy as np
    import torch
    import transformers

    from __graft_entry__ import hf_config
    from oracle import videomae_oracle as vo  # synthetic volume + mask restatement only
    from oracle.mim_mask import OracleMaskGenerator

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    ocfg = vo.OracleConfig(**BASE)
    cfgd = {k: getattr(ocfg, k) for k in ocfg.__dataclass_fields__}
    x = vo.synthetic_volume(ocfg, 1, 7)
    np.random.seed(0)
    mask = torch.from_numpy(OracleMaskGenerator(512, 320, 32, 16, 0.65)()).unsqueeze(0)
    hc = hf_config(cfgd)
    hc._attn_implementation = "sdpa"
    torch.manual_seed(1234)
    t0 = time.perf_counter()
    model = transformers.VideoMAEForPreTraining(hc)  # (its __init__ builds two sin-cos tables in pure Python: ≈ 1 min at this size)
    t_init = time.perf_counter() - t0
    nd = lambda n: ("bias" in n or "norm" in n)  # Trainer.get_decay_parameter_names
    opt = torch.optim.AdamW([{"params": [p for n, p in model.named_parameters() if not nd(n)], "weight_decay": 0.01},
                             {"params": [p for n, p in model.named_parameters() if nd(n)], "weight_decay": 0.0}], lr=5e-5)

    def train_step():
        t0 = time.perf_counter()
        opt.zero_grad(set_to_none=True)
        loss = model(x, mask).loss
        loss.backward()
        torch.nn.utils.clip_grad_norm_(model.parameters(), 1.0)
        opt.step()
        return time.perf_counter() - t0, float(loss)

    model.train()
    t_warm, _ = train_step()  # one untimed warm-up step (allocator, thread pools)
    steps = int(max(1, min(args.steps, args.ref_budget_s // max(t_warm, 1e-3))))
    times, loss = [], float("nan")
    for _ in range(steps):
        t, loss = train_step()
        times.append(t)
    t_train = sum(times) / len(times)

    enc = model.videomae.eval()
    with torch.no_grad():
        t0 = time.perf_counter()
        y = enc(x).last_hidden_state
        t_iw = time.perf_counter() - t0
        isteps = int(max(1, min(args.steps, (args.ref_budget_s / 2) // max(t_iw, 1e-3))))
        itimes = []
        for _ in range(isteps):
            t0 = time.perf_counter()
            y = enc(x).last_hidden_state
            itimes.append(time.perf_counter() - t0)
    assert tuple(y.shape) == (1, N_TOK, D)
    t_inf = sum(itimes) / len(itimes)
    sample = (f"transformers.VideoMAEForPreTraining (the class the reference imports), unmodified, 12 + 4 layers, fp32, sdpa, {cores} threads, whole "
              f"512x512x320 volume, 65 % masked: {steps} real training steps (forward + backward + clip_grad_norm_ + AdamW) after 1 warm-up, "
              f"mean {t_train:.2f} s/step (min {min(times):.2f}, max {max(times):.2f}); model construction {t_init:.0f} s not timed")
    line = {
        "impl": "reference", "metric": METRIC, "value": 1.0 / t_train, "unit": UNIT, "n_gpus": args.gpus, "steps": steps, "warmup": 1,
        "steps_requested": args.steps, "warmup_requested": args.warmup, "extrapolated": False,
        "ms_per_step": t_train * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "arm": "the reference's own CPU path (upstream VideoMAEForPreTraining, fp32, sdpa, full depth) on the host cores, rank 0 only; "
                                                "every step is a complete real step, the step count is bounded by --ref-budget-s"},
        "cpu_baseline": {"value": 1.0 / t_train, "unit": UNIT, "cores": cores, "kind": "reference", "sample": sample},
        "e2e": {"value": 1.0 / t_train, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "loss_last": loss,
        "inference": {"workload": INFER_WORKLOAD, "value": 1.0 / t_inf, "unit": UNIT, "ms_per_step": t_inf * 1e3, "steps": isteps, "warmup": 1,
                      "e2e": {"value": 1.0 / t_inf, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                      "sample": f"model.videomae(x).last_hidden_state under no_grad, all 12 layers, {isteps} real forwards after 1 warm-up, mean {t_inf:.2f} s"},
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--ref-budget-s", type=float, default=120.0, help="reference arm: time budget of the timed training steps (inference: half)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-inference", action="store_true")
    ap.add_argument("--no-cls", action="store_true")
    ap.add_argument("--no-vjepa", action="store_true")
    ap.add_argument("--no-cuda-graph", action="store_true", help="time the eager step (475 launches) instead of the CUDA-graph replay of forward + backward")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what each timed block returned in its last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    import numpy as np
    import torch
    import torch.distributed as dist

    from __graft_entry__ import hf_config
    from oracle import videomae_oracle as vo  # synthetic inputs only; never on the timed path
    from oracle.mim_mask import OracleMaskGenerator
    from smb_vision_b200 import _lib, ops
    from smb_vision_b200.data import MaskGenerator, VolumePreprocessor
    from smb_vision_b200.modeling import B200VideoMAEForPreTraining, _prep_mask
    from smb_vision_b200.optim import FusedAdamW
    from smb_vision_b200.training import DataParallelStep

    assert torch.cuda.is_available(), "bench.py needs a GPU (use --impl reference for the CPU arm)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    args.warmup = max(args.warmup, 3)
    pk = peaks()

    ocfg = vo.OracleConfig(**BASE)
    cfgd = {k: getattr(ocfg, k) for k in ocfg.__dataclass_fields__}
    torch.manual_seed(1234)
    model = B200VideoMAEForPreTraining(hf_config(cfgd)).to(dev)
    x_host = vo.synthetic_volume(ocfg, 1, 7 + rank).pin_memory()  # [1,320,1,512,512] fp32, 335.5 MB (> 126 MB L2)
    x_dev = x_host.to(dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = t.item()
        return ms

    def timed(fn, steps, hook=None, clocks=False, warmup=None):
        """W warm-up calls, then EXACTLY `steps` calls bracketed by barrier + synchronize on both sides, CUDA events on the
        launching stream, max over ranks.  Returns (ms, wall_ms, launches, clock summary or None)."""
        cs_cm = ClockSampler(local_rank) if clocks else contextlib.nullcontext()
        with cs_cm as cs:  # the sampler starts before the warm-up (same load) so that samples exist when the timed region begins
            for _ in range(args.warmup if warmup is None else warmup):
                fn()
            gc.collect()
            gc.disable()  # a collection in the middle of the timed region stalls the launching thread for tens of ms
            barrier()
            _lib.launch_count = 0
            _lib.event_hook = hook
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.perf_counter()
            e0.record()
            for _ in range(steps):
                fn()
            e1.record()
            barrier()
            wall = (time.perf_counter() - t0) * 1e3
            _lib.event_hook = None
            gc.enable()
            if clocks:
                time.sleep(0.15)
        return max_over_ranks(e0.elapsed_time(e1)), max_over_ranks(wall), _lib.launch_count, (cs.summary() if clocks else None)

    # =====================================================================================================================
    # (1) HEADLINE: MIM pre-training step, inputs resident in HBM (fp32 volume + index lists of the mask)
    # =====================================================================================================================
    np.random.seed(rank)
    mask = torch.from_numpy(OracleMaskGenerator(512, 320, 32, 16, 0.65)()).unsqueeze(0)
    n_mask = int(mask.sum())
    vol_dev = model.videomae._volume(x_dev)
    mp = _prep_mask(mask, dev, n_mask)
    model.train()
    opt = FusedAdamW(model, lr=5e-5, weight_decay=0.01, max_grad_norm=1.0)  # scripts/training/run_mim.sh:17-21
    use_graph = not args.no_cuda_graph
    # the product step: forward + backward (+ all-reduce) replayed from a CUDA graph, clip + AdamW launched behind it (DataParallelStep docstring)
    dp = DataParallelStep(model, optimizer=opt, cuda_graph=use_graph)
    # the same step launch by launch: the pass in which single kernels can be bracketed by CUDA events (roofline) and launches counted
    dp_eager = DataParallelStep(model, optimizer=opt) if use_graph else dp
    steps = args.steps
    dump = {} if args.dump_outputs and rank == 0 else None  # name -> host array, written by write_dump at the end

    # CUDA events around the dominant kernel (attention backward, 16 calls per step): the library records them on the launching
    # stream right before / after the main kernel (smbv_flash_attn_bwd_fused: the fused one-pass kernel + its combine pass;
    # SMBV_ATTN_BWD_DETERMINISTIC=1 -> smbv_flash_attn_bwd_ex: the dK/dV kernel, with dQ beside it on a forked stream)
    n_ev = 16 * steps
    ev_pool = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n_ev)]
    for a, b in ev_pool:
        a.record(), b.record()  # creates the cudaEvent_t handles
    torch.cuda.synchronize()
    ev_used, ev_shapes = [], []

    call_events = []

    @contextlib.contextmanager
    def bwd_hook(name):  # installed only inside the timed region; also the marker the event source below looks for
        if name in ("smbv_flash_attn_bwd_ex", "smbv_flash_attn_bwd_fused"):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            yield
            b.record()
            call_events.append((a, b))
        else:
            yield

    def ev_source():
        if _lib.event_hook is not bwd_hook or len(ev_used) >= n_ev:
            return (None, None)
        a, b = ev_pool[len(ev_used)]
        ev_used.append((a, b))
        return (a.cuda_event, b.cuda_event)

    _orig_bwd = ops.flash_attn_bwd

    def bwd_spy(q, *a, **k):  # remembers (H, N) of every timed attention-backward call
        if _lib.event_hook is bwd_hook:
            ev_shapes.append((q.shape[-3], q.shape[-2]))
        return _orig_bwd(q, *a, **k)

    ops.flash_attn_bwd = bwd_spy
    ops.attn_bwd_event_source = ev_source
    losses = []
    mim_out = []  # (loss, logits) of the latest MIM step

    def mim_step(d):
        mim_out.clear()  # the last step's outputs are freed before this step allocates its own
        mim_out.extend(d.step(vol_dev, mp))
        losses.append(mim_out[0].clone())

    # the event pass runs with the second-stream queue OFF (training.SideQueue, SMBV_WGRAD_STREAM=0): with it the weight-gradient GEMMs of
    # the previous layer share the SMs with the bracketed attention backward and its CUDA-event duration is no longer the kernel's own
    _side_prev = os.environ.get("SMBV_WGRAD_STREAM")
    os.environ["SMBV_WGRAD_STREAM"] = "0"
    ms_single, _, launches, _ = timed(lambda: mim_step(dp_eager), steps, hook=bwd_hook, clocks=False)
    if _side_prev is None:
        os.environ.pop("SMBV_WGRAD_STREAM")
    else:
        os.environ["SMBV_WGRAD_STREAM"] = _side_prev
    ops.attn_bwd_event_source = None
    ops.flash_attn_bwd = _orig_bwd
    torch.cuda.synchronize()
    # the product's eager step (second stream on): launch by launch, no per-kernel events
    ms_eager, wall_eager, _, clocks_eager = timed(lambda: mim_step(dp_eager), steps, clocks=True)
    if use_graph:  # HEADLINE: the graph replay (the inputs are resident: vol_dev / mp are copied into the static buffers device to device)
        ms_mim, wall_mim, _, clocks = timed(lambda: mim_step(dp), steps, clocks=True)
    else:
        ms_mim, wall_mim, clocks = ms_eager, wall_eager, clocks_eager
    if dump is not None:  # now: the steps of (1b) overwrite the graph's static loss / logits
        dump["mim_loss"] = host(mim_out[0])
        dump["mim_logits"] = sample_rows(mim_out[1], 1024)  # [13312 masked tokens, 4096] bf16 -> 1024 rows, 16 MB
    dk_ms = [a.elapsed_time(b) for a, b in ev_used]  # dK/dV kernel alone (library-recorded events); dQ runs beside it, so it is NOT an isolated time
    call_ms = [a.elapsed_time(b) for a, b in call_events]  # the whole call: prep + dK/dV || dQ + join
    call_fl = [8.0 * N * N * 64 * H for H, N in ev_shapes[:len(call_ms)]]
    dk_total_ms, dk_total_fl = sum(call_ms), sum(call_fl)
    ach = dk_total_fl / (dk_total_ms / 1e3) / 1e12 if dk_total_ms > 0 else 0.0
    by_shape, dk_by_shape = {}, {}
    for (H, N), t in zip(ev_shapes, call_ms):
        by_shape.setdefault(f"H{H}_N{N}", []).append(t)
    for (H, N), t in zip(ev_shapes, dk_ms):
        dk_by_shape.setdefault(f"H{H}_N{N}", []).append(t)
    vps = world * steps / (ms_mim / 1e3)
    fused_bwd = not ops.ATTN_BWD_DETERMINISTIC
    traffic, traffic_src = ncu_traffic("flash_attn_bwd_fused_kernel" if fused_bwd else "flash_attn_bwd_dkdv_kernel")

    # (1b) the same step END TO END from HOST data through the public API, every step: raw int16 CT volume (pinned host, 167.8 MB)
    #      -> H2D (side stream, double-buffered, overlaps the previous step) -> VolumePreprocessor (scale / pad / crop / permute
    #      kernel) -> MaskGenerator.device_batch (fresh mask from the reference RNG stream, index lists on the GPU) ->
    #      DataParallelStep.step -> the loss is read back on the host (one step behind, so the CPU can run ahead)
    gen = torch.Generator().manual_seed(11 + rank)
    raw_hosts = [torch.randint(-1100, 1500, (512, 512, 320), generator=gen, dtype=torch.int16).pin_memory() for _ in range(2)]
    raw_dev = [torch.empty((512, 512, 320), dtype=torch.int16, device=dev) for _ in range(2)]
    prep, mgen = VolumePreprocessor(512, 320, device=dev), MaskGenerator(512, 320, 32, 16, 0.65)
    s_in = torch.cuda.Stream(dev)
    ev_in, ev_free = [torch.cuda.Event() for _ in range(2)], [torch.cuda.Event() for _ in range(2)]
    loss_host = torch.zeros(2, dtype=torch.float32).pin_memory()
    ev_loss = [torch.cuda.Event() for _ in range(2)]
    seen = []

    def h2d(i):
        k = i & 1
        with torch.cuda.stream(s_in):
            s_in.wait_event(ev_free[k])
            raw_dev[k].copy_(raw_hosts[k], non_blocking=True)
            ev_in[k].record(s_in)

    vol_static = dp.static_inputs(vol_dev, mp)[0] if use_graph else None  # the preprocessing kernel writes the graph's input in place

    def e2e_train(n):
        cur = torch.cuda.current_stream(dev)
        h2d(0)
        for i in range(n):
            k = i & 1
            if i + 1 < n:
                h2d(i + 1)  # next volume's copy runs under this step's compute
            cur.wait_event(ev_in[k])
            vol = (prep(raw_dev[k], out=vol_static) if use_graph else prep(raw_dev[k])).view(1, 320, 512, 512)
            if use_graph:
                vol = vol_static
            ev_free[k].record(cur)
            loss, _ = dp.step(vol, mgen.device_batch(1, dev))
            loss_host[k:k + 1].copy_(loss.reshape(1), non_blocking=True)
            ev_loss[k].record(cur)
            if i > 0:
                ev_loss[k ^ 1].synchronize()
                seen.append(float(loss_host[k ^ 1]))
        ev_loss[(n - 1) & 1].synchronize()
        seen.append(float(loss_host[(n - 1) & 1]))

    e2e_train(args.warmup)
    ms_te, wall_te, _, _ = timed(lambda: e2e_train(steps), 1, warmup=0)

    line = {
        "metric": METRIC, "value": vps, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": args.warmup,
        "ms_per_step": ms_mim / steps, "wall_ms_per_step": wall_mim / steps, "eager_ms_per_step": ms_eager / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic",
        "config": {"workload": WORKLOAD,
                   "parallelism": f"dp{world}: one process per GPU, bucketed bf16 gradient all-reduce (NCCL) overlapped with backward" if world > 1 else "dp1 (no collective at N=1)",
                   "l2": "inputs larger than L2 (335.5 MB volume; 6.5 GB of saved activations streamed per step)",
                   "tflops_per_volume": TRAIN_FLOPS / 1e12, "optimizer_in_step": True,
                   "launch_mode": ("forward + backward (+ all-reduce) captured once in a CUDA graph and replayed every step (DataParallelStep(cuda_graph=True)); clip + AdamW launched behind it; "
                                   "eager_ms_per_step = the same step launch by launch") if use_graph else "eager (one launch per kernel)"},
        "model_tflops": TRAIN_FLOPS * vps / world / 1e12,
        "model_frac_of_sustained_peak": TRAIN_FLOPS * vps / world / 1e12 / pk["tf_sust"],
        "e2e": {"value": world * steps / (ms_te / 1e3), "unit": UNIT, "ms_per_step": ms_te / steps, "wall_ms_per_step": wall_te / steps,
                "h2d_bytes_per_step": raw_hosts[0].numel() * 2 + 2560, "d2h_bytes_per_step": 4,
                "api": "VolumePreprocessor + MaskGenerator.device_batch + DataParallelStep.step(FusedAdamW): raw int16 volume from pinned "
                       "host memory each step, fresh mask each step, loss read back on the host",
                "loss_last": seen[-1]},
        "gpu_launches": launches,
        "clocks": clocks,
        "roofline": {"kernel": ("attention backward = ONE smbv_flash_attn_bwd_fused call (D = rowsum(dO.O) prep + flash_attn_bwd_fused_kernel + combine of "
                                "the split last wave + fp32 -> bf16 dQ finishing pass, all timed together; 12 calls at H=12,N=7168 + 4 at H=6,N=20480 per step)")
                               if fused_bwd else
                               ("attention backward = flash_attn_bwd_dkdv_kernel || flash_attn_bwd_dq_kernel (ONE smbv_flash_attn_bwd call: the two kernels run "
                                "concurrently on the caller's and a forked stream, so they are timed together; 12 calls at H=12,N=7168 + 4 at H=6,N=20480 per step)"),
                     "bound": "tensor", "achieved": ach, "peak": pk["tf_sust"], "unit": "TFLOP/s", "frac": ach / pk["tf_sust"],
                     "traffic": traffic, "traffic_source": traffic_src + ("" if fused_bwd else " (dK/dV kernel; the dQ kernel is the next entry of that file)"),
                     "algorithmic": "8*N^2*64*H flops per call (dP, dV, dK, dQ: the four products of the reference's stored-P backward; the S = QK^T recomputation every flash backward needs is not counted), summed over the timed calls / summed CUDA-event durations",
                     "peak_source": pk["src"] + ", sustained bf16 (kernels timed inside a long step)",
                     "achieved_counting_score_recompute": ach * 1.25,  # 10*N^2*64*H (S = QK^T recomputed once, as every flash backward must): the convention of the flash-attention papers
                     "launch_ms_mean": dk_total_ms / max(len(call_ms), 1), "launches_timed": len(call_ms),
                     "launch_ms_by_shape": {k: sum(v) / len(v) for k, v in by_shape.items()},
                     ("fused_kernel_ms_by_shape" if fused_bwd else "dkdv_kernel_ms_by_shape_with_dq_beside_it"): {k: sum(v) / len(v) for k, v in dk_by_shape.items()},
                     "share_of_step": dk_total_ms / ms_single if ms_single > 0 else None,
                     "single_stream_eager_ms_per_step": ms_single / steps,
                     "timed_in": "an eager pass of the same step on ONE stream (launch by launch, SMBV_WGRAD_STREAM=0 so that no weight-gradient kernel shares the SMs with the bracketed kernel; CUDA events around every attention-backward call; share_of_step is relative to that pass); the headline step replays the same kernels from a CUDA graph with the weight / bias gradients on a second stream"},
        "loss_first": float(losses[0]), "loss_last": float(losses[-1]), "peak_mem_gb": torch.cuda.max_memory_allocated() / 2**30,
    }

    # (1c) N > 1: the same step with the all-reduce switched off (independent replicas), same box, same process — the raw
    #      number the cost of the collective can be read from (bench.py reports no efficiency)
    if world > 1:
        dp_solo = DataParallelStep(model, optimizer=opt, process_group=False, cuda_graph=use_graph)
        ms_solo, _, _, _ = timed(lambda: dp_solo.step(vol_dev, mp), steps)
        line["no_collective"] = {"value": world * steps / (ms_solo / 1e3), "unit": UNIT, "ms_per_step": ms_solo / steps,
                                 "what": "identical step with the gradient all-reduce disabled (independent replicas)"}
        del dp_solo

    # =====================================================================================================================
    # (2) embedding inference (BASELINE configs[1]); same model object, eval mode
    # =====================================================================================================================
    model.eval()
    if not args.no_inference:
        attn_events = []

        @contextlib.contextmanager
        def fwd_hook(name):
            if name == "smbv_flash_attn_fwd_ex":
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                yield
                e1.record()
                attn_events.append((e0, e1))
            else:
                yield

        inf_out = []

        def infer():
            with torch.no_grad():  # the reference's inference loop (src/run_inference.py:78-86); with grad enabled the forward would keep activations
                inf_out.clear()
                inf_out.append(model.videomae(x_dev).last_hidden_state)

        ms_dev, wall_dev, il, _ = timed(infer, steps, hook=fwd_hook)
        if dump is not None:
            dump["inference_last_hidden_state"] = sample_rows(inf_out[0], 4096)  # [20480, 768] -> 4096 rows, 12 MB
        inf_out.clear()
        attn_ms = [a.elapsed_time(b) for a, b in attn_events]
        attn_avg = sum(attn_ms) / max(len(attn_ms), 1)
        from smb_vision_b200.inference import EmbeddingRunner

        runner = EmbeddingRunner(model)
        x_hosts = [x_host, x_host.clone().pin_memory()]

        def e2e_run(n, r, srcs):
            tot = 0.0
            for emb in r.embed_stream(srcs[i & 1] for i in range(n)):
                tot += float(emb[0, 0, 0])  # touch the host result
            return tot

        e2e_run(args.warmup, runner, x_hosts)
        ms_e2e, wall_e2e, _, _ = timed(lambda: e2e_run(steps, runner, x_hosts), 1, warmup=0)
        gen_r = torch.Generator().manual_seed(23 + rank)
        raw_inf = [torch.randint(-1100, 1500, (512, 512, 320), generator=gen_r, dtype=torch.int16).pin_memory() for _ in range(2)]
        runner_raw = EmbeddingRunner(model, preprocess=VolumePreprocessor(512, 320, device=dev))
        e2e_run(args.warmup, runner_raw, raw_inf)
        ms_raw, wall_raw, _, _ = timed(lambda: e2e_run(steps, runner_raw, raw_inf), 1, warmup=0)
        del runner, runner_raw
        ach_f = ATTN_FWD_FLOPS / (attn_avg / 1e3) / 1e12 if attn_avg > 0 else 0.0
        tr_f, tr_f_src = ncu_traffic("flash_attn_fwd2_kernel")
        ivps = world * steps / (ms_dev / 1e3)
        line["inference"] = {
            "workload": INFER_WORKLOAD, "value": ivps, "unit": UNIT, "ms_per_step": ms_dev / steps, "wall_ms_per_step": wall_dev / steps,
            "parallelism": f"volume-sharded x{world}, no collective", "gpu_launches": il,
            "model_tflops": EMBED_FLOPS * ivps / world / 1e12, "model_frac_of_sustained_peak": EMBED_FLOPS * ivps / world / 1e12 / pk["tf_sust"],
            "e2e": {"value": world * steps / (ms_e2e / 1e3), "unit": UNIT, "ms_per_step": ms_e2e / steps, "wall_ms_per_step": wall_e2e / steps,
                    "h2d_bytes_per_step": x_host.numel() * 4, "d2h_bytes_per_step": N_TOK * D * 4,
                    "api": "smb_vision_b200.inference.EmbeddingRunner.embed_stream (pinned host fp32 volume in, pinned host fp32 embedding out, copies overlapped with compute)"},
            "e2e_raw_int16": {"value": world * steps / (ms_raw / 1e3), "unit": UNIT, "ms_per_step": ms_raw / steps, "wall_ms_per_step": wall_raw / steps,
                              "h2d_bytes_per_step": raw_inf[0].numel() * 2, "d2h_bytes_per_step": N_TOK * D * 4,
                              "api": "EmbeddingRunner(model, preprocess=VolumePreprocessor(512, 320)).embed_stream: raw int16 HU volume in, fp32 embedding out"},
            "roofline": {"kernel": "flash_attn_fwd2_kernel (H=12, N=20480, d=64)", "bound": "tensor", "achieved": ach_f, "peak": pk["tf_sust"],
                         "unit": "TFLOP/s", "frac": ach_f / pk["tf_sust"], "traffic": tr_f, "traffic_source": tr_f_src,
                         "algorithmic": "4*N^2*64*H = 1.2885 TFLOP per launch; Q,K,V,O bytes = 125.8 MB",
                         "peak_source": pk["src"] + ", sustained bf16", "launch_ms": attn_avg, "launches_timed": len(attn_ms),
                         "share_of_step": attn_avg * LAYERS / (ms_dev / steps)},
        }

    # =====================================================================================================================
    # (3) BASELINE configs[3]: classification fine-tune step, 224x224x160 (1960 tokens), batch 4 per GPU, age / sex features, DP
    # =====================================================================================================================
    if not args.no_cls:
        try:
            line["classification"] = bench_classification(timed, dev, world, rank, steps, pk, use_graph, dump)
        except Exception as e:  # a secondary block must not take the headline down
            line["classification"] = {"error": f"{type(e).__name__}: {e}"}
    # (4) BASELINE configs[4]: V-JEPA2-3D training step + the encoder forward at 512x512x320
    if not args.no_vjepa:
        try:
            line.update(bench_vjepa(timed, dev, world, rank, steps, pk, x_dev, use_graph, dump))
        except Exception as e:
            line["vjepa_step"] = {"error": f"{type(e).__name__}: {e}"}

    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        torch.cuda.empty_cache()
        line["cpu_baseline"] = cpu_baseline_mim()
    if dump is not None:
        write_dump(args.dump_outputs, dump)
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        # Teardown: the CUDA graphs hold captured NCCL all-reduces; destroying the communicator (or the interpreter's own teardown)
        # with them alive hung for minutes at N=2.  Release the graphs, rendezvous, and leave without the NCCL destructor path.
        for o in (dp, dp_eager):
            getattr(o, "_graphs", {}).clear()
        gc.collect()
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush(), sys.stderr.flush()
        os._exit(0)


def bench_classification(timed, dev, world, rank, steps, pk, use_graph=True, dump=None):
    """src/run_classification.py:452-504 / scripts/training/run_cls.sh: smb-vision-base encoder, 224x224x160 = 1960 tokens, batch 4 per
    GPU, 2 additional features, 2 labels; forward + cross-entropy + backward + all-reduce + clip + AdamW."""
    import torch
    from transformers import VideoMAEConfig

    from smb_vision_b200.modeling import B200VideoMAEForVideoClassification
    from smb_vision_b200.optim import FusedAdamW
    from smb_vision_b200.training import DataParallelStep

    c = VideoMAEConfig()
    c.update(dict(image_size=224, patch_size=16, num_channels=1, num_frames=160, tubelet_size=16, num_labels=2, additional_features_size=2,
                  problem_type="single_label_classification"))
    torch.manual_seed(0)
    model = B200VideoMAEForVideoClassification(c).to(dev).train()
    B = 4
    g = torch.Generator().manual_seed(40 + rank)
    x = torch.rand(B, 160, 1, 224, 224, generator=g).to(dev)
    feats = torch.randn(B, 2, generator=g).to(dev)
    labels = torch.tensor([0, 1, 1, 0]).to(dev)
    opt = FusedAdamW(model, lr=5e-5, weight_decay=0.01, max_grad_norm=1.0)
    vol = model.videomae._volume(x)
    losses, last = [], []

    def step(d):
        last.clear()
        last.extend(d.step(vol, feats, labels))
        losses.append(last[0].clone())

    dp_eager = DataParallelStep(model, optimizer=opt)
    ms_eager, _, launches, _ = timed(lambda: step(dp_eager), steps)
    ms = ms_eager
    if use_graph:  # 1975 launches of mostly 5-10 us kernels: the eager step is launch-bound, the graph replay is the product path
        dp = DataParallelStep(model, optimizer=opt, cuda_graph=True)
        ms, _, _, _ = timed(lambda: step(dp), steps)
    if dump is not None:
        dump["cls_loss"], dump["cls_logits"] = host(last[0]), host(last[1])
    N, d, L, mlp = 1960, 768, 12, 3072
    flops = 3 * B * (2 * N * 4096 * d + L * (2 * N * d * (3 * d + d + 2 * mlp) + 4 * N * N * 64 * 12))
    vps = world * B * steps / (ms / 1e3)
    return {"workload": "smb-vision-base classification fine-tune step (BASELINE configs[3]): 224x224x160 = 1960 tokens, batch 4 per GPU, 2 additional "
                        "features, cross-entropy; forward + backward + gradient all-reduce + clip + AdamW, inputs resident in HBM",
            "value": vps, "unit": UNIT, "ms_per_step": ms / steps, "eager_ms_per_step": ms_eager / steps, "cuda_graph": bool(use_graph), "batch_per_gpu": B, "gpu_launches": launches,
            "model_tflops_per_gpu": flops * steps / (ms / 1e3) / 1e12, "frac_of_sustained_peak": flops * steps / (ms / 1e3) / 1e12 / pk["tf_sust"],
            "loss_first": float(losses[0]), "loss_last": float(losses[-1]), "losses": [round(float(v), 5) for v in losses[:12]]}


def bench_vjepa(timed, dev, world, rank, steps, pk, x_dev, use_graph=True, dump=None):
    """src/run_vjepa.py:101-141 at the reference's own input size (384x384x256 = 9216 tokens, ViT-L 1024/16/24 + predictor 384/12/12,
    src/run_vjepa.py:73-84, facebook/vjepa2-vitl-fpc64-256), batch 1 per GPU: online forward (encoder on context tokens + predictor),
    momentum-target encoder forward, L1, backward, all-reduce, clip + AdamW, EMA update.  Plus the ViT-L encoder forward alone at 512x512x320."""
    import torch
    from transformers import VJEPA2Config

    from examples.train_vjepa import vjepa_step
    import smb_vision_b200.attention_interface as ai
    from smb_vision_b200.data import VJEPAMaskGenerator, vjepa_collate_fn
    from smb_vision_b200.optim import EmaTarget, FusedAdamW
    from smb_vision_b200.vjepa import B200VJEPA2Model

    out = {}
    ai.register()
    T, S = 256, 384
    vc = VJEPA2Config(patch_size=16, crop_size=S, frames_per_clip=T, tubelet_size=16, in_chans=1)
    vc._attn_implementation = ai.NAME
    torch.manual_seed(1)
    model = B200VJEPA2Model(vc).to(dev).train()
    opt = FusedAdamW(model, lr=3e-5, weight_decay=0.01, max_grad_norm=1.0)  # scripts/training/run_vjepa.sh
    grads = opt.grad_arena()
    target = EmaTarget(model, momentum=0.99925)
    torch.manual_seed(100 + rank)
    g = torch.Generator().manual_seed(1 + rank)
    masks = VJEPAMaskGenerator(input_size=(T, S, S), patch_size=(16, 16, 16), num_blocks=3)
    batch = vjepa_collate_fn([masks({"image": torch.rand(T, 1, S, S, generator=g)})])
    x = batch["pixel_values_videos"].to(dev)
    ctx, tgt = [m.to(dev) for m in batch["context_mask"]], [m.to(dev) for m in batch["target_mask"]]
    losses = []
    ms_eager, _, launches, _ = timed(lambda: losses.append(vjepa_step(model, target, opt, grads, x, ctx, tgt).clone()), steps, warmup=2)
    ms, graph_note = ms_eager, "eager"
    if use_graph:
        try:  # forward + backward replayed from a CUDA graph (examples/train_vjepa.GraphedVJEPAStep); optimiser + EMA behind it
            from examples.train_vjepa import GraphedVJEPAStep

            gstep = GraphedVJEPAStep(model, target, opt, grads)
            ms, _, _, _ = timed(lambda: losses.append(gstep(x, ctx, tgt).clone()), steps, warmup=2)
            graph_note = "CUDA graph of forward + backward, optimiser + EMA launched behind it"
            gstep._graphs.clear()
        except Exception as e:
            ms, graph_note = ms_eager, f"eager (graph capture failed: {type(e).__name__}: {str(e)[:200]})"
    out["vjepa_step"] = {
        "workload": "V-JEPA2-3D training step (BASELINE configs[4]): ViT-L encoder (1024/16/24) + predictor (384/12/12), 384x384x256 = 9216 tokens "
                    "(the reference's own input size), batch 1 per GPU: online forward on the context tokens + predictor, momentum-target forward, L1, backward, "
                    "gradient all-reduce, clip + AdamW, EMA update",
        "value": world * steps / (ms / 1e3), "unit": UNIT, "ms_per_step": ms / steps, "eager_ms_per_step": ms_eager / steps, "launch_mode": graph_note,
        "gpu_launches_ours": launches,
        "context_tokens": int(ctx[0].shape[1]), "target_tokens": int(tgt[0].shape[1]),
        "native": "everything: encoder forward + backward (online and momentum target), predictor forward + backward (context gather, position-sort index "
                  "kernel, rotary with sorted ids, head_dim 32 zero-padded onto the tcgen05 attention kernels, LayerNorm, projection), L1, clip + AdamW, EMA",
        "loss_first": float(losses[0]), "loss_last": float(losses[-1])}
    gstep = None
    del model, opt, grads, target
    torch.cuda.empty_cache()
    vc2 = VJEPA2Config(patch_size=16, crop_size=512, frames_per_clip=320, tubelet_size=16, in_chans=1)  # src/run_vjepa.py:220-232
    torch.manual_seed(1)
    with torch.device(dev):
        vmodel = B200VJEPA2Model(vc2, with_predictor=False).eval()
    vj_out = []

    def vj_infer():
        with torch.no_grad():
            vj_out.clear()
            vj_out.append(vmodel.get_vision_features(x_dev))

    ms_vj, _, n_launch, _ = timed(vj_infer, steps, warmup=2)
    if dump is not None:
        dump["vjepa_loss"] = host(losses[-1])
        dump["vjepa_encoder_features"] = sample_rows(vj_out[0], 4096)  # [20480, 1024] -> 4096 rows, 16 MB
    VJ_FLOPS = 2 * 20480 * 4096 * 1024 + 24 * (2 * 20480 * 1024 * 12 * 1024 + 4 * 20480 * 20480 * 1024)
    out["vjepa_encoder"] = {"workload": "V-JEPA2-3D ViT-L (1024/16 heads/24 layers) encoder forward, 512x512x320 = 20480 tokens, batch 1/GPU, bf16, random init",
                            "value": world * steps / (ms_vj / 1e3), "unit": UNIT, "ms_per_volume": ms_vj / steps, "gpu_launches": n_launch,
                            "model_tflops_per_gpu": VJ_FLOPS * steps / (ms_vj / 1e3) / 1e12,
                            "frac_of_sustained_peak": VJ_FLOPS * steps / (ms_vj / 1e3) / 1e12 / pk["tf_sust"]}
    return out


if __name__ == "__main__":
    main()
