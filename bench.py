#!/usr/bin/env python
"""bench.py -- images/sec of the ViT-B/16 224^2 forward path (BASELINE.json metric) on N B200s of one node.

    python bench.py --gpus 1 --steps 10 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
           bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # the reference's own ggml CPU path (oracle/_ref) on the host cores

A "step" is one forward pass (pixels f32 HWC -> probabilities + top-5) over one batch of 256 synthetic images per
GPU (BASELINE.json configs[1]: vit_base_patch16_224 f16, batch=256, 1xB200).  Images shard across ranks, weights are
replicated, there is no collective on the data path (SURVEY.md 8e) => "scaling": "weak".

`value`     : whole-job images/s with inputs already resident in HBM (CUDA events on the launching stream, max over ranks),
              exactly K timed steps after W >= 3 warm-up steps.
`e2e`       : same metric through the reference-facing C-ABI call with HOST (pinned) buffers: H2D of the 154 MB batch and
              D2H of probabilities + top-5 inside the timed region.
`sustained` : the same step repeated back to back for >= 2 s (the K-step burst runs at boost clocks; under the 1 kW power cap the
              SM clock settles lower), with the clocks sampled over that window.
`roofline`  : tensor-core roofline of the dominant kernel (an fc1 / fc2 / qkv tcgen05 GEMM), timed live with a CUDA-event pair
              around each of its launches in a profiled pass that runs right after the sustained window (hot GPU); the fraction is
              given against BOTH measured cuBLAS peaks of MEASURED_PEAKS.json (sustained = `frac`, burst = `frac_burst`).
`parity`    : the engine's logits for the 64 seeded fixture images of tests/golden/base_f16_b64.npz (generated from the unmodified
              reference) -- per-image max|dlogit| / max|ref logit| distribution next to the CPU noise floor stored with the fixture,
              and how many of the 64 top-5 index lists are identical.
`configs`   : the other single-GPU configurations of BASELINE.json (ViT-L/16-384 bf16 weights batch 128; ViT-B/16 q8_0 file batch
              256), each with its own images/s, dominant-kernel roofline and parity sample; they run after the headline so `value`
              is not affected.  (N = 1 only.)
`cpu_baseline`: the reference (oracle/_ref, unmodified ggml CPU path) timed on this box's host cores, bounded sample.
"""
import argparse
import ctypes as C
import json
import math
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

BATCH = 256
MODEL_CFG = "base"
# algorithmic FLOPs per image (2 x MACs of patch embed + L x (qkv + QK^T + PV + proj + fc1 + fc2) + head), SURVEY.md 8(d)
FLOPS_PER_IMAGE = {"base": 35.128e9, "large384": 382.133e9, "tiny": 2.507e9}
KERNEL_NAMES = ["patch", "qkv", "proj", "fc1", "fc2", "head", "attention", "layernorm"]


def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of each GEMM of the step, from the committed
    `ncu --set full` capture (profiles/traffic.json, written by tools/summarize_ncu.py); None when no capture exists."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    return json.load(open(p)) if os.path.exists(p) else {}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        burst = float(d.get("bf16_tflops", 1590.0))
        return {"tflops_sustained": float(d.get("bf16_tflops_sustained", burst)), "tflops_burst": burst, "hbm_gbs": float(d.get("hbm_gbs", 6650.0)),
                "sustained_clock_mhz": (d.get("clocks_under_load") or {}).get("sm_mhz_median"), "which": "measured (MEASURED_PEAKS.json)"}
    return {"tflops_sustained": 1400.0, "tflops_burst": 1590.0, "hbm_gbs": 6650.0, "sustained_clock_mhz": 1300.0,
            "which": "fallback (B200_PROFILING.md: 1.59 PFLOP/s burst, ~1.4 sustained, 6.65 TB/s)"}


class ClockSampler(threading.Thread):
    """Samples SM clock + throttle reasons of one GPU through NVML while the timed region runs."""
    REASONS = {0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x10: "sync_boost",
               0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown", 0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.sm, self.reasons, self.max_mhz = index, False, [], set(), None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        while not self.stop_flag and self.nv is not None:
            try:
                self.sm.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                r = self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in self.REASONS.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.02)

    def result(self):
        self.stop_flag = True
        if self.nv is None or not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["nvml_unavailable"]}
        return {"sm_mhz": float(np.median(self.sm)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.sm)}


def host_cpu_info():
    """CPU model string, logical / physical core counts and SMT state of the host (BASELINE.md 4.3 asks for them next to the CPU number)."""
    info = {"model": None, "logical_cpus": os.cpu_count(), "physical_cores": None, "smt": None}
    try:
        cores = set()
        phys = core = None
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name") and info["model"] is None:
                info["model"] = line.split(":", 1)[1].strip()
            elif line.startswith("physical id"):
                phys = line.split(":", 1)[1].strip()
            elif line.startswith("core id"):
                core = line.split(":", 1)[1].strip()
            elif not line.strip():
                if phys is not None and core is not None:
                    cores.add((phys, core))
                phys = core = None
        if cores:
            info["physical_cores"] = len(cores)
    except Exception:
        pass
    try:
        info["smt"] = open("/sys/devices/system/cpu/smt/active").read().strip() == "1"
    except Exception:
        if info["physical_cores"] and info["logical_cpus"]:
            info["smt"] = info["logical_cpus"] > info["physical_cores"]
    return info


def host_threads():
    n = os.cpu_count() or 8
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        pass
    return n


def thread_candidates():
    nproc = host_threads()
    top = min(nproc, 64)  # the reference's spin barriers stop scaling long before that (SURVEY.md section 6)
    return sorted({top, max(1, top // 2), max(1, top // 4), max(1, top // 8)}, reverse=True)


def cpu_reference_rate(n_images, threads_list):
    """images/s of the reference vit_predict (oracle/_ref, reference vit.cpp:1004) on host cores; model load excluded.
    Every candidate thread count is timed on the same n_images; the best one is reported."""
    from tests.util import gf, model_path
    from oracle import ref
    m = ref.RefModel(model_path(MODEL_CFG, "f16"))
    imgs = gf.synthetic_images(n_images, 224, seed=4321)
    m.predict(imgs[0], threads_list[0])  # warm (page in weights)
    best = None
    tried = {}
    for nt in threads_list:
        t = time.perf_counter()
        for i in range(n_images):
            m.predict(imgs[i], nt)
        dt = time.perf_counter() - t
        rate = n_images / dt
        tried[nt] = rate
        if best is None or rate > best[0]:
            best = (rate, nt, dt)
    m.close()
    return best + (tried,)


def run_reference_arm(args, rank, world):
    if rank != 0:
        return
    nproc = host_threads()
    cand = thread_candidates()
    per_step = 4
    # choose the better thread count on a probe of the same size as a step, then time exactly `steps` steps of `per_step` images
    rate, nt, _, tried = cpu_reference_rate(per_step, cand)
    from tests.util import gf, model_path
    from oracle import ref
    m = ref.RefModel(model_path(MODEL_CFG, "f16"))
    imgs = gf.synthetic_images(per_step, 224, seed=99)
    for _ in range(min(args.warmup, 1)):
        m.predict(imgs[0], nt)
    t = time.perf_counter()
    for _ in range(args.steps):
        for i in range(per_step):
            m.predict(imgs[i], nt)
    dt = time.perf_counter() - t
    val = args.steps * per_step / dt
    line = {"impl": "reference", "metric": "images/sec ViT-B/16 224^2 forward", "value": val, "unit": "images/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
            "config": {"workload": "vit_base_patch16_224 f16 legacy-ggml file, reference ggml CPU vit_predict, %d images per step (bounded sample of the batch-256 workload)" % per_step,
                       "threads": nt, "host_cores": nproc},
            "cpu_baseline": {"value": val, "unit": "images/s", "cores": nt, "kind": "reference",
                             "sample": "%d steps x %d images through oracle/_ref vit_predict" % (args.steps, per_step),
                             "threads_tried_images_per_s": {str(k): round(v, 2) for k, v in tried.items()}, "host": host_cpu_info()},
            "e2e": {"value": val, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def read_profile(L, model, steps, ms_profiled):
    prof = {}
    for kind, name in enumerate(KERNEL_NAMES):
        ms, cnt, fl = C.c_double(), C.c_int(), C.c_double()
        if L.vitb200_profile_read(model.handle, kind, C.byref(ms), C.byref(cnt), C.byref(fl)) == 0 and cnt.value > 0:
            prof[name] = {"ms_total": ms.value, "launches": cnt.value, "flops_per_launch": fl.value}
    return prof


def dominant_roofline(prof, ms_profiled, peaks, clocks, note):
    dom = max((k for k in prof if k in ("qkv", "proj", "fc1", "fc2")), key=lambda k: prof[k]["ms_total"], default=None)
    if not dom:
        return None
    d = prof[dom]
    avg_s = d["ms_total"] * 1e-3 / d["launches"]
    ach = d["flops_per_launch"] / avg_s / 1e12
    return {"bound": "tensor", "kernel": f"gemm_tcgen05_kernel ({dom})", "achieved": ach, "peak": peaks["tflops_sustained"], "unit": "TFLOP/s",
            "frac": ach / peaks["tflops_sustained"], "peak_burst": peaks["tflops_burst"], "frac_burst": ach / peaks["tflops_burst"],
            "sm_mhz_during": clocks.get("sm_mhz"), "peak_sustained_measured_at_mhz": peaks["sustained_clock_mhz"],
            "traffic": ncu_traffic().get(dom), "traffic_unit": "bytes per launch (ncu dram read+write)", "peak_source": peaks["which"],
            "avg_launch_ms": avg_s * 1e3, "share_of_step": d["ms_total"] / ms_profiled, "timed_in": note}


def kernel_table(prof, steps):
    return {k: {"ms_per_step": v["ms_total"] / steps, "launches_per_step": v["launches"] / steps,
                "tflops": (v["flops_per_launch"] * v["launches"] / (v["ms_total"] * 1e-3) / 1e12) if v["flops_per_launch"] else None}
            for k, v in prof.items()}


def parity_stats(logits, idx, g):
    """Per-image distribution of max|dlogit| / max|ref logit| against a golden fixture (+ its noise floor when stored)."""
    ref = g["logits"]
    re = np.abs(logits - ref).max(1) / np.abs(ref).max(1)
    order = np.argsort(-ref, 1)[:, :5]
    out = {"n_images": int(ref.shape[0]), "metric": "per image max|dlogit| / max|ref logit| vs the unmodified reference (golden fixture)",
           "median": float(np.median(re)), "p90": float(np.quantile(re, 0.9)), "max": float(re.max()), "images_above_1e-3": int((re > 1e-3).sum()),
           "top1_identical": int((order[:, 0] == idx[:, 0]).sum()), "top5_lists_identical": int((order == idx).all(1).sum())}
    if "floor" in g:
        fl = g["floor"]
        out["cpu_noise_floor"] = {"what": "restatement with double accumulation + reference rounding points vs the reference, same images",
                                  "median": float(np.median(fl)), "p90": float(np.quantile(fl, 0.9)), "max": float(fl.max())}
        out["median_over_floor_median"] = float(np.median(re) / np.median(fl))
    return out


def run_extra_config(eng, L, gf, torch, name, cfg, ftype, batch, steps, warmup, golden, peaks, local_rank, stream):
    """One more BASELINE.json single-GPU configuration: device-timed images/s, dominant-kernel roofline, parity sample."""
    from tests.util import model_path
    t_build = time.perf_counter()
    path = model_path(cfg, ftype)
    model = eng.vit_model_load(path, device=local_rank, max_batch=batch)
    t_build = time.perf_counter() - t_build
    S = model.img_size
    dev_imgs = [torch.from_numpy(gf.synthetic_images(batch, S, seed=4242 + j)).cuda() for j in range(2)]  # 2 x (batch x S x S x 3 x 4 B) > L2
    d_probs = torch.empty(batch, model.num_classes, device="cuda")
    d_idx = torch.empty(batch, 5, dtype=torch.int32, device="cuda")
    d_val = torch.empty(batch, 5, device="cuda")

    def step(i):
        rc = L.vitb200_forward_device(model.handle, dev_imgs[i & 1].data_ptr(), batch, d_probs.data_ptr(), None, d_idx.data_ptr(), d_val.data_ptr(), 5, stream)
        if rc != 0:
            raise RuntimeError(L.vitb200_last_error().decode())
    for i in range(warmup):
        step(i)
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        step(i)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    clocks = sampler.result()
    launches = model.last_launch_count()
    L.vitb200_profile_enable(model.handle, 1)
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p0.record()
    for i in range(steps):
        step(i)
    p1.record()
    torch.cuda.synchronize()
    ms_prof = p0.elapsed_time(p1)
    prof = read_profile(L, model, steps, ms_prof)
    L.vitb200_profile_enable(model.handle, 0)
    value = batch * steps / (ms * 1e-3)
    out = {"workload": name, "images_per_s": value, "ms_per_step": ms / steps, "steps": steps, "warmup": warmup, "batch": batch,
           "gpu_launches_per_step": launches, "clocks": clocks,
           "model_tflops": value * FLOPS_PER_IMAGE[cfg] / 1e12, "model_frac_of_peak_sustained": value * FLOPS_PER_IMAGE[cfg] / 1e12 / peaks["tflops_sustained"],
           "roofline": dominant_roofline(prof, ms_prof, peaks, clocks, "profiled pass of the same %d steps (CUDA-event pair around every tracked kernel)" % steps),
           "kernels": kernel_table(prof, steps), "model_file_build_s": round(t_build, 1)}
    if golden and os.path.exists(golden):
        g = np.load(golden)
        imgs = gf.synthetic_images(int(g["n_images"]), S, seed=int(g["image_seed"]))
        probs, idx, val, logits = eng.vit_predict(model, imgs, 5, want_logits=True)
        out["parity"] = parity_stats(logits, idx, g)
    model.close()
    del dev_imgs
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the extra BASELINE.json configurations (ViT-L/16-384, q8_0)")
    ap.add_argument("--sustained-seconds", type=float, default=2.0)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned (probabilities, top-5 indices and "
                    "values) as DIR/<name>.npy")
    args = ap.parse_args()

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from tests.util import pkg, gf, model_path

    eng = pkg.engine
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the vit.cpp_b200 forward path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    B = args.batch
    W = max(args.warmup, 3)
    L = eng.lib()

    # synthetic weights (legacy-ggml file through the product loader) + synthetic inputs, per rank
    if rank == 0:
        path = model_path(MODEL_CFG, "f16")
    if world > 1:
        dist.barrier()
    path = model_path(MODEL_CFG, "f16")
    model = eng.vit_model_load(path, device=local_rank, max_batch=B)
    # two distinct input batches (2 x 154 MB > 126 MB L2), alternated so no step finds its input in L2
    host_imgs = [torch.from_numpy(gf.synthetic_images(B, 224, seed=1234 + 17 * rank + j)).pin_memory() for j in range(2)]
    dev_imgs = [h.cuda(non_blocking=True) for h in host_imgs]
    d_probs = torch.empty(B, model.num_classes, device="cuda")
    d_idx = torch.empty(B, 5, dtype=torch.int32, device="cuda")
    d_val = torch.empty(B, 5, device="cuda")
    # a non-default torch stream: its handle is what the C ABI launches on (NULL would mean "engine's own stream"),
    # and torch.cuda.Event timings on it see exactly those launches
    tstream = torch.cuda.Stream()
    torch.cuda.set_stream(tstream)
    stream = tstream.cuda_stream
    assert stream != 0

    def step_device(i):
        rc = L.vitb200_forward_device(model.handle, dev_imgs[i & 1].data_ptr(), B, d_probs.data_ptr(), None, d_idx.data_ptr(),
                                      d_val.data_ptr(), 5, stream)
        if rc != 0:
            raise RuntimeError(L.vitb200_last_error().decode())

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- region A: resident-data throughput, exactly K timed steps of the product path (at batch 256 every kernel runs >= 80 us, so
    # the schedule is launched eagerly with programmatic dependent launch; CUDA-graph replay is used below 8192 tokens per batch)
    for i in range(W):
        step_device(i)
    sync_all()

    def timed_region(n_steps):
        sampler = ClockSampler(local_rank)
        sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n_steps):
            step_device(i)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), sampler.result()

    ms_local, clocks = timed_region(args.steps)
    # a run that saw a hardware / thermal slowdown is rejected and re-measured once (sw_power_cap is kept and reported)
    bad = {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    again = torch.tensor([1 if bad & set(clocks.get("reasons", [])) else 0], device="cuda", dtype=torch.int32)
    if world > 1:
        dist.all_reduce(again, op=dist.ReduceOp.MAX)  # every rank repeats if any rank was throttled (the barriers are collective)
    if int(again.item()):
        first = clocks
        sync_all()
        ms_local, clocks = timed_region(args.steps)
        clocks["remeasured_after"] = first.get("reasons", [])
    launches_per_step = model.last_launch_count()
    if args.dump_outputs:
        # the inputs are seeded, so two builds given the same arguments can be compared output for output
        os.makedirs(args.dump_outputs, exist_ok=True)
        suffix = "" if world == 1 else "_rank%d" % rank
        for name, arr in (("probs", d_probs), ("topk_idx", d_idx), ("topk_prob", d_val)):
            np.save(os.path.join(args.dump_outputs, name + suffix + ".npy"), arr.cpu().numpy().astype(np.float32))
    t = torch.tensor([ms_local], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    value = world * B * args.steps / (ms_total * 1e-3)

    # ---- region S: the same step back to back for >= sustained_seconds (clock under the power cap settles within ~1 s)
    n_sus = max(args.steps, int(math.ceil(args.sustained_seconds * 1e3 / (ms_local / args.steps))))
    sync_all()
    ms_sus, clocks_sus = timed_region(n_sus)
    t = torch.tensor([ms_sus], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    sustained_value = world * B * n_sus / (float(t.item()) * 1e-3)

    # ---- region B: K more steps right behind the sustained window (hot GPU) with CUDA-event pairs around every tracked kernel
    L.vitb200_profile_enable(model.handle, 1)
    sampler = ClockSampler(local_rank)
    sampler.start()
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p0.record()
    for i in range(args.steps):
        step_device(i)
    p1.record()
    torch.cuda.synchronize()
    clocks_prof = sampler.result()
    ms_profiled = p0.elapsed_time(p1)
    prof = read_profile(L, model, args.steps, ms_profiled)
    L.vitb200_profile_enable(model.handle, 0)

    # ---- end to end through the host-buffer C-ABI call (H2D + forward + D2H) ------------------------------
    # Every step copies its 154 MB input batch from pinned host memory and reads probabilities + top-5 back into pinned
    # host memory; vitb200_forward_async double-buffers so step i+1's H2D overlaps step i's kernels.
    h_probs = [torch.empty(B, model.num_classes).pin_memory() for _ in range(2)]
    h_idx = [torch.empty(B, 5, dtype=torch.int32).pin_memory() for _ in range(2)]
    h_val = [torch.empty(B, 5).pin_memory() for _ in range(2)]

    def step_e2e(i):
        j = i & 1
        rc = L.vitb200_forward_async(model.handle, host_imgs[j].data_ptr(), B, h_probs[j].data_ptr(), None, h_idx[j].data_ptr(),
                                     h_val[j].data_ptr(), 5)
        if rc != 0:
            raise RuntimeError(L.vitb200_last_error().decode())
    for i in range(2):
        step_e2e(i)
    L.vitb200_sync(model.handle)
    sync_all()
    t0 = time.perf_counter()
    for i in range(args.steps):
        step_e2e(i)
    L.vitb200_sync(model.handle)
    e2e_s = time.perf_counter() - t0
    t = torch.tensor([e2e_s], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = world * B * args.steps / float(t.item())
    top1_check = int(h_idx[0][0, 0])

    # ---- end to end from u8 images (what load_image_from_file hands to vit_image_preprocess, vit.h:91-96): 256 x 256 RGB u8 per image,
    # packed + copied (4x fewer PCIe bytes than the f32 batch), resized / normalised on the GPU straight into the f16 patch matrix
    rng = np.random.default_rng(77 + rank)
    u8_batches = [[rng.integers(0, 256, size=(256, 256, 3), dtype=np.uint8) for _ in range(B)] for _ in range(2)]
    u8_args = []
    for imgs_u8 in u8_batches:
        ptrs = (C.c_void_p * B)(*[a.ctypes.data for a in imgs_u8])
        nx = (C.c_int * B)(*[a.shape[1] for a in imgs_u8])
        ny = (C.c_int * B)(*[a.shape[0] for a in imgs_u8])
        u8_args.append((ptrs, nx, ny))

    def step_u8(i):
        j = i & 1
        ptrs, nx, ny = u8_args[j]
        rc = L.vitb200_forward_u8_async(model.handle, ptrs, nx, ny, B, 0, h_probs[j].data_ptr(), None, h_idx[j].data_ptr(), h_val[j].data_ptr(), 5)
        if rc != 0:
            raise RuntimeError(L.vitb200_last_error().decode())
    for i in range(2):
        step_u8(i)
    L.vitb200_sync(model.handle)
    sync_all()
    t0 = time.perf_counter()
    for i in range(args.steps):
        step_u8(i)
    L.vitb200_sync(model.handle)
    u8_s = time.perf_counter() - t0
    t = torch.tensor([u8_s], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_u8_value = world * B * args.steps / float(t.item())

    # optional tail of the north-star design: gather the top-k pairs on rank 0 over NCCL (not on the timed path)
    if world > 1:
        gathered = [torch.empty_like(d_idx) for _ in range(world)] if rank == 0 else None
        dist.gather(d_idx, gathered, dst=0)

    if rank == 0:
        peaks = measured_peaks()
        line = {
            "metric": "images/sec ViT-B/16 224^2 forward", "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps,
            "warmup": W, "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f16", "data": "synthetic",
            "config": {"workload": "vit_base_patch16_224 f16 (legacy-ggml model file), batch=%d per GPU, 224x224x3 f32 HWC synthetic images" % B,
                       "global_batch": B * world, "parallelism": "dp%d (images sharded, weights replicated, no collective on the data path)" % world,
                       "l2": "two alternating 154 MB input batches + >1 GB of activations per step exceed the 126 MB L2; no explicit flush",
                       "attention_operands": "split precision (hi + lo f16 pairs for q, k, v: the reference's f32-operand attention)" if os.environ.get("VITB200_ATTN_HILO", "1") != "0" else "f16 only (VITB200_ATTN_HILO=0)"},
            "e2e": {"value": e2e_value, "unit": "images/s", "h2d_bytes_per_step": B * 3 * 224 * 224 * 4,
                    "d2h_bytes_per_step": B * (model.num_classes * 4 + 5 * 4 + 5 * 4)},
            "e2e_u8": {"value": e2e_u8_value, "unit": "images/s", "h2d_bytes_per_step": B * 256 * 256 * 3 + B * 16,
                       "d2h_bytes_per_step": B * (model.num_classes * 4 + 5 * 4 + 5 * 4),
                       "what": "vitb200_forward_u8_async: 256x256 RGB u8 images from host memory -> pinned staging -> one H2D -> bicubic resize + normalise on the "
                               "GPU (reference vit_image_preprocess semantics) -> forward -> probabilities + top-5 back to pinned host memory"},
            "gpu_launches": launches_per_step * args.steps,
            "clocks": clocks,
            "sustained": {"value": sustained_value, "unit": "images/s", "steps": n_sus, "seconds": ms_sus * 1e-3, "ms_per_step": ms_sus / n_sus,
                          "clocks": clocks_sus, "model_tflops": sustained_value * FLOPS_PER_IMAGE[MODEL_CFG] / 1e12 / world,
                          "model_frac_of_peak_sustained": sustained_value * FLOPS_PER_IMAGE[MODEL_CFG] / 1e12 / world / peaks["tflops_sustained"]},
            "roofline": dominant_roofline(prof, ms_profiled, peaks, clocks_prof,
                                          "%d profiled steps launched right behind the %.1f s sustained window, a CUDA-event pair around every tracked kernel "
                                          "(%.3f ms/step profiled vs %.3f ms/step in the K-step burst that `value` reports, %.3f sustained)"
                                          % (args.steps, ms_sus * 1e-3, ms_profiled / args.steps, ms_local / args.steps, ms_sus / n_sus)),
            "model_tflops": value * FLOPS_PER_IMAGE[MODEL_CFG] / 1e12 / world,
            "model_frac_of_peak": value * FLOPS_PER_IMAGE[MODEL_CFG] / 1e12 / world / peaks["tflops_sustained"],
            "model_frac_of_peak_burst": value * FLOPS_PER_IMAGE[MODEL_CFG] / 1e12 / world / peaks["tflops_burst"],
            "kernels": kernel_table(prof, args.steps),
            "top1_sample": top1_check,
        }
        gold = os.path.join(ROOT, "tests", "golden", "base_f16_b64.npz")
        if os.path.exists(gold):
            g = np.load(gold)
            imgs = gf.synthetic_images(int(g["n_images"]), 224, seed=int(g["image_seed"]))
            probs, idx, val, logits = eng.vit_predict(model, imgs, 5, want_logits=True)
            line["parity"] = parity_stats(logits, idx, g)
        model.close()
        model = None
        del dev_imgs, host_imgs
        torch.cuda.empty_cache()
        if world == 1 and not args.no_configs:
            gd = os.path.join(ROOT, "tests", "golden")
            line["configs"] = [
                run_extra_config(eng, L, gf, torch, "vit_large_patch16_384, bf16-representable weights (f32 container), batch=128, 577-token attention",
                                 "large384", "bf16w", 128, 5, 3, os.path.join(gd, "large384_bf16w_b8.npz"), peaks, local_rank, stream),
                run_extra_config(eng, L, gf, torch, "vit_base_patch16_224 q8_0 model file (weights dequantised to f16 at upload), batch=256",
                                 "base", "q8_0", 256, 10, 3, os.path.join(gd, "base_q8_0.npz"), peaks, local_rank, stream),
            ]
        from oracle import ref
        if world == 1 and not args.no_cpu_baseline and not ref.available():
            line["cpu_baseline"] = None   # the compiled reference (oracle/_ref) is only built where its sources are present
        elif world == 1 and not args.no_cpu_baseline:
            nproc = host_threads()
            rate, nt, dt, tried = cpu_reference_rate(8, thread_candidates())
            line["cpu_baseline"] = {"value": rate, "unit": "images/s", "cores": nt, "kind": "reference",
                                    "sample": "8 images of the same ViT-B/16 f16 model through oracle/_ref vit_predict (%.1f s at %d threads), host has %d usable cpus" % (dt, nt, nproc),
                                    "threads_tried_images_per_s": {str(k): round(v, 2) for k, v in tried.items()}, "host": host_cpu_info()}
        print(json.dumps(line), flush=True)
    if model is not None:
        model.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
