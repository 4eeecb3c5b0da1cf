#!/usr/bin/env python
"""bench.py — LFDM hot-path benchmark (contract: see the task brief / DESIGN.md §Measurement).

One "step" = one full pass of the hot path over one batch: Generator.compute_fea -> 1000-step DDPM sampling of the
(B,3,40,32,32) latent flow/occlusion volume with the 3-D UNet -> 40-frame LFAE decode (+ all-gather of the frames
when more than one GPU takes part).  Metric: frames/s = global_batch * 40 / seconds (BASELINE.json).

  python bench.py --gpus 1 --steps 3 --warmup 3                      # our B200 path
  torchrun --nproc-per-node N bench.py --gpus N ...                  # weak scaling, one rank per GPU, NCCL
  python bench.py --impl reference ...                               # the reference's CPU arithmetic (oracle port)
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FRAMES = 40
# BASELINE.json configs (SURVEY.md §8d table).  `batch` = samples per GPU of the config as BASELINE.json quotes it.
CONFIGS = {
    "mug128": dict(yaml="mug128.yaml", image=128, latent=32, steps=1000, batch=8, unet_kw={},
                   name="MUG-128", baseline_config=2, unet_gflop_ref=235.10),
    "mhad128": dict(yaml="mhad128.yaml", image=128, latent=32, steps=1000, batch=8, unet_kw={},
                    name="MHAD-128", baseline_config=3, unet_gflop_ref=235.10),
    "natops128": dict(yaml="natops128.yaml", image=128, latent=32, steps=250, batch=8,
                      unet_kw=dict(learn_null_cond=True, use_deconv=False, padding_mode="reflect"),   # demo/demo_natops.py:23-32
                      name="NATOPS-128", baseline_config=4, unet_gflop_ref=None),
    "mug256": dict(yaml="mug256.yaml", image=256, latent=64, steps=1000, batch=2, unet_kw={},
                   name="MUG-256", baseline_config=5, unet_gflop_ref=940.48),
}
UNET_GFLOP_REF = 235.10       # reference-executed FLOPs per UNet eval per sample (SURVEY.md §8d)
# roofline.traffic: dram__bytes_read.sum + dram__bytes_write.sum per conv_tc_kernel launch, parsed at run time from the ncu
# launch list of one UNet evaluation at the bench geometry that is COMMITTED with the code (tools/measure_round.sh writes
# it; ncu cannot wrap the timed region).  null when the file is absent or predates the kernels.
NCU_LAUNCH_CSV = os.path.join(ROOT, "profiles", "r02_launches_eval.csv")


def ncu_conv_traffic():
    """-> (bytes per conv_tc launch, n launches, source) from the committed ncu CSV, or (None, 0, reason)"""
    import csv
    if not os.path.exists(NCU_LAUNCH_CSV):
        return None, 0, "profiles/r02_launches_eval.csv not present"
    rd = wr = 0.0
    n = 0
    ids = set()
    with open(NCU_LAUNCH_CSV, newline="") as f:
        rows = [r for r in csv.reader(f) if len(r) > 8]
    hdr = next((r for r in rows if "Kernel Name" in r and "Metric Name" in r), None)
    if hdr is None:
        return None, 0, "unrecognised ncu csv"
    ik, im, iu, iv, ii = hdr.index("Kernel Name"), hdr.index("Metric Name"), hdr.index("Metric Unit"), hdr.index("Metric Value"), hdr.index("ID")
    scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    for r in rows:
        if r is hdr or "conv_tc_kernel" not in r[ik]:
            continue
        if r[im] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
            v = float(r[iv].replace(",", "")) * scale.get(r[iu], 1.0)
            if r[im].endswith("read.sum"):
                rd += v
            else:
                wr += v
            ids.add(r[ii])
    n = len(ids)
    if n == 0:
        return None, 0, "no conv_tc_kernel rows with dram metrics"
    return (rd + wr) / n, n, f"profiles/r02_launches_eval.csv ({n} conv_tc_kernel launches: {rd / 1e9:.2f} GB read + {wr / 1e9:.2f} GB written)"


UNET_GFLOP_ALGO = 169.3       # after the legal hoists (what the kernels must do)
WARP_MB_PER_FRAME = 25.1      # K12 algorithmic bytes per frame per sample (SURVEY.md §8d)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sustained=d["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sustained=1400.0, src="fallback")


class ClockSampler:
    def __init__(self, dev_index):
        self.idx, self.rows, self.proc = dev_index, [], None

    def start(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i",
                                          str(self.idx), "-lms", "200"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i].lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


def usable_cores():
    """cores this process may really use: min(affinity mask, cgroup cpu quota) — os.cpu_count() over-counts in containers"""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(float(q) / float(per))))
    except Exception:
        pass
    return max(1, min(n, 64))


def build_model(cfg_name, sampling_steps=None):
    import torch
    import cvpr23_lfdm_b200 as P
    cfg = CONFIGS[cfg_name]
    torch.manual_seed(1234)
    import contextlib
    with contextlib.redirect_stdout(sys.stderr):       # the reference-shaped constructor prints ("using ddim samping ..."): stdout is ONE JSON line
        return _build(P, cfg, cfg_name, sampling_steps)


def _build(P, cfg, cfg_name, sampling_steps):
    return P.FlowDiffusion(is_train=False, sampling_timesteps=sampling_steps or cfg["steps"], img_size=cfg["latent"],
                           num_frames=FRAMES, timesteps=1000, config_pth=os.path.join(ROOT, "config", cfg["yaml"]),
                           pretrained_pth="", **cfg["unet_kw"])


DUMP_BYTES = 60 * 2 ** 20     # --dump-outputs: float32 bytes written in all, split evenly over the arrays


def dump_outputs(out_dir, arrays):
    """Writes each array as out_dir/<name>.npy (float32).  An array over its share of DUMP_BYTES is written as the 1-D
    vector of its elements at a fixed set of flat indices (seeded permutation, ascending), the same for every run."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    cap = DUMP_BYTES // 4 // len(arrays)
    for name, t in arrays.items():
        a = t.detach().float()
        if a.numel() > cap:
            idx = torch.randperm(a.numel(), generator=torch.Generator().manual_seed(0))[:cap].sort().values
            a = a.reshape(-1)[idx.to(a.device)]
        np.save(os.path.join(out_dir, f"{name}.npy"), a.cpu().numpy())


def cpu_baseline(threads=None, cfg_name="mug128", sampling_steps=None):
    """The reference's CPU arithmetic (oracle port, bit-exact vs the reference on this path) on a bounded sample:
    B=1, F=8-frame probe first; if the box is fast enough 2 full 40-frame UNet evals, else the probe scaled by 5;
    + compute_fea + 2 decoded frames; EXTRAPOLATED to the config's sampling steps + 40 frames."""
    import torch
    from oracle import lfdm_oracle as O
    cfg = CONFIGS[cfg_name]
    n_steps = sampling_steps or cfg["steps"]
    lat, isz = cfg["latent"], cfg["image"]
    threads = threads or usable_cores()
    torch.set_num_threads(threads)
    m = build_model(cfg_name, n_steps)
    pm = cfg["unet_kw"].get("padding_mode", "zeros")
    usd = {k: v.detach().cpu() for k, v in m.unet.state_dict().items()}
    gsd = {k: v.detach().cpu() for k, v in m.generator.state_dict().items()}
    img, cond = torch.rand(1, 3, isz, isz), torch.randn(1, 768)
    with torch.no_grad():
        t0 = time.perf_counter()
        skips = O.generator_encode(gsd, img)
        t_fea = time.perf_counter() - t0
        x = torch.randn(1, 3, FRAMES, lat, lat)
        fea5 = skips[-1].unsqueeze(2).repeat(1, 1, FRAMES, 1, 1)
        # probe: 8 of the 40 frames (the UNet is linear in F except the 40x40 temporal attention, <4 % of the FLOPs)
        xp = torch.cat([x, fea5], 1)[:, :, :8].contiguous()
        O.unet3d_forward(usd, xp, torch.tensor([999]), cond, padding_mode=pm)            # warm-up
        t0 = time.perf_counter()
        O.unet3d_forward(usd, xp, torch.tensor([999]), cond, padding_mode=pm)
        t_probe = time.perf_counter() - t0
        how = "2 full 40-frame UNet evals + sampler steps"
        if t_probe * 5 < 8.0:
            ts = []
            for i in range(2):
                t0 = time.perf_counter()
                eps = O.unet3d_forward(usd, torch.cat([x, fea5], 1), torch.tensor([998 - i]), cond, padding_mode=pm)
                x = O.p_sample_step(O.diffusion_buffers(1000), x, 998 - i, eps, torch.randn_like(x))
                ts.append(time.perf_counter() - t0)
            t_step = min(ts)
        else:
            t_step = t_probe * 5
            how = "one 8-frame UNet eval scaled x5 (box too slow for full evals inside the time bound)"
        flow, occ = x[:, :2, 0].permute(0, 2, 3, 1).contiguous(), (x[:, 2:3, 0] + 1) * 0.5
        t0 = time.perf_counter()
        for _ in range(2):
            O.generator_forward_with_flow(gsd, img, flow, occ)        # reference decodes per frame incl. the encoder
        t_frame = (time.perf_counter() - t0) / 2
    total = t_fea + n_steps * t_step + FRAMES * t_frame
    return dict(value=FRAMES / total, unit="frames/s", cores=threads, kind="port", extrapolated=True,
                sample=f"{cfg['name']} B=1: {how} ({t_step:.2f} s per 40-frame step), compute_fea ({t_fea:.2f} s), 2 decoded frames "
                       f"({t_frame:.3f} s each); EXTRAPOLATED to {n_steps} sampling steps + 40 frames = {total:.0f} s/video "
                       "(the unmodified reference ran BASELINE config 1 in full in the build container: 50 DDIM steps in 52.0 s "
                       "on 8 threads = 0.77 frames/s, tests/golden/r2_config1.pt)",
                t_step=t_step, t_frame=t_frame, t_fea=t_fea)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    vals = []
    base = None
    for i in range(args.warmup + args.steps):
        if i >= 1 and base is not None and args.steps + args.warmup > 2:
            # every step is the same bounded sample; keep the run short: re-measure at most 3 times in total
            if len(vals) >= 2:
                vals.append(vals[-1])
                continue
        base = cpu_baseline(cfg_name=args.config, sampling_steps=args.sampling_steps)
        vals.append(base["value"])
    v = sorted(vals[-args.steps:])[len(vals[-args.steps:]) // 2]
    total_s = FRAMES / v
    cfg = CONFIGS[args.config]
    line = {"metric": metric_name(args), "value": v, "unit": "frames/s", "impl": "reference",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": total_s * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(args),
                       "cpu_note": "reference arithmetic on the host cores, measured at B=1 on a bounded sample and extrapolated "
                                   "(CPU frames/s does not depend on the batch size)"},
            "cpu_baseline": {k: base[k] for k in ("value", "unit", "cores", "kind", "extrapolated", "sample")},
            "e2e": {"value": v, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def metric_name(args):
    cfg = CONFIGS[args.config]
    n = args.sampling_steps
    kind = "DDPM" if n >= 1000 else "DDIM"
    return f"frames/s ({cfg['image']}x{cfg['image']}, 40f, {n} {kind} steps)"


def workload_name(args):
    cfg = CONFIGS[args.config]
    n = args.sampling_steps
    return (f"{cfg['name']} batch={args.batch}/GPU, 40 frames, {n} {'DDPM' if n >= 1000 else 'DDIM'} steps, "
            "1 pass = compute_fea + sampling + 40-frame decode")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="mug128", choices=sorted(CONFIGS), help="BASELINE.json config family (default: config 2)")
    ap.add_argument("--strong", type=int, default=0, metavar="GLOBAL_BATCH",
                    help="strong scaling: fixed global batch split over the ranks (per-rank batch = GLOBAL_BATCH / gpus)")
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=0, help="samples per GPU (default: the config's, 8 for config 2)")
    ap.add_argument("--sampling-steps", type=int, default=0, help="default: the config's (1000 DDPM for config 2)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write the last step's outputs (sample_out_vid, sample_warped_vid, "
                         "sample_vid_grid, sample_vid_conf; a seeded sample of the larger ones) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs --impl ours")
    cfg = CONFIGS[args.config]
    args.sampling_steps = args.sampling_steps or cfg["steps"]
    if args.strong:
        assert args.strong % args.gpus == 0, "--strong GLOBAL_BATCH must be divisible by --gpus"
        args.batch = args.strong // args.gpus
    args.batch = args.batch or cfg["batch"]
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    import cvpr23_lfdm_b200 as P
    from cvpr23_lfdm_b200 import _lib
    from cvpr23_lfdm_b200.engine import ops

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    _lib.lib()   # fail loudly if the CUDA library is missing

    B = args.batch
    ISZ, LAT = cfg["image"], cfg["latent"]
    model = build_model(args.config, args.sampling_steps)
    model = model.to(dev).eval()
    g = torch.Generator().manual_seed(1234 + rank)
    img_h = torch.rand(B, 3, ISZ, ISZ, generator=g).pin_memory()
    cond_h = torch.randn(B, 768, generator=g).pin_memory()
    img_d, cond_d = img_h.to(dev), cond_h.to(dev)
    out_h = torch.empty((B, 3, FRAMES, ISZ, ISZ), pin_memory=True)
    gather = torch.empty((world * B, 3, FRAMES, ISZ, ISZ), device=dev) if world > 1 else None
    flush = torch.empty(256 * 1024 * 1024 // 4, device=dev)

    def one_pass(e2e):
        if e2e:
            i_d, c_d = img_h.to(dev, non_blocking=True), cond_h.to(dev, non_blocking=True)
        else:
            i_d, c_d = img_d, cond_d
        model.set_sample_input(i_d, c_d)
        model.sample_one_video(cond_scale=1.0)
        if world > 1:
            dist.all_gather_into_tensor(gather, model.sample_out_vid.contiguous())
        if e2e:
            out_h.copy_(model.sample_out_vid, non_blocking=True)

    def timed(n, e2e):
        times = []
        for _ in range(n):
            flush.fill_(1.0)                      # L2 flush between timed iterations (256 MiB > 126 MB L2)
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            one_pass(e2e)
            e1.record()
            torch.cuda.synchronize()
            t = torch.tensor([e0.elapsed_time(e1)], device=dev)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            times.append(t.item())
        return times

    for _ in range(args.warmup):
        one_pass(False)
    torch.cuda.synchronize()
    calls0 = _lib.launch_count
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    t_dev = timed(args.steps, False)
    clocks = sampler.stop() if rank == 0 else None
    seng = model.diffusion._engine()
    t_e2e = timed(args.steps, True)
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, {
            "sample_out_vid": gather if world > 1 else model.sample_out_vid, "sample_warped_vid": model.sample_warped_vid,
            "sample_vid_grid": model.sample_vid_grid, "sample_vid_conf": model.sample_vid_conf})

    ms = sum(t_dev) / len(t_dev)
    ms_e2e = sorted(t_e2e)[len(t_e2e) // 2]
    frames = world * B * FRAMES
    value = frames / (ms / 1e3)
    e2e_value = frames / (ms_e2e / 1e3)

    # ---- live roofline of the dominant kernel (tcgen05 implicit-GEMM conv): CUDA events around every launch of one
    # eager UNet evaluation at the bench batch (outside the timed region)
    roof = None
    if rank == 0:
        pk = peaks()
        eng = model.unet.engine()
        fea = model.generator.compute_fea(img_d)
        fea_conv = eng.prepare_fea(fea)
        x = torch.randn(B, 3, FRAMES, LAT, LAT, device=dev)
        ss = eng.scale_shift(torch.full((B,), 500, device=dev, dtype=torch.long), cond_d)
        eng.forward_hoisted(x, fea_conv, ss)
        torch.cuda.synchronize()
        ops.PROFILE = []
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        # park the GPU for ~30 ms so the host enqueues the whole evaluation ahead of it: every event pair below then
        # brackets pure device time of its launch (no host launch latency inside the interval)
        torch.cuda._sleep(int(30e-3 * 1.9e9))
        ev0.record()
        eng.forward_hoisted(x, fea_conv, ss)
        ev1.record()
        torch.cuda.synchronize()
        prof, ops.PROFILE = ops.PROFILE, None
        tc = [(f, a.elapsed_time(b)) for (_, e, f, a, b, _) in prof if e == "tc"]
        simt = [(f, a.elapsed_time(b)) for (_, e, f, a, b, _) in prof if e != "tc"]
        tc_ms, tc_fl = sum(t for _, t in tc), sum(f for f, _ in tc)
        tc_bytes = sum(ab for (_, e, _, _, _, ab) in prof if e == "tc")
        achieved = tc_fl / (tc_ms * 1e-3) / 1e12 if tc_ms > 0 else 0.0
        traffic, traffic_n, traffic_src = ncu_conv_traffic() if args.config == "mug128" and B == 8 else (None, 0, "ncu launch list is committed for config 2 (MUG-128, B=8) only")
        roof = {"bound": "tensor", "kernel": "conv_tc_kernel (tcgen05 implicit GEMM, split-bf16 x3)",
                "achieved": achieved, "peak": pk["tf_sustained"], "unit": "TFLOP/s", "frac": achieved / pk["tf_sustained"],
                "traffic": traffic, "traffic_unit": "bytes/launch (dram read+write, ncu)", "traffic_source": traffic_src,
                "algorithmic_bytes_per_launch": tc_bytes / max(1, len(tc)),
                "peak_source": pk["src"] + " bf16 sustained", "launches": len(tc),
                "avg_launch_ms": tc_ms / max(1, len(tc)), "algorithmic_gflop_per_eval": tc_fl / 1e9,
                "executed_mma_flops_x": 3, "conv_ms_per_eval": tc_ms, "simt_conv_ms_per_eval": sum(t for _, t in simt),
                "unet_eval_ms_eager": ev0.elapsed_time(ev1)}

    cpu = None
    if rank == 0 and not args.no_cpu_baseline:
        try:
            cpu = cpu_baseline(cfg_name=args.config, sampling_steps=args.sampling_steps)
            cpu = {k: cpu[k] for k in ("value", "unit", "cores", "kind", "extrapolated", "sample")}
        except Exception as e:      # never lose the measured line to a baseline problem
            cpu = {"error": repr(e)}

    if rank == 0:
        st = getattr(seng, "last_stats", {})
        per_step = st.get("calls_per_step", 0)
        launches = per_step * st.get("steps", 0) + st.get("other_calls", 0)
        line = {
            "metric": metric_name(args),
            "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms, "higher_is_better": True, "scaling": "strong" if args.strong else "weak", "vs_baseline": None,
            "dtype": "f32 (split-bf16 x3 tensor-core products, fp32 accumulate)",
            "data": "synthetic",
            "config": {"workload": workload_name(args), "baseline_config": cfg["baseline_config"],
                       "global_batch": world * B, "l2": "256 MiB flush buffer written between timed iterations; per-step working set >> L2",
                       "weights": "random init, seed 1234", "cuda_graph": os.environ.get("LFDM_CUDA_GRAPH", "1") == "1",
                       "fused_temporal_attention": os.environ.get("LFDM_FUSED_ATTN", "1") == "1"},
            "e2e": {"value": e2e_value, "unit": "frames/s", "ms_per_step": ms_e2e, "samples_ms": [round(t, 2) for t in t_e2e],
                    "h2d_bytes_per_step": (img_h.numel() + cond_h.numel()) * 4, "d2h_bytes_per_step": out_h.numel() * 4},
            "gpu_launches": int(launches), "gpu_launches_per_sampling_step": int(per_step),
            "clocks": clocks, "roofline": roof, "cpu_baseline": cpu,
            "ref_equiv_tflops": world * B * (args.sampling_steps * cfg["unet_gflop_ref"]) / (ms / 1e3) / 1e3 if cfg["unet_gflop_ref"] else None,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
