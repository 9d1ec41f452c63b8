#!/usr/bin/env python
"""bench.py — faces/sec of the SMIRK hot path (encode -> FLAME -> render @224^2, and the full cycle with
SmirkGenerator) on N B200s.

Contract (see DESIGN.md §Measurement):
  python bench.py --gpus N --steps K --warmup W            product arm (under torchrun for N > 1)
  python bench.py --impl reference ...                     the reference's CPU path (oracle port) arm

A step = one pass of the hot path over one batch of synthetic 224x224 RGB faces per GPU.  One run measures TWO
workloads and prints ONE JSON line:
  headline      BASELINE.json configs[1]: encoder + FLAME + raster, batch 32 per GPU (`--batch`);
  `full_cycle`  BASELINE.json configs[2]/[4]: encoder -> FLAME -> raster -> SmirkGenerator, batch 256 per GPU
                (`--full-batch`; `--no-full-cycle` skips it, `--generator` makes it the headline instead).
For each workload:
  value     faces/s with the input batches resident in HBM: CUDA-graph replay over `--slots` pipeline lanes, CUDA events
            around exactly K timed steps, split into `--windows` back-to-back windows; the reported figure is the MEDIAN
            window (min / max / relative spread alongside), max over ranks per window.  Inputs rotate over a set of
            batches larger than L2.  For N > 1 the NCCL all-gather of the final outputs runs INSIDE the timed region
            (on a communication stream, overlapping the next batch); `no_gather` repeats the measurement without it.
  e2e       the same metric through SmirkPipeline.run_host(): pinned host images -> H2D -> graph -> D2H of rendered
            image + vertices + FLAME parameters (+ reconstructed image) into pinned host memory, every step.
  roofline  dominant kernel (largest share of device time) from the library's built-in event profiler, live in this
            run: algorithmic bytes (or FLOPs) per launch / mean launch time; plus `in_situ`: step-level compulsory
            bytes, measured DRAM traffic and FLOPs divided by the TIMED ms_per_step (what the mix achieves, not the
            kernel alone).
  parity    max errors of the timed configuration against the CPU oracle, checked in-run on one batch.
  cpu_baseline: `bench.py --impl reference` run as a child process on the host cores (so both arms share one code path
            and one thread-count choice).
--dump-outputs DIR writes, after the timed steps, the outputs of the last timed step of each workload as float32 .npy
files (headline: <key>.npy, full cycle: full_cycle_<key>.npy); inputs and weights are seeded, so two builds run with the
same arguments can be compared output for output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True                              # the tree may be read-only: bench.py writes nothing there

METRIC = "faces/sec encode->FLAME->render @224^2"
UNIT = "faces/s"
FLOPS_PER_FACE = {False: 0.941e9, True: 28.77e9}            # SURVEY.md §8d: encoder+FLAME ; + generator
COMPULSORY_BYTES_PER_FACE = {False: 1.328e6, True: 2.532e6}
CONSTANT_BYTES = {False: 38.0e6, True: 163.5e6}             # weights / FLAME constants read once per step
DUMP_BYTES = 60_000_000                                     # --dump-outputs: all files together stay below 64 MB


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=float(d["hbm_gbs"]), tensor=float(d.get("bf16_tflops", 1590.0)),
                    tensor_sustained=float(d.get("bf16_tflops_sustained", 1400.0)), source="measured")
    return dict(hbm=6650.0, tensor=1590.0, tensor_sustained=1400.0, source="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.rows.append([x.strip() for x in ln.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); pw.append(float(r[3]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


def workload_name(generator, batch):
    if generator:
        return "configs[2]: full cycle encoder->FLAME->raster->masking->smirk_generator 224x224, batch %d per GPU" % batch
    return "configs[1]: encoder+FLAME+raster 224x224, batch %d per GPU" % batch


# ------------------------------------------------------------------------------------------- CPU arm
_CPU_STATE = {}


def cpu_reference_pass(root, sample, with_generator, threads=None, seed=9001):
    """One pass of the reference's CPU path (oracle port) over `sample` faces; returns seconds."""
    import torch
    from smirk_b200 import synth_inputs
    from oracle import encoder_ref, flame_ref, render_ref, generator_ref
    if threads:
        torch.set_num_threads(threads)
    st = _CPU_STATE
    if "enc_sd" not in st:
        import smirk_b200
        enc = smirk_b200.SmirkEncoder()
        st["enc_sd"] = synth_inputs.random_state_dict(enc.state_dict(), seed=7)
        st["fc"], st["rc"] = flame_ref.FlameConstants(root), render_ref.RenderConstants(root)
    if with_generator and "gen_sd" not in st:
        import smirk_b200
        gen = smirk_b200.SmirkGenerator(6, 3, 32, 5)
        st["gen_sd"] = synth_inputs.random_state_dict(gen.state_dict(), seed=7)
    img = synth_inputs.images(sample, seed)
    hull = synth_inputs.hull_masks(sample, seed + 1) if with_generator else None
    if with_generator:
        from oracle import masking_ref
        base_prob = synth_inputs.face_probabilities(st["fc"].faces_tensor.shape[0])
    t0 = time.perf_counter()
    with torch.no_grad():
        p = encoder_ref.encoder_forward_ref(st["enc_sd"], img)
        p = {k: v for k, v in p.items() if not k.startswith("_")}
        fo = flame_ref.flame_forward_ref(st["fc"], p)
        ro = render_ref.render_forward_ref(st["rc"], fo["vertices"], p["cam"], landmarks_fan=fo["landmarks_fan"],
                                           landmarks_mp=fo["landmarks_mp"])
        if with_generator:                                                     # demo.py:138-167 on the CPU (torch RNG draws)
            tv, faces, N = ro["transformed_vertices"], st["fc"].faces_tensor, int(0.05 * 224 * 224)
            w = masking_ref.face_probabilities_ref(tv, faces, base_prob)
            idx = torch.multinomial(w, N, replacement=True)
            u, v = torch.rand(sample * N), torch.rand(sample * N)
            o = u + v > 1
            u[o], v[o] = 1 - u[o], 1 - v[o]
            pts = masking_ref.points_from_coords_ref(tv, faces, idx, torch.stack((1 - (u + v), u, v), 1).view(sample, N, 3))
            rsing = torch.randint(0, 2, (sample,)) * 2 - 1
            rbound = (N * 0.2 * (torch.rand(sample) * 4 + 1) ** rsing).long()
            rmask = 1 - (ro["rendered_img"] == 0).all(dim=1, keepdim=True).float()
            masked = masking_ref.masking_ref(img, hull, img * masking_ref.point_mask_ref(pts, rbound, 224), 10, rendered_mask=rmask,
                                             noise_mult=torch.randn(img.shape) * 0.05 + 1,
                                             random_centres=torch.bernoulli(torch.ones(sample, 1, 224, 224) * 0.01))
            generator_ref.generator_forward_ref(st["gen_sd"], torch.cat([ro["rendered_img"], masked], 1))
    return time.perf_counter() - t0


def pick_cpu_threads(root, with_generator):
    """torch's intra-op pool is pathological at some thread counts on small-kernel workloads (SURVEY.md §6: lbs() 1.4 ms
    at 1 thread vs 27 ms at 8).  Time a 4-face pass (best of two) at a few thread counts and keep the fastest; the
    choice is cached per host so the product arm's cpu_baseline and the reference arm report the same configuration."""
    import torch
    n = os.cpu_count() or 1
    cache = os.path.join(tempfile.gettempdir(), "smk_cpu_threads_%d_%d.json" % (n, int(with_generator)))
    try:
        c = int(json.load(open(cache))["threads"])
        if 1 <= c <= n:
            torch.set_num_threads(c)
            return c
    except Exception:
        pass
    cands = sorted({max(1, n // 8), max(1, n // 4), max(1, n // 2), n, min(n, 16), min(n, 32)})
    cpu_reference_pass(root, 1, with_generator, threads=cands[0])                 # build state, warm caches
    best = None
    for c in cands:
        sec = min(cpu_reference_pass(root, 4, with_generator, threads=c) for _ in range(2))
        if best is None or sec < best[1]:
            best = (c, sec)
    torch.set_num_threads(best[0])
    try:
        json.dump({"threads": best[0]}, open(cache, "w"))
    except OSError:
        pass
    return best[0]


def run_reference_arm(args, root, rank):
    """--impl reference: the reference's own CPU implementation (oracle port; the reference is pure Python + third-party
    wheels that are not installable offline and cannot travel to the GPU box).  Rank 0 only.  K timed steps, each one
    pass over a full batch of the same synthetic workload."""
    if rank != 0:
        return
    import torch
    B = args.batch
    threads = pick_cpu_threads(root, args.generator)
    W = max(1, min(args.warmup, 2))
    for i in range(W):
        cpu_reference_pass(root, B, args.generator, threads=threads, seed=8000 + i)
    K = max(1, args.steps)
    t = [cpu_reference_pass(root, B, args.generator, threads=threads, seed=9001 + 2 * i) for i in range(K)]
    sec = statistics.median(t)
    val = B / sec
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": K,
        "warmup": W, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args.generator, B), "global_batch": B, "faces_per_gpu_per_step": B,
                   "image": "224x224 RGB fp32", "faces_per_step": B, "timing": "median of %d passes (min %.1f ms, max %.1f ms)" % (K, min(t) * 1e3, max(t) * 1e3)},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port", "host_cpus": os.cpu_count(),
                         "sample": "%d faces per step (one full batch of the same synthetic workload), %d steps; oracle port: torch CPU ops (oneDNN) + C rasteriser" % (B, K)},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def child_cpu_baseline(args, generator, batch, steps=3):
    """Run the reference arm as a child process (full CPU affinity, its own torch thread pool) and return its
    cpu_baseline object — the product arm and the reference arm thereby report the same baseline."""
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--gpus", "1", "--steps", str(steps), "--warmup", "1",
           "--batch", str(batch)] + (["--generator"] if generator else [])
    env = dict(os.environ)
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "MASTER_ADDR", "MASTER_PORT"):
        env.pop(k, None)
    try:
        allcpus = set(range(os.cpu_count() or 1))
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env,
                           preexec_fn=lambda: os.sched_setaffinity(0, allcpus))
        for ln in reversed(r.stdout.splitlines()):
            if ln.startswith("{"):
                return json.loads(ln)["cpu_baseline"]
        return {"error": (r.stderr or "no output")[-300:]}
    except Exception as e:                                    # the baseline is a report, never a reason to lose the GPU numbers
        return {"error": repr(e)[:300]}


# --------------------------------------------------------------------------------------- product arm
PRECISIONS = {"fp32": 0, "tf32-unfused": 1, "tf32": 2, "tf32x3": 3}


class Ctx:
    pass


def timed_windows(cx, step, join, K, W, R):
    """W warm-up steps (indices 0..W-1), then exactly K timed steps (indices W..W+K-1) split into min(R, K) back-to-back
    windows whose lengths differ by at most one, each bracketed by CUDA events on the current stream (which joins every
    lane / copy / communication stream before the closing event); barrier + synchronize on both sides.  Returns the
    per-window ms per step, max over ranks, and the window lengths."""
    import torch
    R = max(1, min(R, K))
    sizes = [K // R + (1 if r < K % R else 0) for r in range(R)]
    for i in range(W):
        step(i)
    join()
    cx.barrier()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(R)]
    it = W
    cx.barrier()
    for r in range(R):
        ev[r][0].record()
        for _ in range(sizes[r]):
            step(it)
            it += 1
        join()
        ev[r][1].record()
    cx.barrier()
    t = torch.tensor([a.elapsed_time(b) / n for (a, b), n in zip(ev, sizes)], device=cx.dev, dtype=torch.float64)
    if cx.dist is not None:
        cx.dist.all_reduce(t, op=cx.dist.ReduceOp.MAX)
    return [float(x) for x in t.tolist()], sizes


def window_stats(ms, sizes):
    """ms: per-window ms per step."""
    med = statistics.median(ms)
    return {"n": len(ms), "steps_per_window": sizes, "median_ms_per_step": med, "min_ms_per_step": min(ms),
            "max_ms_per_step": max(ms), "rel_spread": (max(ms) - min(ms)) / med if med > 0 else None}


def sample_outputs(outs, max_bytes, seed=0):
    """Host float32 copies of one step's outputs (every array is batch-major).  When the whole batch exceeds
    ``max_bytes``, every array keeps the same fixed, seeded subset of the faces, in batch order."""
    import torch
    B = next(iter(outs.values())).shape[0]
    per_face = sum(t[0].numel() * 4 for t in outs.values())
    n = min(B, max(1, max_bytes // per_face))
    idx = torch.randperm(B, generator=torch.Generator().manual_seed(seed))[:n].sort().values
    return {k: t[idx.to(t.device)].float().cpu().numpy() for k, t in outs.items()}


def run_workload(cx, args, B, generator, slots, R, with_cpu, dump_bytes=0):
    """Measure one workload (device-resident, e2e, ± gather for N > 1, kernel breakdown, parity).  Returns a dict."""
    import torch
    import smirk_b200
    from smirk_b200 import _lib, synth_inputs
    from smirk_b200.pipeline import SmirkPipeline
    dev, world, rank = cx.dev, cx.world, cx.rank
    K, W = args.steps, max(args.warmup, 3)
    enc = smirk_b200.SmirkEncoder()
    enc.load_state_dict(synth_inputs.random_state_dict(enc.state_dict(), seed=7))
    enc = enc.eval().to(dev)
    enc.precision = PRECISIONS[args.precision]
    gen = None
    if generator:
        gen = smirk_b200.SmirkGenerator(6, 3, 32, 5)
        gen.load_state_dict(synth_inputs.random_state_dict(gen.state_dict(), seed=7))
        gen = gen.eval().to(dev)
        gen.precision = 0 if args.precision == "fp32" else 1
    fl, rd = smirk_b200.FLAME().to(dev), smirk_b200.Renderer().to(dev)
    stage = None
    if generator:                               # the real masking step between renderer and generator (demo.py:138-165), draws on the device
        from smirk_b200.masking import MaskingStage
        stage = MaskingStage(fl.faces_tensor, synth_inputs.face_probabilities(fl.faces_tensor.shape[0]), seed=1234 + rank)
    pipe = SmirkPipeline(enc, fl, rd, gen, device=dev, slots=slots, masking=stage)

    # rotating input set larger than L2 (126 MB): Rset batches of B x 602 KB (x2 with the masked image)
    per = B * 224 * 224 * 4 * (4 if generator else 3)
    Rset = max(2, -(-160_000_000 // per))
    host_imgs = [synth_inputs.images(B, 5000 + rank * 100 + i).pin_memory() for i in range(Rset)]
    host_masks = [synth_inputs.hull_masks(B, 6000 + rank * 100 + i).pin_memory() for i in range(Rset)] if generator else None
    dev_imgs = [h.to(dev) for h in host_imgs]
    dev_masks = [h.to(dev) for h in host_masks] if generator else None
    rec = pipe.capture(B)
    for lane in range(1, pipe.slots):
        pipe.capture(B, lane)
    keys = ("rendered_img", "vertices", "params") + (("reconstructed_img",) if generator else ())

    def dev_step(i):            # batch i goes to lane i % slots (own stream + graph replica): consecutive batches overlap
        pipe.submit(i, dev_imgs[i % Rset], dev_masks[i % Rset] if generator else None)

    def host_step(i):
        cx.last = pipe.run_host(host_imgs[i % Rset], i, host_masks[i % Rset] if generator else None, keys)

    out = {"batch": B, "launches_per_step": int(rec["launches"])}
    faces = B * world
    gather_keys = pipe.enable_gather(keys, backend=args.gather_backend) if (world > 1 and not args.no_gather) else ()
    sampler = ClockSampler(cx.local)
    if rank == 0:
        sampler.start()
    ms, sizes = timed_windows(cx, dev_step, pipe.join, K, W, R)
    out["clocks"] = sampler.stop() if rank == 0 else None
    if dump_bytes and rank == 0:                # the lane of the last timed step still holds its outputs
        out["dump"] = sample_outputs(pipe.capture(B, (W + K - 1) % pipe.slots)["out"], dump_bytes)
    out["windows"] = window_stats(ms, sizes)
    out["ms_per_step"] = out["windows"]["median_ms_per_step"]
    out["value"] = faces / (out["ms_per_step"] / 1e3)
    h2d, d2h = pipe.bytes_per_step(B, keys)
    ms2, sizes2 = timed_windows(cx, host_step, pipe.join, K, W, R)
    out["e2e"] = {"value": faces / (statistics.median(ms2) / 1e3), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                  "ms_per_step": statistics.median(ms2), "windows": window_stats(ms2, sizes2),
                  "api": "SmirkPipeline.run_host (pinned host in/out, %d lanes, copies on their own streams)" % pipe.slots,
                  "host_checksum": float(cx.last["params"].double().abs().sum())}          # touches the host result
    if gather_keys:
        gb = pipe.gather_bytes_per_step(B)
        how = {"nccl": "NCCL all_gather_into_tensor", "p2p": "copy-engine pushes of every output into the CUDA-IPC mapped gather buffers of the peers over NVLink (csrc/peer.cu; own shard stays in place)"}.get(pipe._gather_backend, str(pipe._gather_backend))
        out["gather"] = {"backend": pipe._gather_backend,
                         "collective": "%s of %s per step, on a communication stream inside the timed region" % (how, "+".join(gather_keys)),
                         "recv_bytes_per_rank_per_step": gb, "recv_gbs_per_rank": gb / (out["ms_per_step"] * 1e-3) / 1e9}
        p2p = getattr(pipe, "_p2p", None)
        if pipe._gather_backend == "p2p" and isinstance(p2p, dict):
            out["gather"]["form"] = "packed: one staging copy, one push per peer, lane released after the pack" if p2p.get("pack") else "direct: one push per (output, peer)"
        pipe.enable_gather(())
        ms3, _ = timed_windows(cx, dev_step, pipe.join, K, W, R)
        ms4, _ = timed_windows(cx, host_step, pipe.join, K, W, R)
        out["no_gather"] = {"value": faces / (statistics.median(ms3) / 1e3), "ms_per_step": statistics.median(ms3),
                            "e2e_value": faces / (statistics.median(ms4) / 1e3)}

    if rank != 0:
        return out
    # ---- per-kernel breakdown (eager, event-bracketed launches) ----
    L = _lib.lib()
    for i in range(2):
        pipe.forward(dev_imgs[i % Rset], dev_masks[i % Rset] if generator else None)
    torch.cuda.synchronize(dev)
    L.smk_profiler_reset(); L.smk_profiler_enable(1)
    NP = 5 if B <= 64 else 2
    for i in range(NP):
        pipe.forward(dev_imgs[(i + 3) % Rset], dev_masks[(i + 3) % Rset] if generator else None)
    torch.cuda.synchronize(dev)
    breakdown = _lib.profiler_report()
    L.smk_profiler_enable(0); L.smk_profiler_reset()
    peaks = cx.peaks
    tot = sum(v["ms"] for v in breakdown.values())
    for v in breakdown.values():
        v["share"] = v["ms"] / tot
        v["ms_per_launch"] = v["ms"] / v["launches"]
        v["gbs"] = v["bytes"] / v["ms"] / 1e6
        v["tflops"] = v["flops"] / v["ms"] / 1e9
    top_tag, top = max(breakdown.items(), key=lambda kv: kv[1]["ms"])
    # Every tensor-core kernel here computes in TF32: its ceiling is HALF the measured bf16 GEMM peak (tcgen05 kind::tf32
    # runs at half the kind::f16 rate), and the hbm/tensor ridge is judged against that.
    tf32_peak = peaks["tensor"] / 2.0
    ai = top["flops"] / max(top["bytes"], 1.0)
    ridge = tf32_peak * 1e3 / peaks["hbm"]
    if "tc" in top_tag and ai > ridge:
        roof = {"bound": "tensor", "achieved": top["tflops"], "peak": tf32_peak, "unit": "TFLOP/s",
                "peak_note": "TF32 = measured bf16 cuBLAS peak / 2"}
    else:
        roof = {"bound": "hbm", "achieved": top["gbs"], "peak": peaks["hbm"], "unit": "GB/s"}
    traffic, step_traffic = None, None
    tname = "r02_ncu_dram_traffic_%s_b%d_%s.json" % ("c3" if generator else "c2", B, args.precision)
    tpath = os.path.join(ROOT, "profiles", tname)
    if os.path.exists(tpath):
        tj = json.load(open(tpath))
        tk = tj.get("kernels", {}).get(top_tag.split(":")[0])
        traffic = tk["traffic_bytes_per_launch"] if tk else None
        step_traffic = tj.get("step_traffic_bytes")
    roof.update(frac=roof["achieved"] / roof["peak"], traffic=traffic, kernel=top_tag, share_of_step=top["share"],
                launches_per_step=top["launches"] / NP, us_per_launch=top["ms_per_launch"] * 1e3, peak_source=peaks["source"],
                arithmetic_intensity=ai, ridge_flop_per_byte=ridge,
                algorithmic_bytes_per_launch=top["bytes"] / top["launches"], algorithmic_flops_per_launch=top["flops"] / top["launches"])
    # in-situ: what the TIMED pipeline (all lanes and streams overlapping) achieves per GPU
    sec = out["ms_per_step"] * 1e-3
    comp = COMPULSORY_BYTES_PER_FACE[generator] * B + CONSTANT_BYTES[generator]
    roof["in_situ"] = {
        "ms_per_step": out["ms_per_step"],
        "compulsory_bytes_per_step": comp, "hbm_frac_compulsory": comp / sec / 1e9 / peaks["hbm"],
        "dram_traffic_bytes_per_step": step_traffic,
        "hbm_frac_traffic": (step_traffic / sec / 1e9 / peaks["hbm"]) if step_traffic else None,
        "tflops": FLOPS_PER_FACE[generator] * B / sec / 1e12,
        "tensor_frac_tf32": FLOPS_PER_FACE[generator] * B / sec / 1e12 / tf32_peak,
        "tensor_frac_tf32_sustained": FLOPS_PER_FACE[generator] * B / sec / 1e12 / (peaks["tensor_sustained"] / 2.0),
        "eager_serial_ms_per_step": tot / NP,
    }
    out["roofline"] = roof
    out["kernel_shares"] = {k: round(v["share"], 4) for k, v in sorted(breakdown.items(), key=lambda kv: -kv[1]["ms"])[:8]}
    if args.profile_out:
        suffix = "_c3" if generator else "_c2"
        with open(args.profile_out.replace(".json", suffix + ".json"), "w") as fh:
            json.dump({"batch": B, "steps_profiled": NP, "eager_ms_per_step": tot / NP, "kernels": breakdown}, fh, indent=1)

    # ---- parity of the timed configuration, in-run on one batch (the oracle is the checker only) ----
    if not args.no_parity:
        try:
            from oracle import parity_check
            nb = min(B, 32)
            img = synth_inputs.images(nb, 5000)
            p = enc(img.to(dev))
            fo = fl.forward(p)
            ro = rd.render_full(fo["vertices"], p["cam"])
            rep = parity_check.pipeline_report(cx.root, enc.state_dict(), img,
                                               {"params_dict": p, "vertices": fo["vertices"], "rendered_img": ro["rendered_img"],
                                                "transformed_vertices": ro["transformed_vertices"], "pix_to_face": ro["pix_to_face"]})
            rep["checked_against"] = "CPU oracle (oracle/: torch fp32 restatement + C rasteriser), %d faces of the timed workload" % nb
            rep["north_star"] = {"vertices_rel<=1e-4": rep["vertices_rel"] <= 1e-4, "pixels_stage_abs<=1.7e-4": rep["pixels_stage_abs"] <= 1.7e-4,
                                 "p2f_stage_bit_exact": rep.get("p2f_stage_mismatch") == 0}
            out["parity"] = rep
        except Exception as e:
            out["parity"] = {"error": repr(e)[:300]}
    if with_cpu:
        out["cpu_baseline"] = child_cpu_baseline(args, generator, min(B, 32), steps=3)
    del pipe
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="smirk_b200", choices=["smirk_b200", "reference"])
    ap.add_argument("--batch", type=int, default=32, help="faces per GPU per step of the headline workload (configs[1] = 32)")
    ap.add_argument("--full-batch", type=int, default=256, help="faces per GPU per step of the full-cycle workload (configs[2]/[4] = 256)")
    ap.add_argument("--generator", action="store_true", help="make the full cycle (with SmirkGenerator) the headline workload at --batch")
    ap.add_argument("--no-full-cycle", action="store_true", help="skip the extra full_cycle block")
    ap.add_argument("--windows", type=int, default=1, help="split the K timed steps into this many back-to-back windows (median reported)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-gather", action="store_true", help="N > 1: leave the NCCL all-gather of the outputs out of the timed region")
    ap.add_argument("--gather-backend", default="auto", choices=["auto", "nccl", "p2p"],
                    help="N > 1: how the final outputs are all-gathered (auto: peer-to-peer copy-engine pushes if every rank can map its peers, else NCCL)")
    ap.add_argument("--no-affinity", action="store_true", help="do not bind the rank to its GPU's NUMA node")
    ap.add_argument("--slots", type=int, default=4, help="pipeline lanes: consecutive batches alternate over this many stream/graph replicas")
    ap.add_argument("--full-slots", type=int, default=2)
    ap.add_argument("--profile-out", default=None, help="write the per-kernel breakdown JSON here (suffix _c2 / _c3 added)")
    ap.add_argument("--precision", default="tf32x3", choices=sorted(PRECISIONS),
                    help="encoder arithmetic.  tf32x3: tcgen05 tensor cores with error-compensated 3xTF32 products (fp32-equivalent; "
                         "the parity path and the default); tf32: plain TF32 tensor cores (the reference's cuDNN default); "
                         "fp32: exact fp32 CUDA cores.  The generator runs TF32 tcgen05 unless fp32 is chosen.")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the timed steps, write the outputs of the last timed step of each workload to DIR/<name>.npy (float32, "
                         "under 64 MB in all: a fixed, seeded subset of the faces when a batch is larger; bench_outputs/ is git-ignored)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "smirk_b200":
        ap.error("--dump-outputs applies to the product arm")
    if args.profile_out:
        args.profile_out = os.path.abspath(args.profile_out)
    if args.dump_outputs:
        args.dump_outputs = os.path.abspath(args.dump_outputs)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    from smirk_b200 import synth_assets
    root = synth_assets.materialize(os.path.join(tempfile.gettempdir(), "smk_assets_bench_%d" % rank))
    os.chdir(root)

    if args.impl == "reference":
        run_reference_arm(args, root, rank)
        return

    affinity = None
    if not args.no_affinity:
        from smirk_b200 import affinity as aff
        affinity = aff.pin_to_gpu(local)                       # before torch allocates any pinned memory
    import torch
    assert torch.cuda.is_available(), "bench.py (product arm) needs a GPU; there is no CPU fallback"
    torch.cuda.set_device(local)
    cx = Ctx()
    cx.dev, cx.rank, cx.world, cx.local, cx.root, cx.peaks, cx.last = torch.device("cuda", local), rank, world, local, root, load_peaks(), None
    cx.dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=cx.dev)
        cx.dist = dist
    assert world == args.gpus, "launch with torchrun --nproc-per-node %d (WORLD_SIZE=%d)" % (args.gpus, world)

    def barrier():
        if cx.dist is not None:
            cx.dist.barrier()
        torch.cuda.synchronize(cx.dev)
    cx.barrier = barrier

    with_full = not args.generator and not args.no_full_cycle
    dump_bytes = DUMP_BYTES // (2 if with_full else 1) if args.dump_outputs else 0
    head = run_workload(cx, args, args.batch, args.generator, args.slots, max(1, args.windows), with_cpu=(world == 1 and not args.no_cpu_baseline),
                        dump_bytes=dump_bytes)
    full = None
    if with_full:
        full = run_workload(cx, args, args.full_batch, True, args.full_slots, max(1, args.windows), with_cpu=False, dump_bytes=dump_bytes)

    if rank == 0:
        B, K = args.batch, args.steps
        line = {
            "metric": METRIC, "value": head["value"], "unit": UNIT, "n_gpus": world, "steps": K, "warmup": max(args.warmup, 3),
            "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": {"tf32x3": "tf32x3", "tf32": "tf32", "tf32-unfused": "tf32", "fp32": "f32"}[args.precision],
            "data": "synthetic",
            "config": {"workload": workload_name(args.generator, B), "precision": args.precision,
                       "arithmetic": {"tf32x3": "encoder convs: tcgen05 TF32 products, 3-term error-compensated (fp32-equivalent), fp32 accumulate; FLAME / rasteriser f32",
                                      "tf32": "encoder convs: tcgen05 TF32, fp32 accumulate; FLAME / rasteriser f32",
                                      "tf32-unfused": "encoder convs: tcgen05 TF32, fp32 accumulate; FLAME / rasteriser f32",
                                      "fp32": "f32 CUDA cores throughout"}[args.precision],
                       "global_batch": B * world,
                       "faces_per_gpu_per_step": B, "image": "224x224 RGB fp32", "parallelism": "frame-shard dp%d" % world,
                       "l2_policy": "inputs rotate over a set of batches > 126 MB L2 (160 MB)",
                       "timing": "%d timed steps in %d back-to-back windows, median window (CUDA events, max over ranks per window)" % (K, head["windows"]["n"]),
                       "execution": "CUDA graph replay, %d kernels per step, %d-lane software pipeline over consecutive steps" % (head["launches_per_step"], args.slots),
                       "host_affinity": affinity},
            "windows": head["windows"],
            "e2e": head["e2e"],
            "gpu_launches": head["launches_per_step"] * K,
            "clocks": head["clocks"], "roofline": head.get("roofline"), "cpu_baseline": head.get("cpu_baseline"),
            "parity": head.get("parity"), "kernel_shares": head.get("kernel_shares"),
        }
        for k in ("gather", "no_gather"):
            if k in head:
                line[k] = head[k]
        if full is not None:
            fc = {"workload": workload_name(True, args.full_batch), "value": full["value"], "unit": UNIT, "ms_per_step": full["ms_per_step"],
                  "global_batch": args.full_batch * world, "windows": full["windows"], "e2e": full["e2e"],
                  "gpu_launches": full["launches_per_step"] * K, "lanes": args.full_slots, "generator_dtype": "tf32 (fp32 accumulate)",
                  "roofline": full.get("roofline"), "kernel_shares": full.get("kernel_shares"), "clocks": full["clocks"], "parity": full.get("parity")}
            for k in ("gather", "no_gather"):
                if k in full:
                    fc[k] = full[k]
            line["full_cycle"] = fc
        if args.dump_outputs:
            import numpy as np
            os.makedirs(args.dump_outputs, exist_ok=True)
            for prefix, res in (("", head), ("full_cycle_", full)):
                for k, a in (res or {}).get("dump", {}).items():
                    np.save(os.path.join(args.dump_outputs, prefix + k + ".npy"), a)
        print(json.dumps(line), flush=True)
    if cx.dist is not None:
        cx.dist.destroy_process_group()


if __name__ == "__main__":
    main()
