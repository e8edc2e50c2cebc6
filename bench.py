# coding: utf-8
"""Benchmark of the autoregressive synthesis path (BASELINE.json metric: audio samples/sec).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--utts-per-gpu U]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one pass of the hot path over one batch: one ``incremental_forward`` of BASELINE
config 2 (MoL 10-mixture, 24 layers / 4 stacks, 512 residual / 512 gate / 256 skip channels,
80-dim mel conditioning, 22.05 kHz, T = 22050 samples) for ``U`` utterance(s) per GPU (default 1;
U=8 is BASELINE config 4's per-GPU share).  Utterances are independent, so N GPUs run N x U
utterances with no data-path collective ("weak" scaling); NCCL carries only the barrier, the
max-over-ranks time and the final waveform gather.

  value   : samples/s, whole job, conditioning already resident in HBM (kernel launches only)
  e2e     : the same through WaveNet.incremental_forward() from pinned HOST mel frames to a HOST
            waveform (H2D of the mel, upsample network, kernel, D2H of the result inside the timed
            region)
  roofline: weight-streaming bound.  One launch generates T samples and every sample needs all
            fp32 weights of the stack once (SURVEY.md 8(d): 98.72 MB/step for config 2), so
            algorithmic bytes/launch = T x weight_bytes_per_step; peak = measured HBM copy
            bandwidth from MEASURED_PEAKS.json.
  config4 : the same launch with 8 utterances per GPU (BASELINE config 4's per-GPU share): samples/s and the
            fraction of the 8-utterance weight roof (8 x peak / weight_bytes_per_step)
  cpu_baseline / --impl reference : the reference's own CPU incremental_forward (the package staged under
            oracle/_ref/ by __graft_entry__.build(); kind "reference") -- or, if it is absent, the oracle
            port of it (kind "port") -- timed on the host cores over a bounded number of samples, with the
            4 threads the reference ships (synthesis.py:37) and with all host cores.

--dump-outputs DIR writes what the last timed step of each path returned, as float32 .npy files: waveform.npy (the
device path, (N x U, T)), e2e_waveform.npy ((U, 1, T_up)) and config4_waveform.npy ((8, T)); the last two are rank 0's.
Inputs and noise seeds depend only on the arguments, so two builds can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

CFG2 = dict(out_channels=30, layers=24, stacks=4, residual_channels=512, gate_channels=512,
            skip_out_channels=256, cin_channels=80, cin_pad=2, gin_channels=-1, scalar_input=True,
            output_distribution="Logistic", dropout=0.0, upsample_conditional_features=True,
            upsample_params={"upsample_scales": [4, 4, 4, 4], "cin_channels": 80, "cin_pad": 2})
SAMPLE_RATE = 22050
T_FULL = 22050
HOP = 256


def build_model(seed=0):
    from wavenet_vocoder_b200 import WaveNet
    torch.manual_seed(seed)
    m = WaveNet(**CFG2).eval()
    with torch.no_grad():
        m.last_conv_layers[3].bias[20:] -= 3.0      # log-scales ~ -3: non-degenerate waveform (SURVEY 8(d))
    return m


def oracle_parts(model):
    from oracle import wavenet_oracle as orc
    cfg = orc.PathConfig(out_channels=30, layers=24, stacks=4, residual_channels=512, gate_channels=512,
                         skip_out_channels=256, kernel_size=3, cin_channels=80, gin_channels=-1,
                         scalar_input=True, output_distribution="Logistic")
    sd = {k: v.detach().cpu() for k, v in model.state_dict().items()}
    return orc, cfg, orc.weights_from_state_dict(cfg, sd)


REF_THREADS = 4       # the reference pins torch.set_num_threads(4) for synthesis (synthesis.py:37)


def load_reference():
    """The reference's own package, staged under oracle/_ref/ by __graft_entry__.build(); None if absent."""
    d = os.path.join(ROOT, "oracle", "_ref")
    if not os.path.isfile(os.path.join(d, "wavenet_vocoder", "wavenet.py")):
        return None
    if d not in sys.path:
        sys.path.insert(0, d)
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        import wavenet_vocoder
    return wavenet_vocoder


def reference_model(model):
    """The unmodified reference WaveNet with this model's weights (sample-rate conditioning: the timed region is
    the per-sample loop of wavenet.py:296-336, as for the port)."""
    ref = load_reference()
    if ref is None:
        return None
    import warnings
    kw = {k: v for k, v in CFG2.items() if k not in ("upsample_conditional_features", "upsample_params")}
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        m = ref.WaveNet(upsample_conditional_features=False, **kw).eval()
        sd = {k: v.detach().cpu() for k, v in model.state_dict().items() if not k.startswith("upsample_net.")}
        m.load_state_dict(sd)
        m.make_generation_fast_()
    return m


def time_cpu(model, n_samples, warm, threads, budget_s=25.0):
    """The reference algorithm on the host: (samples/s, seconds, samples, kind) after ``warm`` samples.  The number
    of timed samples is cut so that the run stays inside ``budget_s`` seconds (probed on the first samples)."""
    refm = reference_model(model)
    kind = "reference" if refm is not None else "port"
    if refm is None:
        orc, cfg, w = oracle_parts(model)
    torch.set_num_threads(threads)
    gen = torch.Generator().manual_seed(1)
    marks = {}

    def run(T, warm_):
        c = torch.randn(1, 80, T, generator=gen)

        def progress(it):
            for t in it:
                if t == warm_:
                    marks["t0"] = time.perf_counter()
                yield t
        torch.manual_seed(0)
        with torch.no_grad():
            if refm is not None:
                refm.incremental_forward(c=c, T=T, tqdm=progress, softmax=True, quantize=True, log_scale_min=-16.0)
            else:
                orc.incremental_forward(cfg, w, c=c, T=T, progress=progress)
        return time.perf_counter() - marks["t0"]

    probe = run(3 + 5, 3) / 5.0                          # seconds per sample (an oversubscribed all-core run can need 2 s)
    n = int(max(8, min(n_samples, budget_s / max(probe, 1e-6))))
    warm = int(min(warm, max(3, 0.25 * budget_s / max(probe, 1e-6))))
    dt = run(warm + n, warm)
    return n / dt, dt, n, kind


def cpu_rows(model, n_samples, warm, budget_s):
    """4-thread row (as the reference ships) and all-cores row."""
    ncpu = os.cpu_count() or 1
    rows = []
    for th in sorted({min(REF_THREADS, ncpu), ncpu}):
        v, dt, n, kind = time_cpu(model, n_samples, warm, th, budget_s=budget_s)
        rows.append({"threads": th, "value": v, "seconds": dt, "samples": n, "kind": kind})
    return rows


class ClockSampler:
    """nvidia-smi clocks/throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i] == "Active"})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def ncu_traffic(T, U):
    """DRAM bytes of one launch (dram__bytes_read.sum + dram__bytes_write.sum) from the committed
    `ncu --set full` capture of the same workload (profiles/r1_ncu_summary.json), else None."""
    try:
        name = "r2_ncu_summary.json" if os.path.exists(os.path.join(ROOT, "profiles", "r2_ncu_summary.json")) \
            else "r1_ncu_summary.json"
        with open(os.path.join(ROOT, "profiles", name)) as f:
            d = json.load(f)
        if d.get("utts_per_gpu") == U:
            # the full-set capture is taken at a shorter T (ncu replays the launch ~40 times); DRAM traffic
            # is proportional to the number of generated samples, so scale to this launch
            return d["dram_bytes_per_sample"] * T
    except Exception:
        pass
    return None


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


DUMP_BYTES = 64 << 20


def dump_outputs(d, arrays):
    """Write each tensor as d/<name>.npy in float32.  Each gets an equal share of DUMP_BYTES; a larger one is replaced
    by a fixed, seeded sample of its elements (flattened, in index order), the same positions on every run."""
    os.makedirs(d, exist_ok=True)
    share = (DUMP_BYTES // len(arrays) - 4096) // 4         # elements, 4 KB left for the .npy header
    for name, t in arrays.items():
        a = t.detach().float().cpu().numpy()
        if a.size > share:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, share, replace=False))]
        np.save(os.path.join(d, name + ".npy"), a)


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU incremental_forward on the host cores, rank 0 only."""
    if rank != 0:
        return
    model = build_model()
    per_step_budget = max(3.0, 100.0 / max(1, args.warmup + args.steps)) / 2.0      # two rows per step
    best = []
    rows_last = None
    for i in range(args.warmup + args.steps):
        rows = cpu_rows(model, args.ref_samples, 20, per_step_budget)
        if i >= args.warmup:
            best.append(max(rows, key=lambda r: r["value"]))
            rows_last = rows
    sps = sum(x["samples"] for x in best) / sum(x["seconds"] for x in best)
    top = best[-1]
    line = {
        "impl": "reference", "metric": "audio samples/sec (22.05 kHz MoL, 24-layer)", "value": sps,
        "unit": "samples/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * sum(x["seconds"] for x in best) / len(best), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "rtf": SAMPLE_RATE / sps,
        "config": {"workload": "BASELINE config 2: MoL-10 24L/4 stacks 512/512/256, 80-mel, B=1; "
                               "each step = %d samples of the same per-sample loop on the host CPU" % top["samples"]},
        "cpu_baseline": {"value": sps, "unit": "samples/s", "cores": top["threads"], "kind": top["kind"],
                         "host_cpus": os.cpu_count(), "rows": rows_last,
                         "sample": "%d samples after 20 warm-up samples per step, torch CPU fp32; rows: the 4 threads the "
                                   "reference ships (synthesis.py:37) and all host cores; value = the faster row"
                                   % top["samples"]},
        "e2e": {"value": sps, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--utts-per-gpu", type=int, default=1)
    ap.add_argument("--T", type=int, default=T_FULL)
    ap.add_argument("--ref-samples", type=int, default=1500)
    ap.add_argument("--cpu-samples", type=int, default=2000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-config4", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step of each path as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    W, K, U, T = max(args.warmup, 3), args.steps, args.utts_per_gpu, args.T

    model = build_model().to(dev)
    eng = model._get_engine()
    plan = eng.plan(U)
    # synthetic mel ~ N(0,1) (mean-var normalised features, compute-meanvar-stats.py:25-32)
    frames = -(-T // HOP) + 2 * CFG2["cin_pad"]
    T_up = (frames - 2 * CFG2["cin_pad"]) * HOP
    gen = torch.Generator().manual_seed(1000 + rank)
    mel_host = torch.randn(U, 80, frames, generator=gen).pin_memory()
    with torch.no_grad():
        c_dev = model.upsample_net(mel_host.to(dev))[:, :, :T].transpose(1, 2).contiguous()   # (U,T,80) resident
    flush = torch.empty(256 * 1024 * 1024 // 4, device=dev)       # > 126 MB L2

    def barrier():
        torch.cuda.synchronize(dev)
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def device_step(i):
        out, _ = eng.generate(B=U, T=T, c=c_dev, seed=i, sync=False)
        return out

    def e2e_step(i):
        y = model.incremental_forward(c=mel_host, T=T_up, seed=i)
        return y.cpu()

    results = {}
    for name, fn, Tn in (("device", device_step, T), ("e2e", e2e_step, T_up)):
        for i in range(W):
            fn(i)
            eng.sync()
        launches0 = eng.plan(U)["launches"]
        clk = ClockSampler(local)
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
        barrier()
        if rank == 0:
            clk.start()
        t_wall0 = time.perf_counter()
        for i in range(K):
            flush.zero_()                                           # flush L2 between timed iterations
            ev[i][0].record()
            out = fn(W + i)
            ev[i][1].record()
        barrier()
        t_wall = time.perf_counter() - t_wall0
        clocks = clk.stop() if rank == 0 else None
        ms = sum(a.elapsed_time(b) for a, b in ev)
        if name == "e2e":
            ms = t_wall * 1e3          # host-side copies are part of the e2e path: wall clock, flushes included
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        results[name] = dict(ms=float(t.item()), samples=Tn * U * world * K, clocks=clocks,
                             launches=eng.plan(U)["launches"] - launches0)
        if name == "device":
            wave_dev = out                       # (U, T) fp32 on this rank's GPU
        else:
            wave_e2e = out                       # (U, 1, T_up) fp32 on the host
    # BASELINE config 4's per-GPU share: 8 independent utterances in one launch
    cfg4 = wave4 = None
    if not args.no_config4:
        U4, K4 = 8, max(1, min(K, 3))
        c4 = c_dev[:1].expand(U4, -1, -1).contiguous() if U < U4 else c_dev[:U4]
        c4 = c4 + 0.01 * torch.randn(c4.shape, device=dev, generator=torch.Generator(device=dev).manual_seed(7 + rank))
        conc = hasattr(eng, "generate_concurrent") and eng.plan(1)["engine"] == 5 and os.environ.get("WN_CONCURRENT_TILES", "1") != "0"

        def step4(seed, sync):
            if conc:      # two tiles of 4 at the same time on two half-grid engines (engine.generate_concurrent)
                return eng.generate_concurrent(B=U4, T=T, c=c4, seed=seed, sync=sync)
            return eng.generate(B=U4, T=T, c=c4, seed=seed, sync=sync)[0]
        for i in range(2):
            step4(100 + i, True)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for i in range(K4):
            wave4 = step4(200 + i, False)
        e1.record()
        barrier()
        if conc:
            eng.sync_concurrent()
        t4 = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        if dist is not None:
            dist.all_reduce(t4, op=dist.ReduceOp.MAX)
        sps4 = U4 * T * K4 * world / (float(t4.item()) * 1e-3)
        peak4, _ = measured_peak()
        roof4 = U4 * peak4 * 1e9 / plan["weight_bytes_per_step"]          # samples/s per GPU if the weights stream at peak
        cfg4 = {"workload": "BASELINE config 4 share: %d utterances per GPU, T=%d, %s" % (
                    U4, T, "two tiles of 4 at the same time on two half-grid engines" if conc else "tiles of <= %d, one after the other" % eng.plan(U4)["batch_tile"]),
                "value": sps4, "unit": "samples/s", "per_gpu": sps4 / world, "steps": K4,
                "ms_per_step": float(t4.item()) / K4, "batch_tile": eng.plan(U4)["batch_tile"],
                "frac_of_weight_roof": (sps4 / world) / roof4, "weight_roof_samples_per_s_per_gpu": roof4}
    if dist is not None:
        # the only data-path collective: gather the waveforms of the last step on rank 0
        gathered = [torch.empty_like(wave_dev) for _ in range(world)] if rank == 0 else None
        dist.gather(wave_dev, gathered, dst=0)
        torch.cuda.synchronize(dev)

    if rank == 0:
        if args.dump_outputs:
            outs = {"waveform": torch.cat(gathered) if dist is not None else wave_dev, "e2e_waveform": wave_e2e}
            if wave4 is not None:
                outs["config4_waveform"] = wave4
            dump_outputs(args.dump_outputs, outs)
        d, e = results["device"], results["e2e"]
        sps = d["samples"] / (d["ms"] * 1e-3)
        e_sps = e["samples"] / (e["ms"] * 1e-3)
        peak, peak_src = measured_peak()
        steps_per_s_per_gpu = (T * K) / (d["ms"] * 1e-3)             # generated time steps per second on one GPU
        achieved = steps_per_s_per_gpu * plan["weight_bytes_per_step"] / 1e9
        line = {
            "metric": "audio samples/sec (22.05 kHz MoL, 24-layer)", "value": sps, "unit": "samples/s",
            "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": d["ms"] / K, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "rtf": SAMPLE_RATE * U * world / sps, "x_realtime_per_utterance": sps / (U * world) / SAMPLE_RATE,
            "config": {"workload": "BASELINE config 2: MoL-10, 24 layers / 4 stacks, 512/512/256 ch, 80-mel local "
                                   "conditioning, T=%d, %d utterance(s) per GPU" % (T, U),
                       "global_batch": U * world, "T": T, "parallelism": "utterance-sharded x%d" % world,
                       "l2": "256 MiB write between timed iterations; weights (98.7 MB) re-read every sample",
                       "plan": {k: plan[k] for k in ("num_ctas", "batch_tile", "resident_blobs", "ring_slots",
                                                     "exchange_copies", "exchanges_per_step", "smem_bytes",
                                                     "rings_in_smem", "streamed_bytes_per_step", "num_clusters",
                                                     "cluster_size", "engine")}},
            "clocks": d["clocks"],
            "e2e": {"value": e_sps, "unit": "samples/s",
                    "h2d_bytes_per_step": int(mel_host.numel() * 4), "d2h_bytes_per_step": int(U * T_up * 4),
                    "T": T_up, "api": "WaveNet.incremental_forward(c=host mel) -> .cpu()", "clocks": e["clocks"]},
            "gpu_launches": d["launches"],
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": ncu_traffic(T, U), "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": T * plan["weight_bytes_per_step"],
                         "flops_per_sample": plan["flops_per_sample"],
                         "fp32_tflops_achieved": sps * plan["flops_per_sample"] / 1e12},
        }
        if cfg4 is not None:
            line["config4"] = cfg4
        if world == 1 and not args.no_cpu_baseline:
            rows = cpu_rows(model.cpu(), args.cpu_samples, 100, 12.0)
            top = max(rows, key=lambda r: r["value"])
            line["cpu_baseline"] = {"value": top["value"], "unit": "samples/s", "cores": top["threads"],
                                    "kind": top["kind"], "host_cpus": os.cpu_count(), "rows": rows,
                                    "sample": "%d samples after 100 warm-up samples of the same config-2 loop (the "
                                              "reference's CPU incremental_forward, torch fp32); rows: 4 threads as the "
                                              "reference ships (synthesis.py:37) and all host cores; value = the faster"
                                              % top["samples"]}
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
