#!/usr/bin/env python
"""
bench.py - backbones/sec of the reverse-diffusion sampler (BASELINE.json metric).

    python bench.py --gpus 1 --steps K --warmup W            # our arm (CUDA, sm_100a)
    python bench.py --impl reference --gpus 1 ...             # the reference's CPU path (oracle port)
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...   # N > 1

One "step" = one pass of the hot path over one batch: the full T-step p_sample loop (T = 1000,
cosine schedule) on 512 chains of lengths 50..127 (BASELINE config 2, "foldingdiff_cath BERT,
batch=512, len 50-128, T=1000") with synthetic weights of the production architecture (the real
checkpoint is not available offline) and synthetic wrapped-Gaussian noise.

  value  whole-job backbones/s with the initial noise already resident in HBM
  e2e    the same through the public API with HOST buffers: sampling.p_sample_loop(host noise) ->
         host tensor; H2D of the noise and D2H of the result inside the timed region
  roofline / kernels  per-kernel device times measured live with CUDA events (fd_profile_*)
  cpu_baseline  the oracle port (torch CPU fp32 restatement + the reference's loop arithmetic)
         timed on this box's host cores on a bounded sample, extrapolated to T steps
Multi-GPU: chains are independent -> each rank runs 512 chains (weak scaling), no collective inside
the loop, one NCCL all-gather of the final angles per pass (inside the timed region).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from foldingdiff_b200 import beta_schedules, datasets, synthetic  # noqa: E402

SEED = 7344
PEAKS_FILE = os.path.join(ROOT, "MEASURED_PEAKS.json")
FALLBACK_HBM_GBS = 6650.0      # /opt/skills/guides/B200_PROFILING.md fallback
FALLBACK_PEAK_TFLOPS = 1590.0  # /opt/skills/guides/B200_PROFILING.md fallback (burst)


def source_sha():
    """Hash of the CUDA sources (tools/summarize_ncu.py computes the same one when it summarises an ncu capture)."""
    import hashlib
    csrc = os.path.join(ROOT, "foldingdiff_b200", "csrc")
    h = hashlib.sha256()
    for name in sorted(os.listdir(csrc)):
        if name.endswith((".cu", ".cuh", ".hpp")):
            h.update(name.encode())
            h.update(open(os.path.join(csrc, name), "rb").read())
    return h.hexdigest()[:16]


def load_ncu_profile():
    """
    The newest committed per-step ncu summary (profiles/rNN_step_ncu.json, written by tools/summarize_ncu.py step from a
    capture of tools/gpu_ncu_step.sh): DRAM bytes and tensor-pipe activity per kernel category.  ncu figures cannot be
    taken inside a timed run, so they are annotations - but self-describing ones: the file names the source hash it was
    captured from, and a mismatch with the sources of THIS run is reported as `stale` instead of passing silently.
    """
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_step_ncu.json")))
    if not files:
        return None
    with open(files[-1]) as f:
        prof = json.load(f)
    prof["file"] = os.path.relpath(files[-1], ROOT)
    prof["stale"] = prof.get("source_sha") != source_sha()
    return prof


def parse_args():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=2)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", choices=["ours", "reference"], default="ours")
    p.add_argument("--workload", choices=["config2", "config3", "config5"], default="config2")
    p.add_argument("--timesteps", type=int, default=1000)
    p.add_argument("--batch", type=int, default=None, help="chains per GPU (default: the workload's)")
    p.add_argument("--gemm", choices=["tc3x", "fp32", "tc1x"], default=os.environ.get("FOLDINGDIFF_B200_GEMM", "tc3x"))
    p.add_argument("--e2e-history", choices=["full", "final"], default="full")
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--cpu-chains", type=int, default=64)
    p.add_argument("--cpu-steps", type=int, default=3)
    p.add_argument("--profile-steps", type=int, default=20, help="reverse steps of the CUDA-event kernel profile")
    p.add_argument("--no-extra-workloads", action="store_true", help="skip the short config 3 / config 5 sub-lines")
    p.add_argument("--no-parity", action="store_true", help="skip the parity block")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="after the timed steps, write what the timed path returned in its last step as DIR/<name>.npy")
    args = p.parse_args()
    if args.steps < 1 or args.warmup < 0:
        p.error("--steps must be at least 1 and --warmup at least 0")
    return args


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(dirname, arrays):
    """
    Write each array as DIR/<name>.npy in float32, so that two builds run with the same arguments (hence the same
    seeded inputs) can be compared output for output.  Where the arrays together exceed 64 MB, each keeps a fixed,
    seeded sample of its rows (leading axis), the same for every build.
    """
    os.makedirs(dirname, exist_ok=True)
    arrays = {k: np.ascontiguousarray(v, dtype=np.float32) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    for name, a in arrays.items():
        if total > DUMP_LIMIT_BYTES:
            keep = max(1, a.shape[0] * DUMP_LIMIT_BYTES // total)
            a = a[np.sort(np.random.default_rng(SEED).choice(a.shape[0], keep, replace=False))]
        np.save(os.path.join(dirname, f"{name}.npy"), a)


def workload(args):
    """-> (lengths per GPU, n_pad, start_t, wrap_all, name)"""
    T = args.timesteps
    if args.workload == "config2":
        B = args.batch or 512
        lengths = synthetic.sweep_lengths(B)
        return lengths, max(lengths), T, False, f"foldingdiff_cath BERT (synthetic weights), batch={B}/GPU, len 50-127, T={T}"
    if args.workload == "config3":
        B = args.batch or 4096
        return [128] * B, 128, T, False, f"foldingdiff_cath (synthetic weights), batch={B}/GPU, len=128, T={T}"
    B = args.batch or 512
    return [128] * B, 128, min(250, T), True, f"partial_noise_reconstruct (synthetic weights/inputs), batch={B}/GPU, len=128, from t={min(250, T)}"


def initial_noise(B, n_pad, T):
    d = datasets.NoisedAnglesDataset(datasets.AnglesEmptyDataset("canonical-full-angles", pad=128),
                                     timesteps=T, beta_schedule="cosine")
    torch.manual_seed(SEED)
    return d, d.sample_noise(torch.zeros(B, 128, 6))[:, :n_pad].contiguous()


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows, self.proc, self.index = [], None, index

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        return self

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *exc):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# CPU baseline / reference arm: the oracle port on the host cores
# ------------------------------------------------------------------------------------------------
_CPU_MODEL = None
_REF = None  # (sampling, beta_schedules, utils) of the reference installed under baseline/_ref, or False


def _reference():
    """The UNMODIFIED reference from baseline/_ref (baseline/reference_arm.py), or False where it is not installed."""
    global _REF
    if _REF is None:
        try:
            sys.path.insert(0, os.path.join(ROOT, "baseline"))
            import reference_arm
            _REF = reference_arm.load_reference()[:3] + (reference_arm,) if reference_arm.available() else False
        except Exception as e:  # noqa: BLE001
            print(f"[bench] baseline/_ref not usable ({e}); timing the oracle port instead", file=sys.stderr)
            _REF = False
    return _REF


def cpu_kind():
    return "reference" if _reference() else "port"


def _cpu_model():
    global _CPU_MODEL
    if _CPU_MODEL is None:
        sd = synthetic.synthetic_state_dict(synthetic.PRODUCTION, seed=0)
        ref = _reference()
        if ref:
            _CPU_MODEL = ref[3].build_model(sd, synthetic.PRODUCTION)
        else:
            from oracle import forward as ofwd  # the one place bench.py may execute oracle/
            _CPU_MODEL = ofwd.OracleModel(sd, ofwd.OracleConfig(**synthetic.PRODUCTION), [True] * 6).eval()
    return _CPU_MODEL


_CPU_TRACE = None  # states of the last reference-arm run: {"x": [x_init, x_1, ...], "t": [...], "seed": int, "sub": lengths}


def _cpu_steps(sub, n_pad, T, start_t, steps, threads, trace=False):
    """
    seconds per reverse step of the reference's CPU path on `threads` host threads (1 untimed warm-up step).
    With baseline/_ref: the stock `sampling.p_sample` + per-column `utils.modulo_with_wrapped_range` + `.cpu()` of the
    reference's loop body (sampling.py:111-131) around the reference-assembled model; otherwise the oracle port.
    """
    torch.set_num_threads(threads)
    model = _cpu_model()
    ref = _reference()
    g = torch.Generator().manual_seed(SEED)
    global _CPU_TRACE
    if ref:
        sampling, beta_schedules, utils = ref[:3]
        betas = beta_schedules.get_variance_schedule("cosine", T)
        x = torch.randn(len(sub), n_pad, 6, generator=g)
        if trace:  # the reference draws its step normals from the global CPU generator: seed it so the GPU can replay them
            torch.manual_seed(SEED + 1)
            _CPU_TRACE = {"x": [x.clone()], "t": [], "seed": SEED + 1, "sub": list(sub), "n_pad": n_pad}

        def step(img, i):
            with torch.no_grad():
                img = sampling.p_sample(model=model, x=img, t=torch.full((len(sub),), i, dtype=torch.long), seq_lens=sub,
                                        t_index=i, betas=betas)
            for j in range(img.shape[2]):
                img[:, :, j] = utils.modulo_with_wrapped_range(img[:, :, j], range_min=-torch.pi, range_max=torch.pi)
            img.cpu()
            return img
        x = step(x, start_t - 1)
        if trace:
            _CPU_TRACE["x"].append(x.clone()); _CPU_TRACE["t"].append(start_t - 1)
        dt = 0.0
        for k in range(steps):  # per-step cost does not depend on t
            t0 = time.perf_counter()
            x = step(x, start_t - 2 - k)
            dt += time.perf_counter() - t0
            if trace:
                _CPU_TRACE["x"].append(x.clone()); _CPU_TRACE["t"].append(start_t - 2 - k)
        return dt / steps
    from oracle import loop as oloop
    from oracle import schedules as osched
    betas = osched.betas_for("cosine", T)
    x = oloop.wrap(torch.randn(len(sub), n_pad, 6, generator=g))
    if trace:
        torch.manual_seed(SEED + 1)
        _CPU_TRACE = {"x": [x.clone()], "t": [], "seed": SEED + 1, "sub": list(sub), "n_pad": n_pad}
    x = oloop.wrap(oloop.p_sample(model, x, torch.full((len(sub),), start_t - 1, dtype=torch.long), sub, betas))
    if trace:
        _CPU_TRACE["x"].append(x.clone()); _CPU_TRACE["t"].append(start_t - 1)
    dt = 0.0
    for k in range(steps):  # per-step cost does not depend on t
        t0 = time.perf_counter()
        x = oloop.wrap(oloop.p_sample(model, x, torch.full((len(sub),), start_t - 2 - k, dtype=torch.long), sub, betas))
        dt += time.perf_counter() - t0
        if trace:
            _CPU_TRACE["x"].append(x.clone()); _CPU_TRACE["t"].append(start_t - 2 - k)
    return dt / steps


_BEST_THREADS = None


def cpu_reference_rate(lengths, n_pad, T, chains, steps, start_t, wrap_all):
    """
    backbones/s of the reference's CPU path from a bounded sample: `chains` chains taken evenly from the
    workload's length mix, `steps` reverse steps timed after one warm-up, extrapolated to the full loop.
    torch's CPU kernels do not scale to every core count, so the thread count is chosen by a one-step
    probe over {all cores, 64, 32, 16} and the best one is used ("all the host threads it can use").
    """
    global _BEST_THREADS, _REF, _CPU_MODEL
    cores = os.cpu_count() or 1
    stride = max(1, len(lengths) // chains)
    sub = [lengths[i] for i in range(0, len(lengths), stride)][:chains]
    if _reference():
        try:  # a reference install that imports but does not run must not cost the measurement: fall back to the port
            _cpu_steps(sub[:2], n_pad, T, start_t, 1, min(cores, 16))
        except Exception as e:  # noqa: BLE001
            print(f"[bench] reference arm failed ({type(e).__name__}: {e}); timing the oracle port instead", file=sys.stderr)
            _REF, _CPU_MODEL = False, None
    if _BEST_THREADS is None:
        cands = sorted({c for c in (cores, 64, 32, 16) if c <= cores}, reverse=True)
        probe = {c: _cpu_steps(sub, n_pad, T, start_t, 1, c) for c in cands}
        _BEST_THREADS = min(probe, key=probe.get)
    dt = _cpu_steps(sub, n_pad, T, start_t, steps, _BEST_THREADS, trace=True)
    rate = len(sub) / (dt * start_t)
    what = ("stock sampling.p_sample + wrap of the reference installed in baseline/_ref around its own GaussianFourierProjection / "
            "BertEmbeddings / AnglesPredictor and the installed transformers' relative_key attention + BERT blocks (4.11.3 is "
            "not installable); " if _reference() else "oracle port of the reference loop and forward (baseline/_ref absent); ")
    sample = (what + f"{len(sub)} chains (every {stride}-th of the workload's lengths, sum len {sum(sub)}), {steps} reverse steps "
              f"timed after 1 warm-up at {dt:.3f} s/step on {_BEST_THREADS} threads (best of a 1-step probe; box has {cores} "
              f"cores), extrapolated x{start_t} steps")
    return rate, _BEST_THREADS, sample, dt


# ------------------------------------------------------------------------------------------------
def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    lengths, n_pad, start_t, wrap_all, wl_name = workload(args)
    T = args.timesteps
    B = len(lengths)
    flops_step = synthetic.algorithmic_flops(synthetic.PRODUCTION, lengths)

    if args.impl == "reference":
        if rank != 0:
            return 0
        # each bench "step" of this arm is one bounded sample (cpu_steps reverse steps over cpu_chains chains of the
        # workload's length mix, extrapolated to the full loop); W warm-up samples, then K timed ones
        reps, dts = [], []
        sample, cores = "", os.cpu_count() or 1
        for i in range(args.warmup + args.steps):
            r, cores, sample, d = cpu_reference_rate(lengths, n_pad, T, args.cpu_chains, max(1, args.cpu_steps), start_t, wrap_all)
            if i >= args.warmup:
                reps.append(r)
                dts.append(d)
        value = float(np.mean(reps))
        dt = float(np.mean(dts))
        if args.dump_outputs:  # the state the last timed sample's reverse steps ended in
            dump_outputs(args.dump_outputs, {"angles": _CPU_TRACE["x"][-1].numpy()})
        line = {
            "impl": "reference", "metric": "backbones/sec", "value": value, "unit": "backbones/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1000.0 * dt * max(1, args.cpu_steps), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": wl_name, "timesteps": T,
                       "note": ("CPU path: the unmodified reference installed in baseline/_ref - its own loop (sampling.p_sample), "
                                "schedules, wrap and model sub-modules; encoder layers from the installed transformers' modules "
                                "because transformers==4.11.3 is not installable (baseline/reference_arm.py)") if _reference() else
                               ("CPU path: fp32 torch restatement of the reference forward (HF 4.11.3 encoder not "
                                "installable) + the reference's loop arithmetic; baseline/_ref absent")},
            "cpu_baseline": {"value": value, "unit": "backbones/s", "cores": cores, "kind": cpu_kind(), "sample": sample},
            "e2e": {"value": value, "unit": "backbones/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
        }
        print(json.dumps(line))
        return 0

    # ---------------------------------------------------------------------------------------------
    assert torch.cuda.is_available(), "bench.py (impl=ours) needs a CUDA device; there is no CPU fallback"
    from foldingdiff_b200 import distributed as fdist
    from foldingdiff_b200 import modelling, sampling
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import torch.distributed as dist
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"  # keep NCCL's version banner off stdout: one JSON line only
        dist.init_process_group("nccl", device_id=dev)

    cfg = modelling.BertConfig(**synthetic.PRODUCTION)
    model = modelling.BertForDiffusionBase(cfg, ft_is_angular=[True] * 6, gemm=args.gemm)
    model.load_state_dict(synthetic.synthetic_state_dict(synthetic.PRODUCTION, seed=0))
    model = model.to(dev)
    eng = model.native_engine()
    dset, noise_host = initial_noise(B, n_pad, T)
    noise_host = noise_host.pin_memory()
    betas = dset.alpha_beta_terms["betas"]
    wrap = [True] * 6
    eng.set_schedule(betas, T)
    eng.set_batch(lengths, n_pad)
    noise_dev = noise_host.to(dev)
    gather = [torch.empty((B, n_pad, 6), device=dev) for _ in range(world)] if world > 1 else None

    last = [None]  # the finished angles of the latest pass

    def one_pass_device():
        x = noise_dev.clone()
        sampling._run_steps(eng, x, start_t, wrap, None)
        if world > 1:
            dist.all_gather(gather, x)  # the job's only collective: finished angles
        last[0] = x
        return x

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, reps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    for _ in range(args.warmup):
        one_pass_device()
    launches0 = eng.launch_count()
    with ClockSampler(local_rank) as clk:
        ms = timed(one_pass_device, args.steps)
    launches = eng.launch_count() - launches0
    clocks = clk.summary()
    ms_per_step = ms / args.steps
    value = world * B / (ms_per_step / 1000.0)
    if args.dump_outputs and rank == 0:  # the finished angles of the last timed pass (all ranks' chains after the gather)
        dump_outputs(args.dump_outputs, {"angles": (torch.cat(gather) if world > 1 else last[0]).cpu().numpy()})

    # ---- e2e: host noise in, host result out, through the public API ------------------------------
    e2e = None
    if not args.no_e2e:
        hist_mode = args.e2e_history

        def one_pass_e2e():
            if wrap_all:
                out = sampling.denoise_from(model, noise_host, lengths, start_t, betas).cpu()
            else:
                out = sampling.p_sample_loop(model, lengths, noise_host, T, betas, is_angle=wrap, history=hist_mode)
            return out

        one_pass_e2e()  # allocator warm-up for the history buffers
        ms_e = timed(one_pass_e2e, args.steps) / args.steps
        steps_out = start_t if (hist_mode == "full" and not wrap_all) else 1
        e2e = {"value": world * B / (ms_e / 1000.0), "unit": "backbones/s",
               "h2d_bytes_per_step": int(noise_host.numel() * 4),
               "d2h_bytes_per_step": int(steps_out * B * n_pad * 6 * 4),
               "ms_per_step": ms_e, "api": "sampling.p_sample_loop(host noise) -> host tensor, history=" + hist_mode}

    # ---- per-kernel device times (CUDA events on the launch stream), rank 0 only -------------------
    roofline, kernels = None, None
    if rank == 0:
        nprof = min(args.profile_steps, start_t)
        x = noise_dev.clone()
        z = torch.randn((nprof, B, n_pad, 6), device=dev)
        torch.cuda.synchronize()
        eng.profile_begin()
        eng.p_sample_steps(x, start_t, start_t - nprof, z, None, wrap)
        prof = eng.profile_end()
        total = sum(v[0] for v in prof.values()) or 1.0
        kernels = {k: {"ms_per_reverse_step": v[0] / nprof, "launches_per_reverse_step": v[1] / nprof,
                       "share": v[0] / total} for k, v in prof.items() if v[1]}
        n = np.asarray(lengths, dtype=np.float64)
        H, I, L = cfg.hidden_size, cfg.intermediate_size, cfg.num_hidden_layers
        gemm_flops = {"gemm_qkv": L * 6 * H * H * n.sum(), "gemm_attn_out": L * 2 * H * H * n.sum(),
                      "gemm_ffn1": L * 2 * H * I * n.sum(), "gemm_ffn2": L * 2 * H * I * n.sum(),
                      "gemm_head": 2 * H * H * n.sum()}
        att_flops = L * 6 * H * (n * n).sum()
        peak_tf, peak_src = FALLBACK_PEAK_TFLOPS, "fallback (B200_PROFILING.md)"
        if os.path.isfile(PEAKS_FILE):
            with open(PEAKS_FILE) as f:
                pk = json.load(f)
            peak_tf, peak_src = float(pk.get("bf16_tflops_sustained", pk.get("bf16_tflops"))), "measured (MEASURED_PEAKS.json bf16_tflops_sustained: kernel timed inside a long step)"
        gemm_ms = sum(prof[k][0] for k in gemm_flops) / nprof
        gemm_tf = sum(gemm_flops.values()) / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else 0.0
        att_ms = prof["attention"][0] / nprof
        att_tf = att_flops / (att_ms * 1e-3) / 1e12 if att_ms > 0 else 0.0
        dominant = "projection GEMMs (tc_gemm_kernel / sgemm_tn_kernel)" if gemm_ms >= att_ms else "relative-key attention (attention_tc_kernel / attention_simt_kernel)"
        dom_tf = gemm_tf if gemm_ms >= att_ms else att_tf
        hbm_gbs, hbm_src = FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"
        if os.path.isfile(PEAKS_FILE):
            hbm_gbs, hbm_src = float(pk.get("hbm_gbs", FALLBACK_HBM_GBS)), "measured (MEASURED_PEAKS.json hbm_gbs)"
        ncu = load_ncu_profile() if (args.workload == "config2" and args.gemm == "tc3x") else None
        ncu_k = (ncu or {}).get("kernels", {})
        gemm_cats = [k for k in ("gemm_qkv", "gemm_attn_out", "gemm_ffn1", "gemm_ffn2") if k in ncu_k]
        traffic = None
        if ncu and gemm_cats and gemm_ms >= att_ms:
            traffic = float(np.mean([ncu_k[k]["dram_bytes_per_launch"] for k in gemm_cats]))
        # per-kernel entries: the tensor-bound kernels against the tensor peak, the streaming kernels against HBM
        per_kernel = {}
        for k, fl in gemm_flops.items():
            if prof[k][1]:
                tf = fl / (prof[k][0] / nprof * 1e-3) / 1e12
                per_kernel[k] = {"bound": "tensor", "achieved_tflops": tf, "frac": tf / peak_tf,
                                 "tensor_pipe_active_pct_ncu": ncu_k.get(k, {}).get("tensor_pipe_active_pct"),
                                 "dram_bytes_per_launch_ncu": ncu_k.get(k, {}).get("dram_bytes_per_launch")}
        per_kernel["attention"] = {"bound": "tensor", "achieved_tflops": att_tf, "frac": att_tf / peak_tf,
                                   "tensor_pipe_active_pct_ncu": ncu_k.get("attention", {}).get("tensor_pipe_active_pct"),
                                   "dram_bytes_per_launch_ncu": ncu_k.get("attention", {}).get("dram_bytes_per_launch")}
        rows_total = float(n.sum())
        stream_bytes = {  # algorithmic bytes per launch of the HBM-bound kernels (packed rows x hidden)
            "embed": rows_total * (6 * 4 + H * (4 + 4)),                 # x in; h fp32 + hi/lo planes out
            "tail_posterior": rows_total * (H * 4 + 6 * 4 * 3),          # u in; x in/out, z in
            "layernorm": rows_total * H * (4 + 4 + 4 + 4),               # fp32 mode only: in + resid, out + planes
        }
        for k, by in stream_bytes.items():
            if k in prof and prof[k][1]:
                gbs = by / (prof[k][0] / prof[k][1] * 1e-3) / 1e9
                per_kernel[k] = {"bound": "hbm", "achieved_gbs": gbs, "frac": gbs / hbm_gbs, "algorithmic_bytes_per_launch": by}
        roofline = {"bound": "tensor", "kernel": dominant, "achieved": dom_tf, "peak": peak_tf, "unit": "TFLOP/s",
                    "frac": dom_tf / peak_tf, "peak_source": peak_src, "hbm_peak_gbs": hbm_gbs, "hbm_peak_source": hbm_src,
                    "traffic": traffic,
                    "traffic_note": "ncu dram__bytes_read + dram__bytes_write per GEMM launch, mean over the four projections of a layer",
                    "ncu_profile": None if not ncu else {"file": ncu["file"], "source_sha": ncu.get("source_sha"), "stale": ncu["stale"],
                                                          "head": ncu.get("head"),
                                                          "dram_bytes_per_reverse_step": ncu.get("dram_bytes_per_reverse_step"),
                                                          "tensor_pipe_active_pct_time_weighted": ncu.get("tensor_pipe_active_pct_time_weighted")},
                    "per_kernel": per_kernel,
                    "gemm_tflops_algorithmic": gemm_tf, "attention_tflops_algorithmic": att_tf,
                    "whole_step_tflops_algorithmic": flops_step * start_t / (ms_per_step * 1e-3) / 1e12,
                    "note": "algorithmic FLOPs (valid tokens, 2 flop/MAC, SURVEY 8d) / CUDA-event kernel time; "
                            "the 3-pass split issues 3x these MMAs; ncu figures come from the committed capture named in "
                            "ncu_profile (stale = the CUDA sources have changed since it was taken). Since round 2 the "
                            "projection launches ALSO do the two LayerNorms of every layer and their residual traffic (folded "
                            "into the epilogues, 24 LayerNorm launches per reverse step removed): on that basis round 1 was "
                            "GEMM 3.65 ms + LayerNorm 1.10 ms = 4.75 ms per reverse step = 268 TFLOP/s algorithmic = 0.186 of the "
                            "same peak (BENCH_r01: 0.242 for the GEMM launches alone)"}

    # ---- section 8f rank-1 row: batched NeRF (angles -> backbone coordinates), reported beside the headline ----
    nerf_line = None
    if rank == 0:
        from foldingdiff_b200 import nerf as fnerf
        names = ["phi", "psi", "omega", "tau", "CA:C:1N", "C:1N:1CA"]
        ang = noise_dev.clone()
        ang[..., 3:] = ang[..., 3:].abs() * 0.2 + 1.7
        for _ in range(3):
            fnerf.build_backbone(ang, lengths, names)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 20
        e0.record()
        for _ in range(reps):
            xyz = fnerf.build_backbone(ang, lengths, names)
        e1.record()
        torch.cuda.synchronize()
        gpu_rate = reps * B / (e0.elapsed_time(e1) / 1000.0)
        nerf_line = {"gpu_structures_per_s": gpu_rate, "atoms_per_structure": "3 x length (N, CA, C)",
                     "api": "foldingdiff_b200.nerf.build_backbone (fd_nerf_build)", "chains": B}
        if world == 1 and not args.no_cpu_baseline:
            from oracle import nerf as onerf  # CPU baseline leg: the reference's per-chain Python loop, restated
            host = ang[:8].cpu().numpy()
            t0 = time.perf_counter()
            for i in range(8):
                onerf.build_chain(host[i, : lengths[i]], names)
            nerf_line["cpu_structures_per_s_1core"] = 8 / (time.perf_counter() - t0)
            nerf_line["cpu_sample"] = "8 chains, oracle restatement of nerf.NERFBuilder (single core, as one pool worker)"

    # ---- section 8f rank-2 row: output writers (csv.gz + PDB per chain), native batch call vs the reference's way ----
    if rank == 0 and nerf_line is not None:
        import shutil
        import tempfile
        from foldingdiff_b200 import writers as fwriters
        tmp = tempfile.mkdtemp(prefix="fd_writers_")
        try:
            ang_h, xyz_h = ang.cpu().numpy(), xyz.cpu().numpy()
            t0 = time.perf_counter()
            fwriters.write_batch(lengths, angles=ang_h, feature_names=names, csv_paths=[f"{tmp}/g{i}.csv.gz" for i in range(B)],
                                 coords=xyz_h, pdb_paths=[f"{tmp}/g{i}.pdb" for i in range(B)])
            dt = time.perf_counter() - t0
            wline = {"native_chains_per_s": B / dt, "files_per_chain": 2, "chains": B,
                     "api": "foldingdiff_b200.writers.write_batch (fd_write_batch)", "host_threads": min(32, os.cpu_count() or 1)}
            if world == 1 and not args.no_cpu_baseline:
                import pandas as pd
                from oracle import writers as owriters  # CPU baseline leg: DataFrame.to_csv + the PDB text restatement
                t0 = time.perf_counter()
                for i in range(16):
                    pd.DataFrame(ang_h[i, : lengths[i]], columns=names).to_csv(f"{tmp}/ref{i}.csv.gz")
                    with open(f"{tmp}/ref{i}.pdb", "w") as f:
                        f.write(owriters.backbone_pdb_text(xyz_h[i, : 3 * lengths[i]]))
                wline["cpu_chains_per_s_1core"] = 16 / (time.perf_counter() - t0)
                wline["cpu_sample"] = "16 chains, DataFrame.to_csv(.csv.gz) + Python PDB text (single core, as one pool worker)"
        finally:
            shutil.rmtree(tmp, ignore_errors=True)
    else:
        wline = None

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        rate, cores, sample, _ = cpu_reference_rate(lengths, n_pad, T, args.cpu_chains, args.cpu_steps, start_t, wrap_all)
        cpu_baseline = {"value": rate, "unit": "backbones/s", "cores": cores, "kind": cpu_kind(), "sample": sample}

    # ---- parity block: what the number above was computed WITH, checked in the same run --------------------------
    parity = None
    if rank == 0 and not args.no_parity:
        parity = {"tolerance_max_abs": 1e-4, "metric": "circular max-abs over valid residues, fp32 angles"}
        # (1) the benchmarked arithmetic against the library's fp32 CUDA-core arithmetic: whole batch, 8 reverse steps
        #     from the middle of the schedule (the first step of a cosine chain has a x100 gain: reported separately)
        if args.gemm != "fp32":
            def short_chain(gemm, t_hi, nst, zz):
                model.set_gemm(gemm)
                xx = noise_dev.clone()
                eng.p_sample_steps(xx, t_hi, t_hi - nst, zz, None, wrap)
                torch.cuda.synchronize()
                return xx
            gz = torch.Generator(device=dev).manual_seed(5)
            zz = torch.randn((8, B, n_pad, 6), device=dev, generator=gz)
            valid = (torch.arange(n_pad, device=dev)[None, :] < torch.as_tensor(lengths, device=dev)[:, None])[..., None]
            def cdiff(a, b):
                d = (a - b).abs()
                return float((torch.minimum(d, 2 * np.pi - d) * valid).max())
            t_mid = max(8, min(start_t, T // 2))
            mid = cdiff(short_chain(args.gemm, t_mid, 8, zz), short_chain("fp32", t_mid, 8, zz))
            first = cdiff(short_chain(args.gemm, start_t, 1, zz), short_chain("fp32", start_t, 1, zz))
            model.set_gemm(args.gemm)
            parity["vs_fp32_cuda_cores"] = {"chains": B, "steps": 8, "from_t": t_mid, "max_abs": mid,
                                            "first_step_from_t_start_max_abs": first, "ok": bool(mid < 1e-4)}
        # (2) against the reference arm's own states (cpu_baseline leg: the stock loop on the host): every CPU step is
        #     replayed on the GPU from the CPU's x_t with the CPU's normals (teacher-forced, SURVEY 8c protocol (2))
        if cpu_baseline is not None and _CPU_TRACE is not None and len(_CPU_TRACE["t"]) >= 1:
            tr = _CPU_TRACE
            torch.manual_seed(tr["seed"])
            eng.set_batch(tr["sub"], tr["n_pad"])
            errs = []
            for k, t in enumerate(tr["t"]):
                zc = torch.randn_like(tr["x"][k]) if t > 0 else torch.zeros_like(tr["x"][k])  # the reference's own draw order
                xg = tr["x"][k].to(dev).contiguous().clone()
                eng.p_sample_steps(xg, t + 1, t, zc.to(dev)[None].contiguous(), None, wrap)
                d = (xg.cpu() - tr["x"][k + 1]).abs()
                d = torch.minimum(d, 2 * np.pi - d)
                errs.append(max(float(d[i, :l].max()) for i, l in enumerate(tr["sub"])))
            eng.set_batch(lengths, n_pad)
            later = errs[1:] if tr["t"][0] == T - 1 and len(errs) > 1 else errs
            parity["vs_reference_arm"] = {"kind": cpu_kind(), "chains": len(tr["sub"]), "steps": len(errs), "t": tr["t"],
                                          "max_abs_per_step": errs, "max_abs_excluding_first_cosine_step": max(later),
                                          "ok": bool(max(later) < 1e-4),
                                          "note": "step k starts from the CPU arm's x_t and uses its normals; t = T-1 of the cosine "
                                                  "schedule multiplies any forward difference by 1/sqrt(alpha_T) = 100"}
        eng.check_status()

    # ---- BASELINE configs 5 and 3 as short driver-visible sub-lines (single GPU, after everything above) ---------
    extra = None
    if rank == 0 and world == 1 and args.workload == "config2" and not args.no_extra_workloads:
        extra = {}
        def short_pass(name, lens, npad, t_from, nsteps, reps):
            eng.set_batch(lens, npad)
            nb = len(lens)
            x0 = torch.randn(nb, npad, 6, device=dev).remainder(2 * np.pi) - np.pi
            zz = torch.randn((min(nsteps, 50), nb, npad, 6), device=dev)
            def run():
                xx = x0.clone()
                done = 0
                while done < nsteps:
                    m_ = min(50, nsteps - done)
                    eng.p_sample_steps(xx, t_from - done, t_from - done - m_, zz[:m_], None, wrap)
                    done += m_
            run()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                run()
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / reps
        ms5 = short_pass("config5", [128] * 512, 128, min(250, T), min(250, T), 2)
        extra["config5"] = {"workload": "partial_noise_reconstruct: 512 chains x 128, denoise from t=250 (250 reverse steps, complete pass)",
                            "ms_per_pass": ms5, "value": 512 / (ms5 / 1000.0), "unit": "backbones/s", "extrapolated": False}
        ms3 = short_pass("config3", [128] * 4096, 128, T, 20, 1)
        extra["config3"] = {"workload": "4096 chains x 128, T=1000: 20 reverse steps timed (per-step cost does not depend on t), x50",
                            "ms_per_reverse_step": ms3 / 20, "value": 4096 / (ms3 / 20 * T / 1000.0), "unit": "backbones/s",
                            "extrapolated": True,
                            "tflops_algorithmic": synthetic.algorithmic_flops(synthetic.PRODUCTION, [128] * 4096) / (ms3 / 20 * 1e-3) / 1e12}
        eng.set_batch(lengths, n_pad)
        eng.check_status()

    # ---- multi-GPU self-check: the sharded public path against a single-rank rerun, bit for bit -------------------
    selfcheck = None
    if world > 1:
        Ts, per = 8, 32
        lens_g = synthetic.sweep_lengths(per * world)
        dsm = datasets.NoisedAnglesDataset(datasets.AnglesEmptyDataset("canonical-full-angles", pad=128), timesteps=Ts, beta_schedule="cosine")
        torch.manual_seed(SEED + 2)
        ng = dsm.sample_noise(torch.zeros(len(lens_g), 128, 6))[:, : max(lens_g)].contiguous()
        torch.manual_seed(SEED + 3)  # same device seed on every rank: parity-mode RNG (distributed.py)
        got = fdist.sample_final_sharded(model, lens_g, ng, Ts, dsm.alpha_beta_terms["betas"], wrap)
        if rank == 0:
            torch.manual_seed(SEED + 3)
            ref1 = sampling.p_sample_loop(model, lens_g, ng, Ts, dsm.alpha_beta_terms["betas"], is_angle=wrap, history="final")[-1]
            selfcheck = {"what": "distributed.sample_final_sharded (NCCL all-gather, parity-mode RNG) == single-rank sampling.p_sample_loop on the same seed",
                         "chains": len(lens_g), "timesteps": Ts, "bit_identical": bool(torch.equal(got, ref1)),
                         "max_abs_diff": float((got - ref1).abs().max())}
        eng.set_schedule(betas, T)
        eng.set_batch(lengths, n_pad)

    if rank == 0:
        line = {
            "metric": "backbones/sec", "value": value, "unit": "backbones/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": {"tc3x": "f32 (fp16 hi/lo 3-pass tensor-core GEMMs, fp32 accumulate)",
                                                              "fp32": "f32", "tc1x": "f16 (single-pass, NOT parity mode)"}[args.gemm],
            "data": "synthetic",
            "config": {"workload": wl_name, "timesteps": T, "reverse_steps_per_pass": start_t, "chains_per_gpu": B,
                       "gemm": args.gemm, "parallelism": f"dp{world} (independent chains, one all-gather of final angles)",
                       "l2": "inputs larger than L2: ~1 GB of activations per reverse step, 1000 steps per pass",
                       "algorithmic_tflop_per_pass": flops_step * start_t / 1e12},
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline, "kernels": kernels,
            "cpu_baseline": cpu_baseline, "parity": parity, "workloads": extra, "multi_gpu_selfcheck": selfcheck,
            "next_rows": {"nerf": nerf_line, "writers": wline},
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
