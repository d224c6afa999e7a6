#!/usr/bin/env python
"""DDIM-100 autoencoding throughput (BASELINE.json metric) for the pdae_b200 hot path.

  python bench.py [--gpus N] [--steps K] [--warmup W]            # our CUDA path, one process per GPU (torchrun for N>1)
  python bench.py --impl reference [...]                          # the UNMODIFIED reference (baseline/_ref) on the host CPU cores

One "step" = one full autoencoding pass over one synthetic batch: 1 semantic-encoder forward + S DDIM-encode steps + S
DDIM-decode steps of the ShiftUNet (S=100 -> 200 decoder forwards + 200 fused DDIM updates).  `value` = images/s with
the batch resident in HBM; `e2e` = the same pass driven through the public API
(GaussianDiffusion.representation_learning_autoencoding) from pinned host memory, H2D and D2H inside the timed region.

Precision: the reference computes in fp32 (TF32 convs on a GPU).  With `--precision auto` (default) rank 0 first runs the
PARITY GATE -- a short autoencoding of the same network / weights through the CPU oracle and through every precision
mode of this package -- and the timed run uses the FASTEST mode whose reconstruction MSE is within 1e-5 of the
reference's (BASELINE.json: "autoencoding MSE within 1e-5 of the reference"); the other tensor-core mode is timed
briefly and reported under `modes`.  Rank 0 prints ONE JSON line.
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
if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
    os.environ["NCCL_DEBUG"] = "WARN"      # NCCL prints its version banner on STDOUT: keep stdout to the one JSON line

import torch  # noqa: E402

from pdae_b200.configs import CELEBA64_PROXY, DIFFUSION, FFHQ128_PROXY, FFHQ256_PROXY  # noqa: E402

WORKLOADS = {
    # name: (decoder cfg, image size, encoder kind, encoder input size, default per-GPU batch, GFLOP per decoder image-step)
    "celeba64": (CELEBA64_PROXY, 64, "celeba64", 64, 256, 48.11),
    "ffhq128": (FFHQ128_PROXY, 128, "ffhq128", 128, 64, 258.40),
    "ffhq256": (FFHQ256_PROXY, 256, "ffhq128", 128, 8, 967.20),
}
ENC_GFLOP = {"celeba64": 0.134, "ffhq128": 0.616}
REF_DIR = os.path.join(ROOT, "baseline", "_ref")
GATE = 1e-5          # |recon-MSE(ours) - recon-MSE(reference)| on [0,1]-scaled images (metric/utils.py:62-63)
MODE_ORDER = ("bf16", "bf16x3", "fp32")     # fastest first
DTYPE = {"bf16": "bf16", "bf16x3": "bf16x3 (split-operand bf16 tcgen05 MMAs, fp32 accumulate: fp32-grade products)", "fp32": "f32"}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="celeba64", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch (0 = workload default)")
    ap.add_argument("--ddim-steps", type=int, default=100)
    ap.add_argument("--precision", default="auto", choices=["auto", "bf16", "fp32", "bf16x3"])
    ap.add_argument("--weights", default="survey", choices=["survey", "synth"],
                    help="survey: reference default init + zero tensors re-drawn N(0,0.02^2) (SURVEY 8d); synth: fan-in noise everywhere")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-profile", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the secondary-mode timing and the ffhq256 strong-scaling line")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the reconstructions of the last timed step to DIR/reconstruction.npy (float32, under 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


DUMP_BYTES = 60 << 20      # keeps the file under 64 MB


def dump_reconstruction(d, rec):
    """rec as d/reconstruction.npy in float32.  Above DUMP_BYTES it is cut to a fixed, seeded sample of its images, so two
    builds run with the same arguments write comparable files.  Compare with a tolerance: the conv epilogues accumulate
    GroupNorm statistics with floating-point atomics and the 200-step loop amplifies their last-bit differences (two runs of
    one build, default celeba64 bf16x3 workload, B200 at 1000 W: max |diff| 7.2e-3)."""
    import numpy as np
    a = rec.float().cpu().numpy()
    if a.nbytes > DUMP_BYTES:
        a = a[np.sort(np.random.default_rng(0).choice(len(a), DUMP_BYTES // a[0].nbytes, replace=False))]
    os.makedirs(d, exist_ok=True)
    np.save(os.path.join(d, "reconstruction.npy"), a)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index=0):
        self.index, self.rows, self.stop = index, [], threading.Event()
        self.th = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        while not self.stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self.stop.wait(0.2)

    def __enter__(self):
        self.th.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.th.join(timeout=6)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for j, n in enumerate(names) if any(r[3 + j].lower().startswith("active") for r in self.rows if len(r) > 3 + j)]
        mx = float(self.rows[0][1]) if self.rows[0][1].replace(".", "").isdigit() else None
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": reasons, "samples": len(self.rows)}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", 1427.1), d.get("hbm_gbs", 6575.1), "measured (MEASURED_PEAKS.json, sustained bf16)"
    return 1400.0, 6650.0, "fallback (B200_PROFILING.md)"


# ----------------------------------------------------------------------------------------------------------------------
# weights: built ONCE on the CPU from this package's parameter holders; the oracle, the reference arm and the CUDA path all
# consume the same state_dict
# ----------------------------------------------------------------------------------------------------------------------
def build_cpu_models(cfg, enc_kind, weights, latent_dim=512, seed=0):
    from pdae_b200.model.representation_learning.encoder import CELEBA64Encoder, FFHQEncoder
    from pdae_b200.model.shift_unet import ShiftUNet
    from pdae_b200.utils.synth import build_survey_init, fill_module_
    Enc = CELEBA64Encoder if enc_kind == "celeba64" else FFHQEncoder
    c = dict(cfg, latent_dim=latent_dim)
    if weights == "survey":
        dec = build_survey_init(lambda: ShiftUNet(**c), seed)
        enc = build_survey_init(lambda: Enc(latent_dim=latent_dim), seed + 1)
    else:
        dec, enc = fill_module_(ShiftUNet(**c), seed=seed), fill_module_(Enc(latent_dim=latent_dim), seed=seed + 1)
    return dec.eval(), enc.eval(), c


def oracle_fns(dec, enc, c, enc_kind):
    from oracle import pdae_oracle as O
    dsd = {k: v.detach().clone() for k, v in dec.state_dict().items()}
    esd = {k: v.detach().clone() for k, v in enc.state_dict().items()}
    return (lambda x: O.encoder_forward(esd, enc_kind, x)), (lambda x, t, z: O.shiftunet_forward(dsd, c, x, t, z)), O


def cpu_sample_port(dec, enc, c, size, enc_kind, enc_size, S, batch, n_steps, warm=1):
    """Oracle port on the host cores: n_steps DDIM steps (ShiftUNet forward + update); images/s extrapolated to 2*S steps +
    1 encoder forward per image (every step is identical work)."""
    from pdae_b200.utils.host import host_cores
    from pdae_b200.utils.synth import synth_images, synth_normal
    enc_f, dec_f, O = oracle_fns(dec, enc, c, enc_kind)
    cores = host_cores()  # affinity and cgroup quota: a box may expose 128 logical CPUs but grant a 16-CPU quota
    torch.set_num_threads(cores)
    D = O.DiffusionOracle(DIFFUSION)
    tabs, tmap, _ = D._ddim(f"ddim{S}")
    x = synth_normal((batch, 3, size, size), 5)
    x0e = synth_images(batch, 3, enc_size, 6)
    with torch.inference_mode():
        t0 = time.perf_counter()
        z = enc_f(x0e)
        t_enc = time.perf_counter() - t0
        t = torch.full((batch,), S // 2, dtype=torch.long)
        for _ in range(warm):
            dec_f(x, tmap[t], z)
        t0 = time.perf_counter()
        for _ in range(n_steps):
            eps, grad = dec_f(x, tmap[t], z)
            x = O.ddim_update(tabs, x, t, eps, grad, "sample")
        t_step = (time.perf_counter() - t0) / n_steps
    return batch / (2 * S * t_step + t_enc), cores, t_step, t_enc


class ReferenceCPU:
    """The UNMODIFIED reference (ckczzj/PDAE, its package directories placed in baseline/_ref, which is git-ignored and not
    fetched by the build) driven through its own public API on the host CPU cores: model.shift_unet.ShiftUNet, the encoder
    class, diffusion.ddim.DDIM.shift_ddim_sample.  None of this package's kernels or modules are on this path; only the
    synthetic state_dict is shared."""

    def __init__(self, dec, enc, c, enc_kind, S):
        sys.path.insert(0, REF_DIR)
        import diffusion.gaussian_diffusion as rgd          # noqa: E402  (reference)
        import model.representation_learning.encoder as renc  # noqa: E402
        from diffusion.ddim import DDIM as RDDIM            # noqa: E402
        from model.shift_unet import ShiftUNet as RShiftUNet  # noqa: E402
        assert os.path.realpath(rgd.__file__).startswith(os.path.realpath(REF_DIR)), "reference import resolved elsewhere"
        self.dec = RShiftUNet(**c).eval()
        self.dec.load_state_dict(dec.state_dict())
        self.enc = getattr(renc, "CELEBA64Encoder" if enc_kind == "celeba64" else "FFHQEncoder")(latent_dim=c["latent_dim"]).eval()
        self.enc.load_state_dict(enc.state_dict())
        self.gd = rgd.GaussianDiffusion(DIFFUSION, device="cpu")
        nb, tmap = self.gd.get_ddim_betas_and_timestep_map(f"ddim{S}", self.gd.alphas_cumprod.cpu().numpy())
        self.ddim = RDDIM(nb, tmap, "cpu")

    def sample(self, size, enc_size, S, batch, n_steps, warm=1):
        from pdae_b200.utils.host import host_cores
        from pdae_b200.utils.synth import synth_images, synth_normal
        cores = host_cores()
        torch.set_num_threads(cores)
        x = synth_normal((batch, 3, size, size), 5)
        x0e = synth_images(batch, 3, enc_size, 6)
        with torch.inference_mode():
            t0 = time.perf_counter()
            z = self.enc(x0e)
            t_enc = time.perf_counter() - t0
            t = torch.full((batch,), S // 2, dtype=torch.long)
            for _ in range(warm):
                self.ddim.shift_ddim_sample(self.dec, z, x, t)
            t0 = time.perf_counter()
            for _ in range(n_steps):
                x = self.ddim.shift_ddim_sample(self.dec, z, x, t)
            t_step = (time.perf_counter() - t0) / n_steps
        return batch / (2 * S * t_step + t_enc), cores, t_step, t_enc


def have_reference():
    return os.path.exists(os.path.join(REF_DIR, "diffusion", "ddim.py")) and os.path.exists(os.path.join(REF_DIR, "model", "shift_unet.py"))


def cpu_batch(size):
    return 32 if size <= 64 else (8 if size <= 128 else 2)     # SURVEY 8(d): large enough that every granted core has work


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg, size, enc_kind, enc_size, _, _ = WORKLOADS[args.workload]
    S = args.ddim_steps
    b = cpu_batch(size)
    dec, enc, c = build_cpu_models(cfg, enc_kind, args.weights)
    kind = "reference" if have_reference() else "port"
    ref = ReferenceCPU(dec, enc, c, enc_kind, S) if kind == "reference" else None
    vals = []
    for i in range(args.warmup + args.steps):
        if ref is not None:
            ips, cores, t_step, t_enc = ref.sample(size, enc_size, S, b, n_steps=1, warm=1 if i == 0 else 0)
        else:
            ips, cores, t_step, t_enc = cpu_sample_port(dec, enc, c, size, enc_kind, enc_size, S, b, n_steps=1, warm=1 if i == 0 else 0)
        if i >= args.warmup:
            vals.append((ips, t_step))
    ips = sum(v[0] for v in vals) / len(vals)
    ms = 1e3 * sum(v[1] for v in vals) / len(vals)
    what = "unmodified reference modules (baseline/_ref: model.shift_unet.ShiftUNet + diffusion.ddim.DDIM.shift_ddim_sample, torch CPU fp32)" \
        if kind == "reference" else "oracle port (baseline/_ref absent)"
    sample = f"{what}; {b} images x 1 ShiftUNet DDIM step per bench step ({ms / 1e3:.2f} s), extrapolated to {2 * S} steps + 1 encoder forward per image"
    line = {"impl": "reference", "metric": "ddim100_autoencoding_images_per_sec", "value": ips, "unit": "images/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{args.workload}-proxy ShiftUNet+encoder, DDIM-{S} encode + DDIM-{S} decode", "batch": b,
                       "weights": args.weights},
            "cpu_baseline": {"value": ips, "unit": "images/s", "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": ips, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------------------------------
def mse01(a, b):
    """metric/utils.py:62-63 on images scaled to [0,1] as the reference's eval loop does (sampler/autoencoding_eval.py:84-85)."""
    return float((((a + 1) / 2 - (b + 1) / 2) ** 2).mean())


def parity_gate(gd, enc, dec, dec_cpu, enc_cpu, c, size, enc_kind, enc_input, dev, weights):
    """The oracle used as the CHECKER on a bounded sample of the bench workload: a short DDIM autoencoding of a few images
    through the CPU oracle and through this package in every precision mode, same weights and inputs.  Reports, per mode,
    the reconstruction MSE (BASELINE.json: "recon MSE vs ref"), its distance to the reference's, the relative L2 distance of
    the reconstructions, and whether the mode passes the 1e-5 gate."""
    from pdae_b200.utils.synth import synth_images
    n, s = (2, 10) if size <= 64 else ((1, 5) if size <= 128 else (1, 3))
    style = f"ddim{s}"
    x0 = synth_images(n, 3, size, 4242)
    enc_o, dec_o, O = oracle_fns(dec_cpu, enc_cpu, c, enc_kind)
    D = O.DiffusionOracle(DIFFUSION)
    from pdae_b200.utils.host import host_cores
    torch.set_num_threads(host_cores())
    with torch.inference_mode():
        z = enc_o(enc_input(x0))
        ref = D.representation_learning_ddim_sample(style, dec_o, D.representation_learning_ddim_encode(style, dec_o, x0, z), z)
    m_ref = mse01(ref, x0)
    out = {"sample": f"{n} image(s), {style} encode + {style} decode, '{weights}' weights, same weights/inputs as the CPU oracle",
           "gate": f"|recon-MSE - reference recon-MSE| <= {GATE:g} on [0,1]-scaled images", "recon_mse_reference": m_ref, "modes": {}}
    prev = (enc.precision, dec.precision)
    for prec in MODE_ORDER:
        enc.precision = dec.precision = prec
        with torch.inference_mode():
            xd = x0.to(dev)
            zz = enc(enc_input(xd))
            rec = gd.representation_learning_ddim_sample(style, None, dec, None,
                                                         gd.representation_learning_ddim_encode(style, None, dec, xd, zz), zz).cpu()
        m = mse01(rec, x0)
        out["modes"][prec] = {"recon_mse": m, "delta_mse": abs(m - m_ref), "rel_l2_vs_reference": float((rec - ref).norm() / ref.norm()),
                              "pass": bool(abs(m - m_ref) <= GATE)}
    enc.precision, dec.precision = prev
    return out


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    import pdae_b200
    from pdae_b200.diffusion.gaussian_diffusion import GaussianDiffusion
    from pdae_b200.utils.synth import synth_images

    cfg, size, enc_kind, enc_size, dflt_b, gflop_step = WORKLOADS[args.workload]
    B = args.batch or dflt_b
    S = args.ddim_steps
    dec_cpu, enc_cpu, c = build_cpu_models(cfg, enc_kind, args.weights)
    import copy
    dec, enc = copy.deepcopy(dec_cpu).to(dev), copy.deepcopy(enc_cpu).to(dev)
    gd = GaussianDiffusion(DIFFUSION, dev)
    style = f"ddim{S}"

    def enc_input(x):
        return x if enc_size == size else torch.nn.functional.avg_pool2d(x, size // enc_size)

    # ---- parity gate (rank 0) and mode selection ---------------------------------------------------------------------
    gate = None
    chosen = args.precision
    if args.precision == "auto":
        code = torch.zeros(1, dtype=torch.int64, device=dev)
        if rank == 0:
            gate = parity_gate(gd, enc, dec, dec_cpu, enc_cpu, c, size, enc_kind, enc_input, dev, args.weights)
            passing = [m for m in MODE_ORDER if gate["modes"][m]["pass"]]
            code[0] = MODE_ORDER.index(passing[0]) if passing else MODE_ORDER.index("fp32")
        if world > 1:
            dist.broadcast(code, 0)
        chosen = MODE_ORDER[int(code.item())]
    pdae_b200.set_default_precision(chosen)
    dec.precision = enc.precision = chosen

    x_host = synth_images(B, 3, size, 100 + rank).pin_memory()
    out_host = torch.empty_like(x_host).pin_memory()
    x_dev = x_host.to(dev)
    gather = torch.empty(world * B, 3, size, size, device=dev) if world > 1 else None

    def autoencode(x, g=gather):
        with torch.inference_mode():
            z = enc(enc_input(x))
            x_T = gd.representation_learning_ddim_encode(style, None, dec, x, z)
            rec = gd.representation_learning_ddim_sample(style, None, dec, None, x_T, z)
            if world > 1:
                dist.all_gather_into_tensor(g, rec)  # the single collective of the sampling path
            return rec

    def timed(fn, k):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(k):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            dist.barrier()
        return float(ms.item())

    W = max(args.warmup, 3)
    for _ in range(W):
        autoencode(x_dev)
    last = {}

    def step():
        last["reconstruction"] = autoencode(x_dev)

    with ClockSampler(local) as clk:
        ms_total = timed(step, args.steps)
    if args.dump_outputs and rank == 0:   # with N > 1, the gathered reconstructions of every rank
        dump_reconstruction(args.dump_outputs, gather if world > 1 else last["reconstruction"])
    ms_step = ms_total / args.steps
    value = world * B / (ms_step / 1e3)

    def e2e_once():
        xd = x_host.to(dev, non_blocking=True)
        rec = autoencode(xd)
        out_host.copy_(rec, non_blocking=True)

    e2e_steps = max(1, min(args.steps, 3))     # (a full pass each; bounded so the default run stays within minutes)
    e2e_once()
    ms_e2e = timed(e2e_once, e2e_steps) / e2e_steps
    e2e_val = world * B / (ms_e2e / 1e3)

    # kernel-level view of ONE decoder step (CUDA events around every launch of the step plan)
    plan, _ = dec.plan_for(B, size, size)
    # + timestep select (+ the DDIM update kernel unless it is fused into the last head conv's epilogue), all inside the step graph
    launches_per_step = plan.n_launch + (1 if plan.head_fuse else 2)
    enc_plan = [v for k, v in enc._plans().items() if k[1] == chosen][0][0]
    gpu_launches = args.steps * (2 * S * launches_per_step + enc_plan.n_launch)
    peak_tf, peak_bw, peak_src = peaks()

    def kernel_view(pl):
        prof = pl.profile(reps=3)
        tot = sum(v["ms"] for v in prof.values())
        kinds = {k: {"ms": round(v["ms"], 4), "share": round(v["ms"] / tot, 4), "launches": v["launches"],
                     "tflops": round(v["flops"] / (v["ms"] * 1e9), 2) if v["flops"] and v["ms"] > 0 else None}
                 for k, v in sorted(prof.items(), key=lambda kv: -kv[1]["ms"])}
        dom = max((k for k in prof if k.startswith("conv")), key=lambda k: prof[k]["ms"])
        n_l = prof[dom]["launches"]
        ach = prof[dom]["flops"] / (prof[dom]["ms"] * 1e9)
        kname = {"conv_tc3": "pdae::conv_tc3_kernel", "conv_tc2": "pdae::conv_tc2_kernel", "conv_tc": "pdae::conv_tc_kernel"}.get(dom, "pdae::conv_simt_kernel")
        x3 = pl.precision == "bf16x3"
        roof = {"bound": "tensor", "kernel": kname, "achieved": round(ach, 2), "peak": peak_tf, "unit": "TFLOP/s",
                "frac": round(ach / peak_tf, 4), "traffic": None, "peak_source": peak_src, "launches_per_decoder_step": n_l,
                "flops_per_launch_avg": prof[dom]["flops"] / n_l, "ms_per_launch_avg": prof[dom]["ms"] / n_l,
                "step_ms_sum_of_kernels": round(tot, 3),
                "note": ("achieved = ALGORITHMIC FLOPs (2*B*H*W*Cout*Cin*k*k per launch) / CUDA-event time.  In the split-operand "
                         "mode every algorithmic product is three bf16 MMAs (hi*hi + lo*hi + hi*lo): the tensor pipe executes "
                         "3x these FLOPs, so the ceiling of `frac` in this mode is 1/3") if x3 else
                        "achieved = ALGORITHMIC FLOPs (2*B*H*W*Cout*Cin*k*k per launch) / CUDA-event time"}
        if x3:
            roof["executed_tflops"] = round(3 * ach, 2)
            roof["frac_executed"] = round(3 * ach / peak_tf, 4)
        tpath = os.path.join(ROOT, "profiles", "conv_traffic.json")
        if os.path.exists(tpath):
            tj = json.load(open(tpath)).get(f"{args.workload}:{B}:{pl.precision}:{dom}")
            if tj:   # ncu dram bytes, per launch like `achieved`
                roof["traffic"] = tj["traffic_bytes_per_launch"]
                roof["traffic_unit"] = "bytes/launch (ncu dram__bytes_read.sum + dram__bytes_write.sum, profiles/conv_traffic.json)"
        return roof, kinds

    roof, kinds = (None, {}) if args.no_profile else kernel_view(plan)

    # ---- extras: the other tensor-core mode, and the FFHQ-256 strong-scaling configuration ---------------------------------
    modes = {}
    extras = {}
    if not args.no_extras:
        other = [m for m in ("bf16", "bf16x3") if m != chosen]
        for m in other:
            try:
                dec.precision = enc.precision = m
                autoencode(x_dev)
                ms_m = timed(lambda: autoencode(x_dev), 1)
                pl_m, _ = dec.plan_for(B, size, size)
                r_m, k_m = (None, None) if args.no_profile else kernel_view(pl_m)
                modes[m] = {"value": round(world * B / (ms_m / 1e3), 4), "unit": "images/s", "ms_per_step": round(ms_m, 3),
                            "steps": 1, "warmup": 1, "roofline": r_m, "kernels_per_decoder_step": k_m,
                            "parity": "see cpu_baseline.parity.modes (N=1 line)"}
            except Exception as e:   # never lose the headline to a secondary measurement
                modes[m] = {"error": repr(e)[:300]}
            finally:   # free the secondary mode's arena
                for k in [k for k in dec._plans() if k[1] == m]:
                    del dec._plans()[k]
        dec.precision = enc.precision = chosen
        torch.cuda.empty_cache()
        extras["ffhq256_global64_strong"] = strong_scaling_extra(gd, chosen, world, rank, dev, timed)
        extras["latent_unconditional_sample"] = latent_sample_extra(gd, dec, chosen, world, rank, dev, timed, B, size)
        extras["pdae_training_step"] = training_step_extra(world, rank, dev, timed)
        if world == 1 and have_reference():
            extras["reference_pytorch_on_this_gpu"] = reference_gpu_extra(dec_cpu, enc_cpu, c, enc_kind, S, B, size, enc_size, dev,
                                                                          enc_input)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    flop_img = (2 * S * gflop_step + ENC_GFLOP[enc_kind]) * 1e9
    line = {
        "metric": "ddim100_autoencoding_images_per_sec", "value": round(value, 4), "unit": "images/s", "n_gpus": world,
        "steps": args.steps, "warmup": W, "ms_per_step": round(ms_step, 3), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": DTYPE[chosen], "data": "synthetic",
        "config": {"workload": f"{args.workload}-proxy ShiftUNet+encoder (proxy decoder config, SURVEY D4), {size}x{size}x3, "
                               f"DDIM-{S} encode + DDIM-{S} decode", "batch_per_gpu": B, "global_batch": world * B,
                   "parallelism": f"dp{world} batch-sharded, one all-gather of results", "precision": chosen,
                   "precision_selection": ("auto: fastest mode passing the 1e-5 recon-MSE gate vs the CPU oracle" if args.precision == "auto" else "forced by --precision"),
                   "weights": args.weights + (" (reference default init, all-zero tensors re-drawn N(0,0.02^2); SURVEY 8d)" if args.weights == "survey" else " (fan-in-scaled noise on every tensor)"),
                   "l2": "activations per step exceed L2 (inputs larger than L2)"},
        "e2e": {"value": round(e2e_val, 4), "unit": "images/s", "h2d_bytes_per_step": x_host.numel() * 4,
                "d2h_bytes_per_step": out_host.numel() * 4, "ms_per_step": round(ms_e2e, 3), "steps": e2e_steps},
        "gpu_launches": gpu_launches,
        "clocks": clk.summary(),
        "model_flops_utilization": {"algorithmic_tflops": round(value * flop_img / 1e12 / world, 2), "peak_tflops": peak_tf,
                                    "frac": round(value * flop_img / 1e12 / world / peak_tf, 4), "peak_source": peak_src},
        "roofline": roof, "kernels_per_decoder_step": kinds, "modes": modes, "extras": extras,
    }
    if not args.no_cpu_baseline and world == 1:   # the CPU baseline is an N=1, rank-0 leg
        b = cpu_batch(size)
        if have_reference():
            ips, cores, t_step, t_enc = ReferenceCPU(dec_cpu, enc_cpu, c, enc_kind, S).sample(size, enc_size, S, b, n_steps=3)
            kind, what = "reference", "unmodified reference modules from baseline/_ref (torch CPU fp32)"
        else:
            ips, cores, t_step, t_enc = cpu_sample_port(dec_cpu, enc_cpu, c, size, enc_kind, enc_size, S, b, n_steps=3)
            kind, what = "port", "oracle (torch-CPU restatement of the reference; baseline/_ref absent)"
        line["cpu_baseline"] = {"value": ips, "unit": "images/s", "cores": cores, "kind": kind,
                                "sample": f"{what}, batch {b}: 1 warm-up + 3 timed ShiftUNet DDIM steps ({t_step:.2f} s/step) + 1 "
                                          f"encoder forward, extrapolated to {2 * S} steps per image"}
    if gate is not None:
        line.setdefault("cpu_baseline", {})["parity"] = gate
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def strong_scaling_extra(gd, precision, world, rank, dev, timed):
    """BASELINE.json config 3: ffhq256-proxy at GLOBAL batch 64 (8 images / GPU at N=8), total work fixed as N grows.
    Timed on a short schedule (ddim10 encode + ddim10 decode: per-step work identical to ddim100, so the N-scaling ratio
    carries over); the images/s figure is also given scaled to 100+100 steps."""
    import torch.distributed as dist
    from pdae_b200.utils.synth import synth_images
    try:
        if 64 % world:
            return {"skipped": f"64 % {world} != 0"}
        b = 64 // world
        dec_cpu, enc_cpu, c = build_cpu_models(FFHQ256_PROXY, "ffhq128", "survey")
        dec, enc = dec_cpu.to(dev), enc_cpu.to(dev)
        dec.precision = enc.precision = precision
        x = synth_images(b, 3, 256, 300 + rank).to(dev)
        gather = torch.empty(64, 3, 256, 256, device=dev) if world > 1 else None
        s = 10

        def run():
            with torch.inference_mode():
                z = enc(torch.nn.functional.avg_pool2d(x, 2))
                xT = gd.representation_learning_ddim_encode(f"ddim{s}", None, dec, x, z)
                rec = gd.representation_learning_ddim_sample(f"ddim{s}", None, dec, None, xT, z)
                if world > 1:
                    dist.all_gather_into_tensor(gather, rec)
        run()
        ms = timed(run, 1)
        ips = 64 / (ms / 1e3)
        out = {"workload": "ffhq256-proxy ShiftUNet + FFHQ encoder (128-px pooled input), 256x256x3", "global_batch": 64,
               "batch_per_gpu": b, "n_gpus": world, "scaling": "strong", "precision": precision, "ddim_steps": f"{s}+{s}",
               "ms_per_pass": round(ms, 3), "images_per_sec_at_10_plus_10_steps": round(ips, 4),
               "images_per_sec_scaled_to_100_plus_100_steps": round(ips * s / 100, 4), "steps": 1, "warmup": 1,
               "algorithmic_tflops_per_gpu": round(ips * (2 * s * 967.20 + 0.616) * 1e9 / 1e12 / world, 2)}
        del dec, enc
        torch.cuda.empty_cache()
        return out
    except Exception as e:
        return {"error": repr(e)[:300]}


def reference_gpu_extra(dec_cpu, enc_cpu, c, enc_kind, S, B, size, enc_size, dev, enc_input):
    """Context, not the contract's reference arm (that one is the CPU run): the UNMODIFIED reference modules (baseline/_ref) on
    THIS GPU through stock PyTorch -- eager mode, fp32 parameters, TF32 convolutions / matmuls as the reference's trainers set
    (trainer/base_trainer.py:24-25).  (1) images/s of the same workload from timed DDIM steps; (2) the same 1e-5 gate probe:
    does the reference's own GPU arithmetic reproduce its CPU fp32 result on these weights?"""
    try:
        import copy
        from pdae_b200.utils.synth import synth_images, synth_normal
        old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
        torch.backends.cudnn.allow_tf32 = True
        torch.backends.cuda.matmul.allow_tf32 = True
        ref = ReferenceCPU(dec_cpu, enc_cpu, c, enc_kind, S)
        rdec, renc = copy.deepcopy(ref.dec).to(dev), copy.deepcopy(ref.enc).to(dev)
        import diffusion.gaussian_diffusion as rgd       # the reference (sys.path set by ReferenceCPU)
        from diffusion.ddim import DDIM as RDDIM
        g = rgd.GaussianDiffusion(DIFFUSION, device=dev)
        nb, tmap = g.get_ddim_betas_and_timestep_map(f"ddim{S}", g.alphas_cumprod.cpu().numpy())
        dd = RDDIM(nb, tmap, dev)
        x = synth_normal((B, 3, size, size), 5).to(dev)
        out = {"what": "unmodified reference modules, stock PyTorch eager on this GPU, TF32 convs/matmuls (trainer/base_trainer.py:24-25)",
               "batch": B}
        with torch.inference_mode():
            z = renc(enc_input(synth_images(B, 3, size, 6).to(dev)))
            t = torch.full((B,), S // 2, dtype=torch.long, device=dev)
            for _ in range(2):
                dd.shift_ddim_sample(rdec, z, x, t)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            n = 5
            for _ in range(n):
                x = dd.shift_ddim_sample(rdec, z, x, t)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / n
            out.update({"ms_per_decoder_step": round(ms, 2), "images_per_sec_extrapolated": round(B / (2 * S * ms / 1e3), 3),
                        "sample": f"{n} timed shift_ddim_sample steps at batch {B}, extrapolated to {2 * S} steps per image"})
            # gate probe: same images / schedule as cpu_baseline.parity
            ns, s = (2, 10) if size <= 64 else ((1, 5) if size <= 128 else (1, 3))
            x0 = synth_images(ns, 3, size, 4242)
            enc_o, dec_o, O = oracle_fns(dec_cpu, enc_cpu, c, enc_kind)
            D = O.DiffusionOracle(DIFFUSION)
            zc = enc_o(enc_input(x0))
            refc = D.representation_learning_ddim_sample(f"ddim{s}", dec_o, D.representation_learning_ddim_encode(f"ddim{s}", dec_o, x0, zc), zc)
            xd = x0.to(dev)
            rec = g.representation_learning_autoencoding(f"ddim{s}", f"ddim{s}", lambda a: renc(enc_input(a)), rdec, xd).cpu()
            m_ref, m_gpu = mse01(refc, x0), mse01(rec, x0)
            out["parity_tf32_vs_cpu_fp32"] = {"recon_mse": m_gpu, "delta_mse": abs(m_gpu - m_ref),
                                              "rel_l2_vs_reference": float((rec - refc).norm() / refc.norm()),
                                              "pass": bool(abs(m_gpu - m_ref) <= GATE)}
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old
        del rdec, renc
        torch.cuda.empty_cache()
        return out
    except Exception as e:
        return {"error": repr(e)[:300]}


def latent_sample_extra(gd, dec, precision, world, rank, dev, timed, B, size):
    """BASELINE.json config 4: unconditional sampling -- MLPSkipNet latent DPM (config/ffhq_latent.yml:16-23: 512 -> 2048 x 10
    layers) for DDIM-100 steps, then the ShiftUNet decoder for DDIM-100 steps with stop_percent = 0.3 (epsilon-only plan on
    the last 30) -- through GaussianDiffusion.latent_diffusion_sample (gaussian_diffusion.py:400-415), on the bench's decoder."""
    try:
        from pdae_b200.configs import FFHQ_LATENT
        from pdae_b200.model.mlp_skip_net import MLPSkipNet
        from pdae_b200.utils.synth import fill_module_, synth_normal
        mlp = fill_module_(MLPSkipNet(**{k: v for k, v in FFHQ_LATENT.items() if k != "model"}), seed=5).eval().to(dev)
        x_T = synth_normal((B, 3, size, size), 400 + rank).to(dev)
        mean, std = torch.zeros(1, 512, device=dev), torch.ones(1, 512, device=dev)

        def run():
            with torch.inference_mode():
                gd.latent_diffusion_sample("ddim100", "ddim100", mlp, dec, x_T, mean, std)
        run()
        ms = timed(run, 1)
        return {"workload": "MLPSkipNet(512, 2048, 10 layers) latent DDIM-100 + celeba64-proxy ShiftUNet DDIM-100 (stop_percent 0.3)",
                "batch_per_gpu": B, "n_gpus": world, "precision": precision, "ms_per_pass": round(ms, 3),
                "images_per_sec": round(world * B / (ms / 1e3), 4), "steps": 1, "warmup": 1}
    except Exception as e:
        return {"error": repr(e)[:300]}


def training_step_extra(world, rank, dev, timed):
    """BASELINE.json config 5: the PDAE training step (representation_learning_train_one_batch + backward + gradient all-reduce
    overlapped with the encoder backward + fused Adam/EMA), celeba64-proxy, 32 images per GPU.  Decoder forward, data gradients and
    weight gradients run on the tensor cores in the split-operand fp32-grade mode (conv_tc2 / conv_tc3 / wgrad_tc); the encoder
    and the stride-2 / 3-channel convs are fp32 CUDA-core kernels (DESIGN.md section 3)."""
    try:
        import copy
        from pdae_b200.diffusion.gaussian_diffusion import GaussianDiffusion
        from pdae_b200.model.representation_learning.encoder import CELEBA64Encoder
        from pdae_b200.model.shift_unet import ShiftUNet
        from pdae_b200.optim import FusedAdamEMA
        from pdae_b200.utils.dist import OverlappedGradAllReduce
        from pdae_b200.utils.synth import fill_module_, synth_images
        Bt = 32
        dec = fill_module_(ShiftUNet(latent_dim=512, **dict(CELEBA64_PROXY, dropout=0.1)), seed=0).to(dev)
        enc = fill_module_(CELEBA64Encoder(latent_dim=512), seed=1).to(dev).train()
        dec.freeze()
        dec.set_train_mode()
        dec.precision = enc.precision = "fp32"
        ema_dec, ema_enc = copy.deepcopy(dec).requires_grad_(False), copy.deepcopy(enc).requires_grad_(False)
        gdt = GaussianDiffusion(DIFFUSION, dev)
        groups = [list(enc.parameters()), list(dec.label_emb.parameters()), list(dec.shift_middle_block.parameters()),
                  list(dec.shift_output_blocks.parameters()), list(dec.shift_out.parameters())]
        opt = FusedAdamEMA([{"params": g} for g in groups], lr=1e-4, ema_decay=0.9999)
        opt.attach_ema(enc, ema_enc)
        opt.attach_ema(dec, ema_dec)
        x0 = synth_images(Bt, 3, 64, 500 + rank).to(dev)
        red = OverlappedGradAllReduce([[p for g in groups[1:] for p in g], groups[0]])

        def step():
            loss = gdt.representation_learning_train_one_batch(enc, dec, x0)["prediction_loss"]
            loss.backward()
            opt.step(grad_scale=red.finish())
            opt.zero_grad(set_to_none=True)
        for _ in range(3):
            step()
        k = 5
        ms = timed(lambda: [step() for _ in range(k)], 1) / k
        n_train = sum(p.numel() for g in groups for p in g)
        red.remove()
        out = {"workload": "celeba64-proxy encoder + ShiftUNet (shift half trainable), dropout 0.1, fused Adam+EMA", "batch_per_gpu": Bt,
               "n_gpus": world, "ms_per_step": round(ms, 2), "images_per_sec": round(world * Bt / ms * 1e3, 2), "steps": k, "warmup": 3,
               "scaling": "weak", "allreduce_bytes_per_step": 4 * n_train if world > 1 else 0,
               "arithmetic": "decoder forward, data and weight gradients on the tensor cores (split-operand, fp32-grade); encoder "
                             "and stride-2 / 3-channel convs fp32 on CUDA cores"}
        del dec, enc, ema_dec, ema_enc, opt
        torch.cuda.empty_cache()
        return out
    except Exception as e:
        return {"error": repr(e)[:300]}


if __name__ == "__main__":
    main()
