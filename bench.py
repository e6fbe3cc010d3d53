#!/usr/bin/env python
"""bench.py — train-step images/sec of the GAN / VAE hot path on N B200s.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload ns|wgp|vae|dcgan] [--dump-outputs DIR]   # this repo's CUDA path
  python bench.py --impl reference [--gpus N] ...                                # the reference's own CPU path
  torchrun --nproc-per-node N bench.py --gpus N ...                              # N > 1 (driver does this)

One "step" = one reference train step: fetch a batch of real images, D update (forward G and
D, loss, backward, Adam), G update (src/ns_gan.py:126-156); VAE: compute_batch + backward + Adam
(src/vae.py:150-167).  Headline workload = BASELINE.json configs[1]: NSGAN 784-400-1 / 20-400-784,
bf16 tensor-core operands, B = 65536 images per GPU per step (weak scaling), synthetic
Bernoulli(0.1307)-like 28x28 binary images, nn.Linear-default random-init weights.  At N = 1 the
same JSON line also carries configs[2] (WGAN-GP, B = 65536) and configs[3] (VAE, B = 131072) under
"workloads", the drop-in Trainer.train throughput ("e2e_trainer") and the small-batch regime.
Prints ONE JSON line (rank 0).
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "generative-models_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

X, H, Z = 784, 400, 20
# SURVEY.md 8a: algorithmic FLOPs of one train step per image
def _dcgan_flop_per_img(hd=64, z=100, ch=3):
    """algorithmic FLOPs of one NSGAN train step with the DCGAN conv nets (2 FLOP / MAC; needed work only, as SURVEY 8a
    counts the MLP: D step = G fwd + 2 D fwd + 2 D bwd (weight grads + input grads above layer 1); G step = G fwd + D fwd +
    D input-grad chain + G bwd)"""
    gc, dc = [8 * hd, 4 * hd, 2 * hd, hd, ch], [hd, 2 * hd, 4 * hd, 8 * hd]
    d_l = [1024 * dc[0] * 16 * ch, 256 * dc[1] * 16 * dc[0], 64 * dc[2] * 16 * dc[1], 16 * dc[3] * 16 * dc[2], 16 * dc[3]]
    g_l = [z * 16 * gc[0], 16 * gc[0] * 16 * gc[1], 64 * gc[1] * 16 * gc[2], 256 * gc[2] * 16 * gc[3], 1024 * gc[3] * 16 * gc[4]]
    Df, Gf = 2.0 * sum(d_l), 2.0 * sum(g_l)
    d_bwd = 2.0 * (2 * sum(d_l) - d_l[0])            # wgrad everywhere + dgrad except into the image
    d_dgrad = 2.0 * sum(d_l)                          # G step: input-gradient chain only, down to the image
    g_bwd = 2.0 * (2 * sum(g_l) - g_l[0])            # wgrad everywhere + dgrad except into z
    return (Gf + 2 * Df + 2 * d_bwd) + (Gf + Df + d_dgrad + g_bwd)


FLOP_PER_IMG = {"ns": 6326400.0, "wgp": 8836800.0, "vae": 3280000.0, "dcgan": _dcgan_flop_per_img()}
DEFAULT_BATCH = {"ns": 65536, "wgp": 65536, "vae": 131072, "dcgan": 1024}
CONFIG_NAME = {"ns": "NSGAN MLP (D 784-400-1, G 20-400-784), BASELINE configs[1]",
               "wgp": "WGAN-GP MLP (ReLU critic, lambda 10 gradient penalty, closed-form double backward), BASELINE configs[2]",
               "vae": "VAE MLP (784-400-(20,20), 20-400-784; SSE + KL as src/vae.py:203,212), BASELINE configs[3]",
               "dcgan": "NSGAN with DCGAN conv G / D (64x64x3, hidden 64, z 100; im2col + tcgen05 GEMM convolutions, BatchNorm), "
                        "BASELINE configs[4]: global batch 8192 on 8 GPUs = 1024 per GPU, NCCL all-reduce of the G / D gradients"}
METRIC = "train_step_images_per_sec"


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return d, "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", "100"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(", ") for r in open(self.f.name).read().strip().splitlines() if r.strip()]
        os.unlink(self.f.name)
        sm, reasons, mx, pw = [], set(), None, []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            if len(r) < 9:
                continue
            try:
                sm.append(float(r[1]))
                mx = float(r[2])
                pw.append(float(r[3]))
            except ValueError:
                continue
            for n, v in zip(names, r[5:9]):
                if v.strip().lower().startswith("active"):
                    reasons.add(n)
        if sm:
            sm.sort()
            out.update(sm_mhz=sm[len(sm) // 2], sm_max_mhz=mx, reasons=sorted(reasons), samples=len(sm),
                       power_w_max=max(pw) if pw else None)
        return out


# ------------------------------------------------------------------------------------------------
# workloads
# ------------------------------------------------------------------------------------------------
def init_gan_weights(eng):
    """nn.Linear default init under torch.manual_seed(1234) on CPU (SURVEY.md 8d)."""
    import torch
    import torch.nn as nn
    torch.manual_seed(1234)
    g1, g2 = nn.Linear(Z, H), nn.Linear(H, X)
    d1, d2 = nn.Linear(X, H), nn.Linear(H, 1)
    eng.load(0, [g1.weight.data, g1.bias.data, g2.weight.data, g2.bias.data])
    eng.load(1, [d1.weight.data, d1.bias.data, d2.weight.data, d2.bias.data])


def init_vae_weights(eng):
    import torch
    import torch.nn as nn
    torch.manual_seed(1234)
    mods = {"encoder.linear": nn.Linear(X, H), "encoder.mu": nn.Linear(H, Z), "encoder.log_var": nn.Linear(H, Z),
            "decoder.linear": nn.Linear(Z, H), "decoder.recon": nn.Linear(H, X)}
    t = {}
    for k, m in mods.items():
        t[k + ".weight"], t[k + ".bias"] = m.weight.data, m.bias.data
    eng.load(t)


class Workload:
    """One engine + its step function.  step(None) = device-resident path (packed pool + on-device sampler,
    on-device Philox noise); step(batch_bits) = the same step on an explicit packed batch (e2e leg)."""

    def __init__(self, name, B, pool_bits, pool_n, rank, world, comm=None, prec="bf16"):
        import torch
        import gm_b200
        from gm_b200 import parallel as par
        self.name, self.B, self.bits, self.N, self.world, self.comm = name, B, pool_bits, pool_n, world, comm
        self.par, self.torch = par, torch
        self.seed = par.rank_seed(1000, rank)
        self.s = 0
        self.overlap = False
        self.split_exchange = False
        self.inv = par.inv_global_batch(B, world)
        if name == "dcgan":
            self.eng = gm_b200.DcganEngine(hidden_dim=64, z_dim=100, channels=3, variant="ns")
            self.hpG, self.hpD = gm_b200.AdamHP.make(2e-4), gm_b200.AdamHP.make(2e-4)
            g = torch.Generator(device=pool_bits.device).manual_seed(77 + rank)
            # device-resident synthetic images, NHWC bf16 rows, 4 batches (100 MB > the per-step reuse window)
            self.pool = (torch.rand(4 * B * 4096, 3, device=pool_bits.device, generator=g) < 0.3).to(torch.bfloat16)
            self.loss_buf = self.eng.loss_buf
        elif name == "vae":
            self.eng = gm_b200.VaeEngine(X, H, Z, max_batch=B, precision=prec)
            init_vae_weights(self.eng)
            self.hp = gm_b200.AdamHP.make(1e-3, weight_decay=1e-5)          # src/vae.py:127,139-142
            self.eng.set_sampler(pool_n, max(pool_n // B, 1), 3435 + rank)
            self.eng.set_lazy_grads(world == 1)                               # gradient gather fused into the Adam kernel
            self.loss_buf = self.eng.loss_buf
        else:
            self.eng = gm_b200.GanEngine(X, H, Z, max_batch=B, variant=name, d_out_act="relu" if name == "wgp" else "sigmoid",
                                         precision=prec)
            init_gan_weights(self.eng)
            lr = 2e-4 if name == "ns" else 1e-4                              # src/ns_gan.py:311-314, src/w_gp_gan.py:338
            self.hpG, self.hpD = gm_b200.AdamHP.make(lr), gm_b200.AdamHP.make(lr)
            # N > 1: the SUM of the flat D / G gradients runs inside the Adam kernel over CUDA-IPC peer mappings
            self.eng.set_lazy_grads(world == 1 or comm is not None)
            self.loss_buf = self.eng.loss_buf
            # GM_DP_OVERLAP=1: the D-gradient exchange + Adam runs on a side stream under the G step's generator
            # forward, which does not depend on the D update (gm_gan_g_forward_stage / gm_gan_g_grad_staged)
            self.overlap = comm is not None and os.environ.get("GM_DP_OVERLAP", "0") == "1"
            # GM_DP_SPLIT=1: two-phase exchange with independent work in between - measured SLOWER than the fused kernel
            # (2 GPUs 0.7235 vs 0.690 ms/step, 8 GPUs 0.7424 vs 0.7125; profiles/r2_exchange.md), so off by default
            self.split_exchange = os.environ.get("GM_DP_SPLIT", "0") == "1"
            if self.overlap:
                self.side = torch.cuda.Stream()
                self.ev_d, self.ev_a = torch.cuda.Event(), torch.cuda.Event()

    def step(self, batch_bits=None):
        eng, B, s = self.eng, self.B, self.s
        self.s += 1
        if self.name == "dcgan":
            if batch_bits is None:
                x = self.pool[(s % 4) * B * 4096:(s % 4 + 1) * B * 4096]
            else:                                   # e2e leg: a uint8 NCHW-flattened host batch that just landed on the device
                x = eng.stage_images(batch_bits)
            eng.d_grad(x, B, inv_global_batch=self.inv, seed=self.seed, step=s)
            self.par.sum_gradients(eng.D.grads)     # NCCL all-reduce (SUM) of the flat D gradient; no-op on one GPU
            eng.apply(1, self.hpD)
            eng.g_grad(B, inv_global_batch=self.inv, seed=self.seed, step=s)
            self.par.sum_gradients(eng.G.grads)
            eng.apply(0, self.hpG)
            return
        if self.name == "vae":
            if batch_bits is None:
                eng.set_sampler(self.N, max(self.N // B, 1), 3435)
                eng.grad(self.bits, fmt="bits", batch=B, seed=self.seed, step=s)
            else:
                eng.set_sampler(0, 0, 0)
                eng.grad(batch_bits, fmt="bits", batch=B, seed=self.seed, step=s)
            if self.world > 1:
                self.par.sum_gradients(eng.grads)
            eng.apply(self.hp)
            return
        if batch_bits is None:
            eng.set_sampler(self.N, self.seed)
            eng.d_grad(self.bits, fmt="bits", batch=B, inv_global_batch=self.inv, seed=self.seed, step=s)
        else:
            eng.set_sampler(0, 0)
            eng.d_grad(batch_bits, fmt="bits", batch=B, inv_global_batch=self.inv, seed=self.seed, step=s)
        if self.comm is not None and self.split_exchange and not self.overlap:
            # two-phase exchange on ONE stream: publish the D gradient, run the G step's generator forward (independent of
            # the D update), then wait + sum + Adam; publish the G gradient, stage the next step's real rows, then finish
            eng.exchange_begin(1, self.comm)
            eng.g_forward_stage(B, seed=self.seed, step=s)
            eng.apply_allreduce(1, self.hpD, self.comm)
            eng.g_grad_staged(B, inv_global_batch=self.inv)
            eng.exchange_begin(0, self.comm)
            if batch_bits is None:
                eng.d_stage(self.bits, fmt="bits", batch=B, step=s + 1)
            eng.apply_allreduce(0, self.hpG, self.comm)
            return
        if self.overlap:
            torch = self.torch
            self.ev_d.record()
            with torch.cuda.stream(self.side):
                self.side.wait_event(self.ev_d)
                eng.apply_allreduce(1, self.hpD, self.comm)
                self.ev_a.record(self.side)
            eng.g_forward_stage(B, seed=self.seed, step=s)
            torch.cuda.current_stream().wait_event(self.ev_a)
            eng.g_grad_staged(B, inv_global_batch=self.inv)
            self._apply(0, self.hpG)
            return
        self._apply(1, self.hpD)
        eng.g_grad(B, inv_global_batch=self.inv, seed=self.seed, step=s)
        self._apply(0, self.hpG)

    def _apply(self, net, hp):
        if self.comm is not None:
            self.eng.apply_allreduce(net, hp, self.comm)     # publish, sum over NVLink, Adam: one kernel
        else:
            if self.world > 1:
                self.par.sum_gradients(self.eng.grads[net])  # NCCL all-reduce fallback (GM_DP=nccl)
            self.eng.apply(net, hp)

    def losses(self):
        return [float(v) for v in self.loss_buf.tolist()]

    def outputs(self):
        """What a caller of step() gets from it: the step's losses and the updated fp32 parameters, by name."""
        eng = self.eng
        out = {"losses": self.loss_buf}
        if self.name == "dcgan":
            for tag, net in (("G", eng.G), ("D", eng.D)):
                out.update(("%s.%s" % (tag, n), net.view(n)) for n in net.names)
        elif self.name == "vae":
            out.update(eng.views())
        else:
            names = [m + s for m in ("G.linear", "G.generate", "D.linear", "D.discriminate") for s in (".weight", ".bias")]
            out.update(zip(names, eng.views(0) + eng.views(1)))
        return out


def dump_outputs(wl, out_dir):
    """wl.outputs() as out_dir/<name>.npy in float32 (at most 26 MB: the DCGAN's parameters), so that two builds can be
    compared output for output on the same seeded inputs."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in wl.outputs().items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())


def make_pool(N, dev, rank):
    """device-resident synthetic dataset, 1 bit per pixel (binarised MNIST carries exactly that:
    src/utils.py:31); Bernoulli(1/8)-like density: AND of three random bytes"""
    import torch
    gen = torch.Generator(device=dev).manual_seed(3435 + rank)
    nbytes = N * X // 8
    bits = torch.randint(0, 256, (nbytes,), device=dev, dtype=torch.uint8, generator=gen)
    bits &= torch.randint(0, 256, (nbytes,), device=dev, dtype=torch.uint8, generator=gen)
    bits &= torch.randint(0, 256, (nbytes,), device=dev, dtype=torch.uint8, generator=gen)
    return bits.view(N, X // 8)


def run_ours(args):
    import torch
    import torch.distributed as dist
    import gm_b200
    from gm_b200 import parallel as par
    rank, world, local = par.init_from_env("nccl")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    name = args.workload
    B = args.batch or DEFAULT_BATCH[name]
    N = max(4 * 65536, 2 * B)                 # pool: 262144 images = 25.7 MB packed (412 MB as bf16 rows)
    bits = make_pool(N, dev, rank)
    comm = par.make_peer_comm(330000) if name in ("ns", "wgp") else None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    host_ms = [0.0]

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        t_host = time.perf_counter()
        for i in range(steps):
            fn(i)
        host_ms[0] = (time.perf_counter() - t_host) * 1e3 / steps    # CPU time to enqueue one step
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    pk, pk_src = peaks()
    peak_burst = float(pk.get("bf16_tflops"))
    peak_sust = float(pk.get("bf16_tflops_sustained", peak_burst))

    def roofline_of(wl, value_per_gpu, reps=3):
        """CUDA events around every GEMM launch of `reps` steps: dominant kernel and whole-step fractions."""
        gm_b200.prof_enable(True)
        for _ in range(reps):
            wl.step()
        prof = gm_b200.prof_collect()
        gm_b200.prof_enable(False)
        dom = max(prof, key=lambda r: r[1])
        dom_tf = dom[2] / (dom[1] * 1e-3) / 1e12 if dom[1] > 0 else 0.0
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath):      # dram bytes per launch of the dominant kernel from the committed ncu --set full capture
            traffic = json.load(open(tpath)).get(wl.name, {}).get("dram_bytes_per_launch")
        return {"bound": "hbm+tensor", "kernel": dom[0], "achieved": round(dom_tf, 1), "peak": peak_burst, "unit": "TFLOP/s",
                "frac": round(dom_tf / peak_burst, 4), "traffic": traffic,
                "peak_source": pk_src + ": burst cuBLAS bf16 (the timed region is a few ms at full clock); sustained %.1f" % peak_sust,
                "frac_of_sustained_peak": round(dom_tf / peak_sust, 4),
                "launches_per_step": dom[3] / float(reps), "avg_launch_ms": round(dom[1] / max(dom[3], 1), 4),
                "all_gemm_ms_per_step": round(sum(r[1] for r in prof) / float(reps), 4),
                "step_frac_of_tensor_roofline": round(value_per_gpu * FLOP_PER_IMG[wl.name] / (peak_burst * 1e12), 4),
                "note": "launch arithmetic intensity is at the B200 ridge (~260 FLOP/B): these GEMMs are co-limited by HBM and the tensor pipe",
                "by_kernel": [{"kernel": r[0], "ms_per_step": round(r[1] / float(reps), 4),
                               "tflops": round(r[2] / (r[1] * 1e-3) / 1e12, 1) if r[1] > 0 else 0.0,
                               "launches_per_step": r[3] / float(reps)} for r in prof if r[3]]}

    # ---------------------------------------------------------------- headline: device-resident step
    wl = Workload(name, B, bits, N, rank, world, comm)
    for _ in range(max(args.warmup, 3)):
        wl.step()
    gm_b200.launch_count(reset=True)
    sampler = ClockSampler(local) if rank == 0 else None
    ms = timed(lambda i: wl.step(), args.steps)
    host_enqueue_ms = host_ms[0]
    clocks = sampler.stop() if sampler else None
    launches = gm_b200.launch_count(reset=True)
    value = B * world * args.steps / (ms * 1e-3)
    losses = wl.losses()
    if args.dump_outputs and rank == 0:
        dump_outputs(wl, args.dump_outputs)

    # ---- e2e: same step through the host-facing call, HOST (pinned) batches; the H2D
    # copy of each step's batch and the D2H read of its losses are inside the timed region
    e2e_steps = args.steps
    nb = 4
    row_bytes = 3 * 64 * 64 if name == "dcgan" else X // 8          # dcgan: one byte per pixel value, NCHW flattened
    host = [torch.empty(B, row_bytes, dtype=torch.uint8).pin_memory() for _ in range(nb)]
    for k, hb in enumerate(host):
        if name == "dcgan":
            hb.copy_((torch.rand(B, row_bytes) < 0.3).to(torch.uint8))
        else:
            hb.copy_(bits[(k * B) % (N - B + 1):(k * B) % (N - B + 1) + B].cpu())
    stage = [torch.empty(B, row_bytes, dtype=torch.uint8, device=dev) for _ in range(2)]
    host_loss = torch.zeros(e2e_steps + 8, 2).pin_memory()
    copy_stream = torch.cuda.Stream()
    ready = [torch.cuda.Event() for _ in range(2)]
    freed = [torch.cuda.Event() for _ in range(2)]

    def prefetch(i):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(freed[i % 2])
            stage[i % 2].copy_(host[i % nb], non_blocking=True)
            ready[i % 2].record(copy_stream)

    def e2e_step(i):
        if i == 0:
            prefetch(0)
        prefetch(i + 1)                       # overlaps with this step's compute
        torch.cuda.current_stream().wait_event(ready[i % 2])
        wl.step(stage[i % 2])
        freed[i % 2].record()
        host_loss[i].copy_(wl.loss_buf, non_blocking=True)
    for f in freed:
        f.record()
    for i in range(3):
        e2e_step(i)
    torch.cuda.synchronize()
    for f in freed:
        f.record()
    ms_e2e = timed(e2e_step, e2e_steps)
    e2e_value = B * world * e2e_steps / (ms_e2e * 1e-3)

    roofline = roofline_of(wl, value / world)
    del wl

    extra = {}
    if world == 1 and not args.headline_only:
        # ---- the other BASELINE configs on the same box, shorter runs (same timing rules)
        others = {}
        for other in [w for w in ("ns", "wgp", "vae", "dcgan") if w != name]:
            Bo = DEFAULT_BATCH[other]
            wo = Workload(other, Bo, bits, N, rank, world, None)
            for _ in range(3):
                wo.step()
            gm_b200.launch_count(reset=True)
            k = min(args.steps, 20)
            mso = timed(lambda i: wo.step(), k)
            lo = gm_b200.launch_count(reset=True)
            vo = Bo * k / (mso * 1e-3)
            others[other] = {"value": round(vo, 1), "unit": "images/s", "ms_per_step": round(mso / k, 4), "steps": k, "batch": Bo,
                             "gpu_launches_per_step": lo / float(k), "flop_per_img": FLOP_PER_IMG[other],
                             "config": CONFIG_NAME[other], "losses_last_step": wo.losses(), "roofline": roofline_of(wo, vo)}
            del wo
        extra["workloads"] = others
        extra["e2e_trainer"] = bench_trainer(args, dev)
        extra["small_batch"] = bench_small_batch(dev)
        if not args.no_parity_mode:
            extra["parity_mode"] = bench_parity_mode(args, bits, N, rank, timed)

    if world > 1:
        dist.barrier()
        if rank != 0:
            if comm is not None:
                comm.close()
            dist.destroy_process_group()
            return
    out = {"metric": METRIC, "value": round(value, 1), "unit": "images/s", "n_gpus": world, "steps": args.steps,
           "warmup": max(args.warmup, 3), "ms_per_step": round(ms / args.steps, 4), "higher_is_better": True,
           "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
           "config": {"workload": "%s: B=%d per GPU, %s" % (CONFIG_NAME[name], B,
                                                           "1 optimizer step per batch, Adam lr 1e-3 wd 1e-5" if name == "vae" else
                                                           "1 D update + 1 G update per step, Adam"),
                      "global_batch": B * world, "parallelism": "dp%d" % world,
                      "gradient_exchange": ("none (1 GPU)" if world == 1 else
                                            "NCCL all-reduce (SUM) of the flat G / D gradients" if name in ("dcgan", "vae") else
                                            "fused peer all-reduce + Adam kernel (push over CUDA-IPC NVLink mappings)%s" % (
                                                ", D exchange overlapped with the G forward" if os.environ.get("GM_DP_OVERLAP") == "1" else "")
                                            if comm is not None
                                            else "NCCL all-reduce"),
                      "inputs": "device-resident 1-bit synthetic images, pool %d (25.7 MB packed, 412 MB as bf16 rows), batch rows drawn "
                                "by the in-kernel permutation sampler; per-step working set ~1.5 GB > L2, no L2 flush needed" % N,
                      "noise": "on-device Philox"},
           "e2e": {"value": round(e2e_value, 1), "unit": "images/s", "ms_per_step": round(ms_e2e / e2e_steps, 4),
                   "h2d_bytes_per_step": B * row_bytes, "d2h_bytes_per_step": 8,
                   "input_format": ("uint8 NCHW-flattened images in pinned host memory, double-buffered H2D" if name == "dcgan" else
                                    "1 bit/pixel packed rows in pinned host memory, double-buffered H2D")},
           "gpu_launches": int(launches), "host_enqueue_ms_per_step": round(host_enqueue_ms, 4), "clocks": clocks, "roofline": roofline,
           "losses_last_step": losses}
    out.update(extra)
    if world == 1 and not args.no_cpu:
        out["cpu_baseline"] = cpu_baseline()
    print(json.dumps(out))
    if comm is not None:
        comm.close()
    if world > 1:
        dist.destroy_process_group()


def bench_trainer(args, dev):
    """Throughput through the reference's plugin API: NSGANTrainer.train over a host
    DataLoader(TensorDataset) at B = 65536 (src/ns_gan.py:94-170 as the user calls it)."""
    import torch
    import ns_gan
    B, N = 65536, 4 * 65536
    g = torch.Generator().manual_seed(3435)
    imgs = (torch.rand(N, 1, 28, 28, generator=g) < 0.1307).float()             # the host dataset, fp32 like src/utils.py:31-42
    loader = torch.utils.data.DataLoader(torch.utils.data.TensorDataset(imgs, torch.zeros(N, dtype=torch.long)), batch_size=B, shuffle=True)
    torch.manual_seed(1234)
    model = ns_gan.NSGAN(784, 400, 20)
    trainer = ns_gan.NSGANTrainer(model, loader, loader, loader, viz=False)
    sink = open(os.devnull, "w")
    so = sys.stdout
    try:
        sys.stdout = sink
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        trainer.train(num_epochs=1, G_lr=2e-4, D_lr=2e-4, D_steps=1)           # first call: engine creation + dataset packing
        torch.cuda.synchronize()
        t_first = time.perf_counter() - t0
        epochs = max(2, (args.steps + 3) // 4)
        t0 = time.perf_counter()
        trainer.train(num_epochs=epochs, G_lr=2e-4, D_lr=2e-4, D_steps=1)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
    finally:
        sys.stdout = so
        sink.close()
    steps = epochs * 4
    return {"value": round(steps * B / dt, 1), "unit": "images/s", "ms_per_step": round(dt / steps * 1e3, 4), "steps": steps,
            "api": "ns_gan.NSGANTrainer(model, DataLoader(TensorDataset(fp32 [N,1,28,28]), batch_size=65536, shuffle=True), ...)"
                   ".train(num_epochs=%d): wall clock around the call incl. the per-epoch loss read-back and print" % epochs,
            "first_call_s": round(t_first, 3),
            "first_call_includes": "engine creation, packing the 822 MB fp32 host dataset to 1 bit/pixel in HBM, 1 epoch",
            "losses_last_step": {"D": trainer.Dlosses[-1], "G": trainer.Glosses[-1]}}


def bench_small_batch(dev):
    """BASELINE configs[0] regime on the GPU: B = 64 and B = 100 (the reference's defaults,
    src/ns_gan.py:311-314, src/utils.py:16), launch-bound; eager launches vs the CUDA-graphed step."""
    import torch
    import gm_b200
    out = {}
    for Bs in (64, 100):
        N = 50000
        bits = make_pool(N, dev, 0)
        wl = Workload("ns", Bs, bits, N, 0, 1, None)
        for _ in range(20):
            wl.step()
        torch.cuda.synchronize()
        k = 300
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(k):
            wl.step()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        rec = {"eager_launch": {"value": round(Bs * k / (ms * 1e-3), 1), "ms_per_step": round(ms / k, 4)}}
        graph = getattr(gm_b200, "graphed_gan_step", None)
        if graph is not None:
            try:
                rec["cuda_graph"] = graph(wl, k)
            except Exception as exc:     # noqa: BLE001
                rec["cuda_graph"] = {"error": str(exc)[:200]}
        out["b%d" % Bs] = rec
        del wl
    out["trainer_b64_epoch"] = bench_trainer_small()
    out["unit"] = "images/s"
    return out


def bench_trainer_small():
    """BASELINE configs[0] through the reference's own API on the GPU: NSGANTrainer.train(1 epoch) over a shuffling
    DataLoader(TensorDataset) of N = 50000 images at B = 64 (782 steps) - what the cpu_baseline leg runs on the host."""
    import torch
    import ns_gan
    g = torch.Generator().manual_seed(3435)
    imgs = (torch.rand(50000, 1, 28, 28, generator=g) < 0.1307).float()
    loader = torch.utils.data.DataLoader(torch.utils.data.TensorDataset(imgs, torch.zeros(50000, dtype=torch.long)), batch_size=64, shuffle=True)
    res = {}
    for mode in ("cuda_graph", "eager_launch"):
        torch.manual_seed(1234)
        model = ns_gan.NSGAN(784, 400, 20)
        tr = ns_gan.NSGANTrainer(model, loader, loader, loader, viz=False)
        tr.cuda_graph = mode == "cuda_graph"
        so, sink = sys.stdout, open(os.devnull, "w")
        try:
            sys.stdout = sink
            tr.train(num_epochs=1)                                   # packing + engine + capture
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            tr.train(num_epochs=1, G_lr=2e-4, D_lr=2e-4, D_steps=1)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
        finally:
            sys.stdout = so
            sink.close()
        res[mode] = {"value": round(782 * 64 / dt, 1), "ms_per_step": round(dt / 782 * 1e3, 4)}
    res["api"] = "ns_gan.NSGANTrainer(...).train(num_epochs=1): 782 steps of B=64 over N=50000, wall clock around the call"
    return res


def bench_parity_mode(args, bits, N, rank, timed):
    """The fp32-grade operand mode (split-bf16, 3 tensor-core passes per product) on the headline config."""
    import gm_b200
    if not getattr(gm_b200, "HAS_SPLIT_PRECISION", False):
        return None
    B = DEFAULT_BATCH["ns"]
    wl = Workload("ns", B, bits, N, rank, 1, None, prec="split")
    for _ in range(3):
        wl.step()
    k = min(args.steps, 10)
    ms = timed(lambda i: wl.step(), k)
    out = {"value": round(B * k / (ms * 1e-3), 1), "unit": "images/s", "ms_per_step": round(ms / k, 4), "steps": k,
           "dtype": "bf16x3 (hi+lo split operands, fp32-grade products)", "losses_last_step": wl.losses()}
    del wl
    return out


# ------------------------------------------------------------------------------------------------
# the reference's own implementation (oracle/_ref byte code of src/ns_gan.py; oracle/ref_runner.py)
# ------------------------------------------------------------------------------------------------
def run_ref_runner(batch, steps, warmup, device="cpu", pool=0, prefetched=False, budget=150.0, threads=0, timeout=900):
    cmd = [sys.executable, os.path.join(ROOT, "oracle", "ref_runner.py"), "--batch", str(batch), "--steps", str(steps),
           "--warmup", str(warmup), "--device", device, "--budget", str(budget)]
    if pool:
        cmd += ["--pool", str(pool)]
    if prefetched:
        cmd += ["--prefetched"]
    if threads:
        cmd += ["--threads", str(threads)]
    env = dict(os.environ)
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "MASTER_ADDR", "MASTER_PORT"):
        env.pop(k, None)
    try:
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, env=env, cwd=ROOT)
    except subprocess.TimeoutExpired:
        return {"error": "timeout"}
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    if r.returncode != 0 or not lines:
        return {"error": (r.stderr or r.stdout)[-300:]}
    return json.loads(lines[-1])


def cpu_baseline():
    """The reference's own NSGANTrainer.train on this box's host cores (oracle/ref_runner.py), bounded samples."""
    c0 = run_ref_runner(64, 782, 20, pool=50000)                       # BASELINE configs[0]: one full N=50000 epoch at B=64
    c0c = run_ref_runner(64, 300, 20, pool=50000, prefetched=True)     # compute-only (no per-step DataLoader fetch)
    big = run_ref_runner(65536, 3, 1, budget=30.0)
    gpu64 = run_ref_runner(64, 782, 50, device="cuda", pool=50000)     # the same reference file through its own to_cuda path
    gpubig = run_ref_runner(65536, 10, 3, device="cuda")
    return {"value": c0.get("images_per_s"), "unit": "images/s", "cores": c0.get("threads"), "host_cores": c0.get("host_cores"),
            "kind": c0.get("kind", "reference"),
            "sample": "BASELINE configs[0]: the reference's NSGANTrainer.train, B=64, all 782 steps of one N=50000 epoch incl. its "
                      "per-step shuffling DataLoader fetch, %.1f s" % c0.get("seconds", float("nan")),
            "compute_only_b64": c0c.get("images_per_s"),
            "large_batch": {"batch": big.get("batch"), "value": big.get("images_per_s"), "seconds": big.get("seconds"), "steps": big.get("steps"),
                            "threads": big.get("threads")},
            "reference_on_b200_eager": {"what": "the same reference file through its own to_cuda path (torch eager, cuBLAS): SURVEY 8d secondary bar",
                                        "b64": gpu64.get("images_per_s", gpu64.get("error")), "b64_ms_per_step": gpu64.get("ms_per_step"),
                                        "b65536": gpubig.get("images_per_s", gpubig.get("error")), "b65536_ms_per_step": gpubig.get("ms_per_step"),
                                        "b65536_batch": gpubig.get("batch")},
            "errors": [r["error"] for r in (c0, c0c, big) if "error" in r] or None}


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the same step on the host
    cores (rank 0 only), same metric/config; a step is bounded by halving the batch until K steps fit the budget."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    B = args.batch or DEFAULT_BATCH["ns"]
    r = run_ref_runner(B, args.steps, args.warmup, budget=120.0)
    if "error" in r:
        print(json.dumps({"impl": "reference", "unavailable": "reference runner failed: " + r["error"][-200:]}))
        return
    ips, batch = r["images_per_s"], r["batch"]
    out = {"impl": "reference", "metric": METRIC, "value": ips, "unit": "images/s", "n_gpus": world,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"],
           "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": "NSGAN MLP (D 784-400-1, G 20-400-784), BASELINE configs[1] on host CPU: the reference's own "
                                  "NSGANTrainer.train (autograd + 2x Adam + per-step DataLoader fetch), batch %d per step%s"
                                  % (batch, "" if batch == B else " (bounded sample of the %d-image step)" % B),
                      "global_batch": batch, "parallelism": "cpu"},
           "cpu_baseline": {"value": ips, "unit": "images/s", "cores": r["threads"], "host_cores": r["host_cores"], "kind": r["kind"],
                            "sample": "%d steps of batch %d, %.1f s, %d threads" % (args.steps, batch, r["seconds"], r["threads"])},
           "e2e": {"value": ips, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--batch", type=int, default=0, help="images per GPU per step (default: the workload's BASELINE batch)")
    ap.add_argument("--workload", default="ns", choices=["ns", "wgp", "vae", "dcgan"])
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--headline-only", action="store_true", help="skip the other workloads / trainer / small-batch legs")
    ap.add_argument("--no-parity-mode", action="store_true", help="skip the split-precision leg")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the last step's losses and updated "
                                                         "parameters as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
