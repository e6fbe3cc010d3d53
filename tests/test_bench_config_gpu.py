"""Parity at the BENCHED settings (BASELINE configs[1..3]): 1-bit packed resident pool + the in-kernel
permutation sampler + in-kernel Philox noise + lazy gradients (gather fused into Adam), at B = 65536
(NSGAN, WGAN-GP) and B = 131072 (VAE) — checked against a plain PyTorch fp32 autograd evaluation of the
reference's formulas on the GPU, fed with exactly the indices / noise the kernels drew.

Also the statistical tests of the on-device Philox draws (compute_noise, src/ns_gan.py:218-220, and the
VAE's eps, src/vae.py:104) and of the sampler.  Measured errors go to gpurun_out/parity_bench_configs.json."""
import ctypes as C
import json
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
X, H, Z = 784, 400, 20
_REPORT = {}

# norm-relative bound on every gradient tensor vs fp32 autograd: north_star's 1e-3 in the fp32-grade
# split-operand mode; the bf16-operand speed mode carries the operands' 2^-9 rounding (measured values in
# gpurun_out/parity_bench_configs.json)
TOL = {"split": 1e-3, "bf16": 8e-3}
TOL_LOSS = 1e-3


def _dump():
    os.makedirs("gpurun_out", exist_ok=True)
    with open("gpurun_out/parity_bench_configs.json", "w") as f:
        json.dump(_REPORT, f, indent=1, sort_keys=True)


def _precisions():
    import gm_b200
    return ["bf16", "split"] if gm_b200.HAS_SPLIT_PRECISION else ["bf16"]


def _nrel(a, b):
    a, b = a.double().reshape(-1), b.double().reshape(-1)
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def _pool(n, seed=3435):
    g = torch.Generator(device="cuda").manual_seed(seed)
    nb = n * X // 8
    bits = torch.randint(0, 256, (nb,), device="cuda", dtype=torch.uint8, generator=g)
    bits &= torch.randint(0, 256, (nb,), device="cuda", dtype=torch.uint8, generator=g)
    bits &= torch.randint(0, 256, (nb,), device="cuda", dtype=torch.uint8, generator=g)
    return bits.view(n, X // 8)


def _unpack(bits_rows):
    w = torch.tensor([128, 64, 32, 16, 8, 4, 2, 1], device="cuda", dtype=torch.uint8)
    return ((bits_rows.unsqueeze(-1) & w) != 0).reshape(bits_rows.shape[0], -1).float()


def _gan_engine(variant, B, prec):
    import gm_b200
    import torch.nn as nn
    eng = gm_b200.GanEngine(X, H, Z, max_batch=B, variant=variant, d_out_act="relu" if variant == "wgp" else "sigmoid", precision=prec)
    torch.manual_seed(1234)
    g1, g2, d1, d2 = nn.Linear(Z, H), nn.Linear(H, X), nn.Linear(X, H), nn.Linear(H, 1)
    eng.load(0, [g1.weight.data, g1.bias.data, g2.weight.data, g2.bias.data])
    eng.load(1, [d1.weight.data, d1.bias.data, d2.weight.data, d2.bias.data])
    return eng


def test_philox_noise_statistics_and_disjoint_streams():
    """stage_noise_kernel's Philox N(0,1): moments, determinism, and independence across step / D-vs-G / seed."""
    eng = _gan_engine("ns", 65536, "bf16")
    B = 65536
    a = eng.debug_noise(B, seed=1000003, step=5)
    n = a.numel()
    se = 1.0 / np.sqrt(n)
    assert abs(float(a.mean())) < 5 * se
    assert abs(float(a.var()) - 1.0) < 0.01                 # bf16 rounding of the operand adds ~2^-18 relative variance
    assert abs(float((a ** 4).mean()) / float(a.var()) ** 2 - 3.0) < 0.05
    assert abs(float((a ** 3).mean())) < 0.02
    assert 4.0 < float(a.abs().max()) < 6.5                 # tails exist and are sane for 1.3 M draws
    assert torch.equal(a, eng.debug_noise(B, seed=1000003, step=5))          # same (seed, step): same numbers
    others = {"next_step": eng.debug_noise(B, seed=1000003, step=6), "g_step": eng.debug_noise(B, seed=1000003, step=5, g_step=True),
              "other_rank_seed": eng.debug_noise(B, seed=1000004, step=5)}
    rep = {"mean": float(a.mean()), "var": float(a.var())}
    for k, b in others.items():
        corr = float((a * b).mean())
        rep["corr_" + k] = corr
        assert abs(corr) < 5 * se, (k, corr)
        assert float((a == b).float().mean()) < 0.01, k
    # rows are independent too (row r vs row r+1 of the same draw)
    assert abs(float((a[:-1] * a[1:]).mean())) < 5 * se
    _REPORT["philox_noise"] = rep
    _dump()


def test_sampler_draws_distinct_rows_and_matches_host_evaluation():
    import gm_b200
    eng = _gan_engine("ns", 4096, "bf16")
    N, B = 50000, 4096
    eng.set_sampler(N, 77)
    idx = eng.sample_indices(B, step=3)
    host = np.empty(B, dtype=np.int32)
    assert gm_b200.lib().gm_sampler_indices_host(N, 77, 3, 0, B, C.c_void_p(host.ctypes.data)) == 0
    assert np.array_equal(idx.cpu().numpy(), host)
    assert idx.unique().numel() == B and int(idx.max()) < N and int(idx.min()) >= 0
    assert not torch.equal(idx, eng.sample_indices(B, step=4))
    # the staging kernel reads exactly these rows: sampled step == explicit gather of the same indices, bit for bit
    bits = _pool(N)
    z = torch.randn(B, Z, device="cuda")
    l1 = eng.d_grad(bits, fmt="bits", batch=B, noise=z, step=3).item()
    g1 = eng.grads[1].clone()
    eng.set_sampler(0)
    l2 = eng.d_grad(bits, fmt="bits", gather_idx=idx, noise=z, step=3).item()
    assert l1 == l2 and torch.equal(g1, eng.grads[1])
    with pytest.raises(gm_b200.GmError, match="pool"):
        eng.set_sampler(100, 1)
        eng.d_grad(bits, fmt="bits", batch=B, noise=z)


def _torch_nets(eng):
    Wg1, bg1, Wg2, bg2 = [t.clone().requires_grad_() for t in eng.views(0)]
    Wd1, bd1, Wd2, bd2 = [t.clone().requires_grad_() for t in eng.views(1)]
    relu_out = eng.variant == "wgp"

    def Gf(zz):
        return torch.sigmoid(torch.relu(zz @ Wg1.t() + bg1) @ Wg2.t() + bg2)

    def Df(xx):
        s = torch.relu(xx @ Wd1.t() + bd1) @ Wd2.t() + bd2
        return torch.relu(s) if relu_out else torch.sigmoid(s)
    return (Wg1, bg1, Wg2, bg2), (Wd1, bd1, Wd2, bd2), Gf, Df


@pytest.mark.parametrize("prec", _precisions())
@pytest.mark.parametrize("variant", ["ns", "wgp"])
def test_gan_step_at_bench_settings_matches_fp32_autograd(variant, prec):
    """configs[1] / configs[2]: B = 65536, bits pool + sampler + Philox noise + lazy gradients."""
    import gm_b200
    torch.backends.cuda.matmul.allow_tf32 = False
    B, N, seed, step = 65536, 4 * 65536, 1000003, 2
    eng = _gan_engine(variant, B, prec)
    bits = _pool(N)
    eng.set_sampler(N, seed)
    eng.set_lazy_grads(True)
    hp = gm_b200.AdamHP.make(1e-4)
    idx = eng.sample_indices(B, step).long()
    x = _unpack(bits[idx])
    zd = eng.debug_noise(B, seed, step)
    zg = eng.debug_noise(B, seed, step, g_step=True)
    eps = torch.rand(B, device="cuda") if variant == "wgp" else None
    Gp, Dp, Gf, Df = _torch_nets(eng)
    if variant == "ns":
        Ld_ref = -torch.mean(torch.log(Df(x) + 1e-8) + torch.log(1 - Df(Gf(zd)) + 1e-8))
    else:
        fake = Gf(zd).detach()
        xh = (eps.view(-1, 1) * x + (1 - eps.view(-1, 1)) * fake).requires_grad_()
        gr = torch.autograd.grad(Df(xh), xh, torch.ones(B, 1, device="cuda"), create_graph=True, retain_graph=True)[0]
        Ld_ref = torch.mean(Df(fake)) - torch.mean(Df(x)) + 10.0 * torch.mean((gr.norm(2, dim=1) - 1) ** 2)   # src/w_gp_gan.py:215-218
    gd = torch.cat([t.reshape(-1) for t in torch.autograd.grad(Ld_ref, Dp)])
    Ld = eng.d_grad(bits, fmt="bits", batch=B, aux=eps, seed=seed, step=step).item()
    eng.apply(1, hp)                      # lazy: the flat gradient is formed inside this Adam kernel
    flatD = eng.grads[1].clone()
    # the G step sees the UPDATED discriminator (src/ns_gan.py:139 precedes :151)
    Gp, Dp, Gf, Df = _torch_nets(eng)
    Lg_ref = -torch.mean(torch.log(Df(Gf(zg)) + 1e-8)) if variant == "ns" else -torch.mean(Df(Gf(zg)))
    gg = torch.cat([t.reshape(-1) for t in torch.autograd.grad(Lg_ref, Gp)])
    Lg = eng.g_grad(B, seed=seed, step=step).item()
    eng.apply(0, hp)
    flatG = eng.grads[0].clone()
    rep = {"D_loss": abs(Ld - Ld_ref.item()) / max(abs(Ld_ref.item()), 0.5), "G_loss": abs(Lg - Lg_ref.item()) / max(abs(Lg_ref.item()), 0.5),
           "gD": _nrel(flatD, gd), "gG": _nrel(flatG, gg)}
    # per-tensor errors (every gradient tensor, not only the flat norm)
    for net, flat, ref, names in ((1, flatD, gd, ["D.W1", "D.b1", "D.w2", "D.b2"]), (0, flatG, gg, ["G.W1", "G.b1", "G.W2", "G.b2"])):
        for nme, a, b in zip(names, eng.views(net, flat), eng.views(net, ref)):
            if float(b.norm()) > 0:
                rep[nme] = _nrel(a, b)
    _REPORT["%s_b65536_%s" % (variant, prec)] = rep
    _dump()
    assert rep["D_loss"] < TOL_LOSS and rep["G_loss"] < TOL_LOSS, rep
    for k, v in rep.items():
        if k not in ("D_loss", "G_loss"):
            assert v < TOL[prec], (k, v, rep)


@pytest.mark.parametrize("prec", _precisions())
def test_vae_step_at_bench_settings_matches_fp32_autograd(prec):
    """configs[3]: B = 131072, bits pool + epoch sampler + Philox eps."""
    import gm_b200
    import torch.nn as nn
    torch.backends.cuda.matmul.allow_tf32 = False
    B, N, seed, step = 131072, 2 * 131072, 77, 3
    eng = gm_b200.VaeEngine(X, H, Z, max_batch=B, precision=prec)
    torch.manual_seed(1234)
    mods = {"encoder.linear": nn.Linear(X, H), "encoder.mu": nn.Linear(H, Z), "encoder.log_var": nn.Linear(H, Z),
            "decoder.linear": nn.Linear(Z, H), "decoder.recon": nn.Linear(H, X)}
    t = {}
    for k, m in mods.items():
        t[k + ".weight"], t[k + ".bias"] = m.weight.data, m.bias.data
    eng.load(t)
    bits = _pool(N)
    eng.set_sampler(N, N // B, seed)
    losses = eng.grad(bits, fmt="bits", batch=B, seed=seed, step=step).clone()
    eps = eng.last_eps(B)
    se = 1.0 / np.sqrt(eps.numel())
    assert abs(float(eps.mean())) < 5 * se and abs(float(eps.var()) - 1) < 0.01          # the Philox eps are N(0,1)
    idx = eng.sample_indices(B, step, N // B, N, seed).long()
    assert idx.unique().numel() == B
    x = _unpack(bits[idx])
    P = {k: v.clone().requires_grad_() for k, v in eng.views().items()}
    h = torch.relu(x @ P["encoder.linear.weight"].t() + P["encoder.linear.bias"])
    mu = h @ P["encoder.mu.weight"].t() + P["encoder.mu.bias"]
    lv = h @ P["encoder.log_var.weight"].t() + P["encoder.log_var.bias"]
    zz = mu + eps * torch.exp(lv / 2)                                                   # src/vae.py:105
    out = torch.sigmoid(torch.relu(zz @ P["decoder.linear.weight"].t() + P["decoder.linear.bias"]) @ P["decoder.recon.weight"].t()
                        + P["decoder.recon.bias"])
    recon = torch.sum((x - out) ** 2)                                                   # src/vae.py:203
    kl = torch.sum(0.5 * (mu ** 2 + torch.exp(lv) - lv - 1))                            # src/vae.py:212
    grads = torch.autograd.grad(recon + kl, list(P.values()))
    rep = {"recon": abs(float(losses[0]) - recon.item()) / recon.item(), "kl": abs(float(losses[1]) - kl.item()) / kl.item()}
    gv = eng.views(eng.grads)
    for (k, _), gref in zip(P.items(), grads):
        rep[k] = _nrel(gv[k], gref)
    _REPORT["vae_b131072_%s" % prec] = rep
    _dump()
    assert rep["recon"] < TOL_LOSS, rep
    assert rep["kl"] < (TOL_LOSS if prec == "split" else 1e-2), rep
    for k, v in rep.items():
        if k not in ("recon", "kl"):
            assert v < (TOL[prec] if prec == "split" else 3e-2), (k, v, rep)


def test_graph_replay_matches_host_driven_steps():
    """Device-step mode + CUDA-graph replay (the small-batch regime): N replays == N host-driven steps, bit for bit
    (same sampler rounds, Philox streams and Adam bias corrections from the device counters)."""
    import gm_b200
    B, N, seed = 64, 50000, 4242
    bits = _pool(N)
    hp = gm_b200.AdamHP.make(2e-4)

    def host_driven(steps):
        eng = _gan_engine("ns", B, "bf16")
        eng.set_lazy_grads(True)
        eng.set_sampler(N, seed)
        for s in range(steps):
            eng.d_grad(bits, fmt="bits", batch=B, seed=seed, step=s)
            eng.apply(1, hp)
            eng.g_grad(B, seed=seed, step=s)
            eng.apply(0, hp)
        return eng
    ref = host_driven(3 + 5)
    eng = _gan_engine("ns", B, "bf16")
    step = gm_b200.GraphedGanStep(eng, bits, N, B, hp, hp, seed=seed, warmup=3)     # 3 eager warm-up steps + capture
    for _ in range(5 - 1):                                                           # the capture itself does not execute
        step()
    step()
    torch.cuda.synchronize()
    assert eng.device_steps() == [8, 8, 8, 8]
    step.close()
    assert eng.steps == [8, 8]
    for net in (0, 1):
        assert torch.equal(eng.params[net], ref.params[net]), net
        assert torch.equal(eng.exp_avg_sq[net], ref.exp_avg_sq[net])
    assert torch.equal(eng.loss_buf, ref.loss_buf)


def test_bench_dump_outputs_hold_the_last_timed_step(tmp_path):
    """bench.py --dump-outputs: the losses the JSON line reports for the last timed step and the updated parameters,
    float32 .npy files; a second run with the same arguments reproduces them bit for bit."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    runs = []
    for k in range(2):
        d = tmp_path / str(k)
        out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--steps", "2", "--warmup", "1", "--headline-only",
                              "--no-cpu", "--dump-outputs", str(d)], capture_output=True, text=True, timeout=600, cwd=root)
        assert out.returncode == 0, out.stderr[-3000:]
        line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
        runs.append((line, {f[:-len(".npy")]: np.load(d / f) for f in os.listdir(d)}))
    line, arrs = runs[0]
    names = [m + s for m in ("G.linear", "G.generate", "D.linear", "D.discriminate") for s in (".weight", ".bias")]
    assert line["steps"] == 2 and sorted(arrs) == sorted(["losses"] + names)
    assert all(a.dtype == np.float32 for a in arrs.values()) and sum(a.nbytes for a in arrs.values()) <= 64 << 20
    assert arrs["G.generate.weight"].shape == (X, H) and arrs["D.discriminate.weight"].shape == (1, H)
    np.testing.assert_array_equal(arrs["losses"], np.float32(line["losses_last_step"]))
    for name, a in runs[1][1].items():
        np.testing.assert_array_equal(a, arrs[name], err_msg=name)
