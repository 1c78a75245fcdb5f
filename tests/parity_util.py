"""Shared helpers for parity tests: build the B200 modules from a seed, run the CPU oracle on the same
state dict, compare outputs / buffers / gradients."""
import hashlib
import os

import torch

from oracle import dgmr_oracle as O

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
GOLDEN = os.path.join(GOLDEN_DIR, "c1_gan.pt")
C1 = dict(forecast_steps=4, output_shape=128, latent_channels=384, context_channels=192, batch=2)


def state_checksum(sd):
    tot, atot = 0.0, 0.0
    for k in sorted(sd):
        v = sd[k].double()
        tot += float(v.sum())
        atot += float(v.abs().sum())
    return [tot, atot]


def build_gan(cfg, seed=0, gamma=None):
    """Seeded construction on CPU (consumes the RNG exactly like the reference constructors)."""
    import skillful_nowcasting_b200 as B

    torch.manual_seed(seed)
    s = cfg["output_shape"]
    gen = B.Generator(
        B.ContextConditioningStack(input_channels=1, output_channels=cfg["context_channels"]),
        B.LatentConditioningStack(shape=(8, s // 32, s // 32), output_channels=cfg["latent_channels"]),
        B.Sampler(forecast_steps=cfg["forecast_steps"], latent_channels=cfg["latent_channels"],
                  context_channels=cfg["context_channels"]))
    disc = B.Discriminator(input_channels=1)
    if gamma is not None:
        with torch.no_grad():
            gen.latent_stack.att_block.gamma.fill_(gamma)
    return gen, disc


def c1_inputs(cfg=C1, seed=1):
    torch.manual_seed(seed)
    s, b, t = cfg["output_shape"], cfg["batch"], cfg["forecast_steps"]
    return torch.rand(b, 4, 1, s, s), torch.rand(b, t, 1, s, s)


def tensor_digest(t):
    """dtype, shape and SHA-256 of the raw bytes: equal digests <=> torch.equal (bitwise), without storing the tensor."""
    t = t.detach().cpu().contiguous()
    return f"{t.dtype} {tuple(t.shape)} {hashlib.sha256(t.reshape(-1).view(torch.uint8).numpy().tobytes()).hexdigest()}"


def rel_err(a, b):
    """max |a-b| / max |b| (the 'rel' used for all tolerances in these tests).

    `b` may also be a sampled fixture entry (tests/golden/make_golden.py: sample_tensor), which holds b's values at a fixed random
    subset of its elements plus its max |b|, L2 norm and sum.  Then the error is the larger of the elementwise error on the subset and
    three whole-tensor terms |max|a| - max|b||, |‖a‖ - ‖b‖| / sqrt(n) and |sum a - sum b| / n (each over max |b|).  Every term is at most
    the exact max |a-b| / max |b|, so a sampled comparison never fails where the full one would pass."""
    if isinstance(b, dict):
        a = a.detach().double().cpu().flatten()
        assert list(a.shape) == [b["numel"]], (a.shape, b["numel"])
        n, scale = a.numel(), max(b["absmax"], 1e-30)
        idx, val = torch.as_tensor(b["idx"]).long(), torch.as_tensor(b["val"]).double()
        terms = ((a[idx] - val).abs().max().item(), abs(a.abs().max().item() - b["absmax"]),
                 abs(a.norm().item() - b["norm"]) / n ** 0.5, abs(a.sum().item() - b["sum"]) / n)
        return max(terms) / scale
    a, b = a.detach().float().cpu(), b.detach().float().cpu()
    return (a - b).abs().max().item() / max(b.abs().max().item(), 1e-30)


def oracle_gan_forward(g_state, d_state, x, y, cfg, training, seed):
    """Oracle forward (+ losses, + grads in training) on cloned state.  Returns dict like the golden fixture."""
    gs = O.clone_state(g_state, requires_grad=training)
    ds = O.clone_state(d_state, requires_grad=training)
    s = cfg["output_shape"]
    torch.manual_seed(seed)
    out = O.generator(gs, x, cfg["forecast_steps"], (8, s // 32, s // 32), training)
    scores = O.discriminator(ds, torch.cat([torch.cat([x, y], 1), torch.cat([x, out], 1)], 0), training)
    b = x.shape[0]
    sr, sg = scores[:b], scores[b:]
    d_loss = O.loss_hinge_disc(sg[:, 0:1], sr[:, 0:1]) + O.loss_hinge_disc(sg[:, 1:2], sr[:, 1:2])
    grid = O.grid_cell_loss(out, y)
    g_loss = O.loss_hinge_gen(sg) + 20.0 * grid
    res = dict(out=out.detach(), scores=scores.detach(), d_loss=d_loss.detach(), grid=grid.detach(), g_loss=g_loss.detach(),
               g_state=gs, d_state=ds)
    if training:
        dn, gn = O._trainable(ds), O._trainable(gs)
        dg = torch.autograd.grad(d_loss, [ds[k] for k in dn], retain_graph=True, allow_unused=True)
        gg = torch.autograd.grad(g_loss, [gs[k] for k in gn], allow_unused=True)
        res["d_grads"] = {k: g for k, g in zip(dn, dg) if g is not None}
        res["g_grads"] = {k: g for k, g in zip(gn, gg) if g is not None}
    return res


def module_gan_forward(gen, disc, x, y, training, seed, device):
    """Same computation through the B200 modules (whatever backend is active)."""
    from skillful_nowcasting_b200 import losses, ops

    gen.train(training)
    disc.train(training)
    for p in list(gen.parameters()) + list(disc.parameters()):
        p.grad = None
    x, y = x.to(device), y.to(device)
    torch.manual_seed(seed)
    out = gen(x)
    scores = disc(torch.cat([torch.cat([x, y], 1), torch.cat([x, out], 1)], 0))
    b = x.shape[0]
    d_loss = losses.loss_hinge_disc_both(scores)
    grid = ops.grid_cell(out, y, 24.0)
    g_loss = losses.loss_hinge_gen(scores[b:]) + 20.0 * grid
    res = dict(out=out.detach(), scores=scores.detach(), d_loss=d_loss.detach(), grid=grid.detach(), g_loss=g_loss.detach())
    if training:
        dn, gn = dict(disc.named_parameters()), dict(gen.named_parameters())
        dg = torch.autograd.grad(d_loss, list(dn.values()), retain_graph=True, allow_unused=True)
        gg = torch.autograd.grad(g_loss, list(gn.values()), allow_unused=True)
        res["d_grads"] = {k: g for k, g in zip(dn, dg) if g is not None}
        res["g_grads"] = {k: g for k, g in zip(gn, gg) if g is not None}
    return res


def compare_grads(got, ref, tol_norm, tol_head, zero_floor):
    """ref entries are either tensors (oracle) or fixture summaries {norm, sum, head[, full]}.
    Gradients whose reference norm is below `zero_floor` x the largest norm are mathematically zero
    (conv bias in front of BatchNorm) and only checked to be comparably small."""
    norms = {k: (float(v.double().norm()) if torch.is_tensor(v) else v["norm"]) for k, v in ref.items()}
    big = max(norms.values())
    # A gradient the B200 path does not produce at all (None = exactly zero: bias / spectral-norm scale of a conv that feeds a train-mode
    # BatchNorm, ops._ConvBNRelu) must be one of the mathematically-zero ones on the reference side (rounding noise there).
    assert set(got) <= set(ref), (set(got) - set(ref))
    for k in set(ref) - set(got):
        assert norms[k] < zero_floor * big, f"{k}: no gradient produced but the reference has norm {norms[k]:.3e} (largest {big:.3e})"
    worst = []
    for k, g in got.items():
        g = g.detach().float().cpu()
        rn = norms[k]
        gn = float(g.double().norm())
        if rn < zero_floor * big:
            assert gn < 10 * zero_floor * big, f"{k}: expected ~0 gradient, got norm {gn:.3e}"
            continue
        e_norm = abs(gn - rn) / rn
        if torch.is_tensor(ref[k]):
            r = ref[k].detach().float()
            e_head = (g - r).abs().max().item() / max(r.abs().max().item(), 1e-30)
        else:
            r = ref[k]["head"]
            e_head = (g.flatten()[:64] - r).abs().max().item() / max(r.abs().max().item(), 1e-30)
        worst.append((max(e_norm / tol_norm, e_head / tol_head), k, e_norm, e_head))
    worst.sort(reverse=True)
    assert not worst or worst[0][0] <= 1.0, f"gradient mismatch (ratio, name, norm err, elem err): {worst[:5]}"
    return worst[:3]


def assert_grads_close(names, got, ref, tol, floor=1e-5, tol_l2=None):
    """Element-wise gradient comparison for block tests.  Gradients that are mathematically zero (a conv bias in front
    of a training-mode BatchNorm) show up as rounding noise on both sides: they are only required to stay tiny."""
    pairs = [(n, a, b) for n, a, b in zip(names, got, ref)]
    scale = max([float(b.abs().max()) for _, _, b in pairs if b is not None and b.numel()] + [1e-30])
    for n, a, b in pairs:
        if a is None and b is not None:   # not produced at all = exactly zero: only legitimate where the reference holds rounding noise
            assert float(b.abs().max()) < floor * scale, f"{n}: no gradient produced but the reference has max {float(b.abs().max()):.3e}"
            continue
        assert (a is None) == (b is None), n
        if a is None or not b.numel():
            continue
        if float(b.abs().max()) < floor * scale:
            assert float(a.abs().max()) < 10 * floor * scale, f"{n}: expected ~0 gradient"
        else:
            e = rel_err(a, b)
            assert e < tol, f"{n}: rel err {e:.3e} > {tol}"
            if tol_l2 is not None:  # ||a-b||_2 / ||b||_2: insensitive to the handful of ReLU-mask flips tf32 rounding causes
                e2 = float((a.double().cpu() - b.double()).norm() / b.double().norm())
                assert e2 < tol_l2, f"{n}: L2 rel err {e2:.3e} > {tol_l2}"


def global_grad_error(got, ref):
    """||g - r|| / ||r|| over ALL parameters at once (oracle tensors only): the coarse end-to-end check used where
    per-parameter comparison is dominated by chaotic amplification (train-mode TF32 end to end).  A gradient the path does not
    produce (None) counts as zero."""
    num = den = 0.0
    for k, r in ref.items():
        r = r.detach().double()
        g = got[k].detach().double().cpu() if k in got else torch.zeros_like(r)
        num += float(((g - r) ** 2).sum())
        den += float((r ** 2).sum())
    return (num / max(den, 1e-300)) ** 0.5


# ------------------------------------------------------------------------------------------------ one full GAN step
def oracle_gan_step(g_state, d_state, x, y, cfg, seed, generation_steps=1):
    """oracle.gan_step on cloned state: returns losses, post-step parameters / buffers and the Adam moments."""
    gs = O.clone_state(g_state, requires_grad=True)
    ds = O.clone_state(d_state, requires_grad=True)
    gn, dn = O._trainable(gs), O._trainable(ds)
    g_opt = O.AdamState([gs[k] for k in gn], lr=5e-5)
    d_opt = O.AdamState([ds[k] for k in dn], lr=2e-4)
    s = cfg["output_shape"]
    torch.manual_seed(seed)
    losses = O.gan_step(gs, ds, g_opt, d_opt, x, y, cfg["forecast_steps"], (8, s // 32, s // 32), generation_steps=generation_steps)
    return dict(losses=losses, g_state=gs, d_state=ds, g_names=gn, d_names=dn,
                g_m=dict(zip(gn, g_opt.m)), g_v=dict(zip(gn, g_opt.v)), d_m=dict(zip(dn, d_opt.m)), d_v=dict(zip(dn, d_opt.v)),
                g_t=g_opt.t, d_t=d_opt.t)


def module_gan_step(gen, disc, x, y, seed, device, generation_steps=1, d_phase_generator=None):
    """training.gan_step through the B200 modules and the fused Adam: the same quantities as oracle_gan_step."""
    from skillful_nowcasting_b200.training import Adam, gan_step

    gen.train(); disc.train()
    g_opt = Adam(gen.parameters(), lr=5e-5, betas=(0.0, 0.999))
    d_opt = Adam(disc.parameters(), lr=2e-4, betas=(0.0, 0.999))
    torch.manual_seed(seed)
    losses = gan_step(gen, disc, g_opt, d_opt, x.to(device), y.to(device), generation_steps=generation_steps, d_phase_generator=d_phase_generator)

    def moments(opt, module):
        names = [n for n, _ in module.named_parameters()]
        sd = opt.state_dict()["state"]
        return ({n: sd[i]["exp_avg"] for i, n in enumerate(names)}, {n: sd[i]["exp_avg_sq"] for i, n in enumerate(names)})

    g_m, g_v = moments(g_opt, gen)
    d_m, d_v = moments(d_opt, disc)
    return dict(losses=losses, g_state=gen.state_dict(), d_state=disc.state_dict(), g_m=g_m, g_v=g_v, d_m=d_m, d_v=d_v,
                g_t=g_opt.steps, d_t=d_opt.steps, requires_grad_after=all(p.requires_grad for p in disc.parameters()))


def _l2(got, ref, names):
    num = den = 0.0
    for k in names:
        a, b = got[k].detach().double().cpu(), ref[k].detach().double()
        num += float(((a - b) ** 2).sum())
        den += float((b ** 2).sum())
    return (num / den) ** 0.5 if den > 0 else num ** 0.5   # all-zero reference (saturated hinge: zero gradient): absolute


# bounds for compare_gan_step.  FP32: fp32 arithmetic on both sides (SIMT kernels, 3xTF32 parity mode, the host emulator) -- set from
# the noise floor "oracle with 8 threads vs oracle with 3 threads" (g_m 5e-3, g_update 3.5e-3, d_uv 2.6e-4, d_bn 7.7e-3) times ~10;
# TF32: 1xTF32 operands end to end through batch-stat BatchNorm at fresh init (chaotic, SURVEY.md section 7).
GAN_STEP_TOL_FP32 = dict(d_loss=2e-3, g_loss=2e-3, grid_loss=2e-3, g_m=5e-2, g_v=1e-1, g_update=5e-2, g_uv=2e-4, g_bn=2e-3,
                         d_m=5e-2, d_v=1e-1, d_update=5e-2, d_uv=2e-2, d_bn=5e-2)
# d_uv in 1xTF32 mode: the discriminator's u, v after the step are power-iteration vectors of weights that already moved by one TF32-noisy Adam
# update and were iterated again by the second D pass -- for a weight with two close leading singular values that is arbitrarily ill-conditioned
# (measured across round-2 runs of the same test: 5e-2, 8e-2, 5e-1); it is judged in the fp32 and 3xTF32 modes (7e-4 / 9e-3 against 2e-2), not here.
GAN_STEP_TOL_TF32 = dict(d_loss=5e-2, g_loss=5e-2, grid_loss=5e-2, g_m=0.3, g_v=0.6, g_update=0.35, g_uv=2e-4, g_bn=5e-2,
                         d_m=0.3, d_v=0.6, d_update=0.35, d_uv=2.0, d_bn=0.2)


def gan_step_report(got, ref, g0, d0):
    """Everything one GAN step leaves behind, as error numbers (see compare_gan_step for how they are judged)."""
    rep = {}
    for k in ("d_loss", "g_loss", "grid_loss"):
        rep[k] = rel_err(got["losses"][k], ref["losses"][k])
    for net, names, s0 in (("g", ref["g_names"], g0), ("d", ref["d_names"], d0)):
        rep[f"{net}_m"] = _l2(got[f"{net}_m"], ref[f"{net}_m"], names)
        rep[f"{net}_v"] = _l2(got[f"{net}_v"], ref[f"{net}_v"], names)
        num = den = 0.0
        for k in names:
            p, pr, p0 = got[f"{net}_state"][k].detach().double().cpu(), ref[f"{net}_state"][k].detach().double(), s0[k].double()
            num += float((p - pr).abs().sum())
            den += float((pr - p0).abs().sum())
        rep[f"{net}_update"] = num / max(den, 1e-300)
        rep[f"{net}_uv"] = rep[f"{net}_bn"] = 0.0
        for k, v in ref[f"{net}_state"].items():
            g = got[f"{net}_state"][k]
            if k.endswith("._u") or k.endswith("._v"):
                rep[f"{net}_uv"] = max(rep[f"{net}_uv"], rel_err(g, v))
            elif "running_" in k:
                rep[f"{net}_bn"] = max(rep[f"{net}_bn"], rel_err(g, v))
            elif "num_batches" in k:
                assert int(g) == int(v), k
    return rep


def compare_gan_step(got, ref, g0, d0, tol):
    """Judge one GAN step against oracle.gan_step.  `tol` maps the report's keys to bounds:
      d_loss / g_loss / grid_loss  relative error of the three logged losses;
      g_m, d_m / g_v, d_v          Adam exp_avg (= the last gradient, beta1 = 0) / exp_avg_sq, global relative L2 over all parameters;
      g_update, d_update           parameters, through the update they received: with beta1 = 0 the first Adam step moves every element
                                   by lr * sign(g) (|g| >> eps), so they are compared by  sum|p - p_ref| / sum|p_ref - p_0|  (a flipped sign
                                   of a ~0 gradient element costs 2 units of lr there);
      g_uv, d_uv / g_bn, d_bn      mutated buffers: spectral-norm u, v / BatchNorm running statistics (max rel err over the buffers);
                                   num_batches_tracked, the Adam step counts and the discriminator's requires_grad flags must be exact.
    The discriminator takes TWO updates per step: everything after the first one (second forward, its gradient, the buffers) runs
    on weights that moved by lr * sign(g), so sign flips of near-zero gradient elements are amplified there -- the d_* bounds are
    looser than the g_* ones even for fp32 arithmetic (the fp32 emulator-vs-oracle numbers are recorded in tests/test_host_logic.py)."""
    rep = gan_step_report(got, ref, g0, d0)
    assert got["g_t"] == ref["g_t"] == 1 and got["d_t"] == ref["d_t"] == 2
    assert got["requires_grad_after"], "gan_step left discriminator parameters frozen"
    bad = {k: (v, tol[k]) for k, v in rep.items() if v >= tol[k]}
    assert not bad, f"GAN step mismatch (value, bound): {bad}\nfull report: {rep}"
    return rep


# ------------------------------------------------------------------------------------------------ discriminators, separately
def run_discriminator_case(which, training, device, tol_fwd, tol_grad_l2=None, cfg=C1, seed=5):
    """SpatialDiscriminator / TemporalDiscriminator alone against the oracle (ref: dgmr/discriminators.py:104-138, 196-232) on a
    [2B, T_in + T, 1, S, S] batch of real || "generated" sequences; forward scores and (training) the global gradient error.

    The seed matters: with seed 3 (used until round 2) the temporal case sits ON a ReLU kink of the head -- relative noise of 1e-7 injected into the
    fp32 host emulator's convolution outputs flips the global gradient error between 2.9e-3 and 6.1e-2 (bimodal, nothing in between), which made the
    device test depend on the summation order of unrelated kernels.  Seed 5 is a generic point: 2.4e-5 for the emulator, growing smoothly with
    injected noise (6e-5 at 1e-6)."""
    import skillful_nowcasting_b200 as B

    torch.manual_seed(seed)
    mod = B.SpatialDiscriminator(input_channels=1) if which == "spatial" else B.TemporalDiscriminator(input_channels=1)
    pfx = "spatial_discriminator." if which == "spatial" else "temporal_discriminator."
    st = O.clone_state({pfx + k: v for k, v in mod.state_dict().items()}, requires_grad=training)
    s, b, t = cfg["output_shape"], cfg["batch"], 4 + cfg["forecast_steps"]
    x = torch.rand(2 * b, t, 1, s, s)
    mod.train(training)
    torch.manual_seed(seed + 1)
    if which == "spatial":
        ref = O.spatial_discriminator(st, pfx[:-1], x, training)
    else:
        ref = O.temporal_discriminator(st, pfx[:-1], x, training)
    mod.to(device)
    torch.manual_seed(seed + 1)
    got = mod(x.to(device))
    e = rel_err(got, ref)
    out = dict(fwd=e, ref=ref.detach().flatten().tolist(), got=got.detach().flatten().cpu().tolist())
    assert got.shape == ref.shape
    assert e < tol_fwd, (which, "scores", e, out["ref"], out["got"])
    if training:
        w = torch.randn_like(ref)
        names = [k for k in st if st[k].requires_grad]
        rg = torch.autograd.grad((ref * w).sum(), [st[k] for k in names], allow_unused=True)
        params = dict(mod.named_parameters())
        mg = torch.autograd.grad((got * w.to(device)).sum(), [params[k[len(pfx):]] for k in names], allow_unused=True)
        keep = [k for k, g in zip(names, rg) if g is not None]
        gd = {k: g for k, g in zip(names, mg) if g is not None}
        rd = {k: g for k, g in zip(names, rg) if g is not None}
        assert set(gd) == set(rd)
        out["grad_l2"] = _l2(gd, rd, keep)
        assert out["grad_l2"] < tol_grad_l2, (which, "gradients", out["grad_l2"])
        for k, v in mod.state_dict().items():
            r = st[pfx + k]
            if k.endswith("._u") or k.endswith("._v"):
                assert rel_err(v, r) < 2e-4, k
            elif "running_" in k:
                assert rel_err(v, r) < max(tol_fwd, 1e-3), k
    return out
