"""Generate golden fixtures by running the UNMODIFIED reference (openclimatefix/skillful_nowcasting) on CPU:

    DGMR_REFERENCE=<checkout of the reference> python tests/golden/make_golden.py

Writes, under tests/golden/:
  c1_gan.pt                      BASELINE config C1 through the reference's generator, discriminators and losses (eval and
                                 train): outputs, losses, gradient summaries, mutated buffers, and a digest of every tensor of
                                 the seeded construction
  reference_blocks.pt            each building block of the reference on small seeded inputs (tests/test_oracle.py)
  reference_wrapper_losses.json  the losses the reference's own `DGMR.training_step` logs (tests/test_host_logic.py)
The reference has no golden vectors of its own for the hot path (SURVEY.md 8c), so these fixtures — outputs of the reference
itself on seeded inputs — are what pins the oracle and, through it, the CUDA path; the tests need no copy of the reference.
The C1 generator outputs and the buffers of more than 1024 elements are stored as a fixed random sample of their elements plus
whole-tensor statistics (sample_tensor; parity_util.rel_err compares against that form), which keeps every file below 1 MB.

Import bypass (SURVEY.md 8c): `import dgmr` fails because dgmr/__init__.py pulls in
pytorch_lightning; registering a bare package object lets the hot-path sub-modules import.
"""
import json
import os
import sys
import types

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path[:0] = [os.path.dirname(HERE), os.path.dirname(os.path.dirname(HERE))]
from parity_util import tensor_digest  # noqa: E402

REF = os.environ.get("DGMR_REFERENCE", "")


def import_reference():
    if "dgmr" in sys.modules and getattr(sys.modules["dgmr"], "__graft_ref__", False):
        return sys.modules["dgmr"]
    for k in [k for k in sys.modules if k == "dgmr" or k.startswith("dgmr.")]:
        del sys.modules[k]
    m = types.ModuleType("dgmr")
    m.__path__ = [os.path.join(REF, "dgmr")]
    m.__graft_ref__ = True
    sys.modules["dgmr"] = m
    if "pytorch_msssim" not in sys.modules:
        try:
            import pytorch_msssim  # noqa: F401
        except Exception:
            stub = types.ModuleType("pytorch_msssim")
            stub.SSIM = type("SSIM", (torch.nn.Module,), {})
            stub.MS_SSIM = type("MS_SSIM", (torch.nn.Module,), {})
            sys.modules["pytorch_msssim"] = stub
    import dgmr.common  # noqa: F401
    import dgmr.discriminators  # noqa: F401
    import dgmr.generators  # noqa: F401
    import dgmr.layers  # noqa: F401
    import dgmr.losses  # noqa: F401
    return m


# BASELINE.json configs[0]: the reference's own CPU smoke config (tests/test_model.py:285-306).
C1 = dict(forecast_steps=4, output_shape=128, latent_channels=384, context_channels=192, batch=2)


def state_checksum(sd):
    """Order-independent fingerprint of a state dict (fp64 sums), used on the GPU box to check
    that seeded construction reproduced the weights this fixture was generated with."""
    tot, atot = 0.0, 0.0
    for k in sorted(sd):
        v = sd[k].double()
        tot += float(v.sum())
        atot += float(v.abs().sum())
    return [tot, atot]


def summarize_grads(named):
    """Full tensors are too big to commit (G 13 M / D 45 M params): (sum, L2 norm, first 64 values) of each, what
    parity_util.compare_grads compares."""
    return {k: {"sum": float(g.detach().double().sum()), "norm": float(g.detach().double().norm()),
                "head": g.detach().flatten()[:64].clone()} for k, g in named.items()}


def sample_tensor(t, k, seed=0):
    """A fixed random subset of k of t's elements (flat indices and values) with t's max |.|, L2 norm and sum (fp64)."""
    t = t.detach().flatten()
    idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(seed))[:k].sort().values
    return {"numel": t.numel(), "idx": idx.int(), "val": t[idx].clone(), "absmax": float(t.double().abs().max()),
            "norm": float(t.double().norm()), "sum": float(t.double().sum())}


def construction_record(sd):
    """Per tensor of a freshly constructed state dict: its digest, except for the spectral-norm vectors u, v.  Those come out of
    power iterations at construction, whose float rounding depends on the host's BLAS and thread count; they get a 32-element
    sample_tensor (as plain lists) instead."""
    out = {}
    for k, v in sd.items():
        if k.endswith("._u") or k.endswith("._v"):
            s = sample_tensor(v, 32)
            out[k] = dict(s, idx=s["idx"].tolist(), val=s["val"].tolist())
        else:
            out[k] = tensor_digest(v)
    return out


def shrink(res, out_k=8192, state_max=1024, state_k=256):
    """Sample the generator outputs and the large buffers (spectral-norm v vectors) of a run_case result in place."""
    res["out"] = sample_tensor(res["out"], out_k)
    for key in ("g_state_after", "d_state_after"):
        for k, v in res.get(key, {}).items():
            if v.numel() > state_max:
                res[key][k] = sample_tensor(v, state_k)
    return res


def build_reference_gan(cfg, seed=0):
    import_reference()
    from dgmr.common import ContextConditioningStack, LatentConditioningStack
    from dgmr.discriminators import Discriminator
    from dgmr.generators import Generator, Sampler

    torch.manual_seed(seed)
    s = cfg["output_shape"]
    gen = Generator(
        ContextConditioningStack(input_channels=1, output_channels=cfg["context_channels"]),
        LatentConditioningStack(shape=(8, s // 32, s // 32), output_channels=cfg["latent_channels"]),
        Sampler(forecast_steps=cfg["forecast_steps"], latent_channels=cfg["latent_channels"],
                context_channels=cfg["context_channels"]),
    )
    disc = Discriminator(input_channels=1)
    return gen, disc


def weight_fn(y, cap=24.0):  # dgmr/dgmr.py:20-33 (cannot import dgmr.dgmr without lightning)
    return torch.max(y + 1, torch.tensor(cap, device=y.device))


def run_case(gen, disc, g0, d0, x, y, training, seed):
    from dgmr.losses import GridCellLoss, loss_hinge_disc, loss_hinge_gen

    gen.load_state_dict(g0)
    disc.load_state_dict(d0)
    gen.train(training)
    disc.train(training)
    # attention gamma is 0 at init, which hides the attention path: give it a value
    with torch.no_grad():
        gen.latent_stack.att_block.gamma.fill_(0.5)
    for p in list(gen.parameters()) + list(disc.parameters()):
        p.grad = None
    torch.manual_seed(seed)
    out = gen(x)
    real = torch.cat([x, y], dim=1)
    fake = torch.cat([x, out], dim=1)
    scores = disc(torch.cat([real, fake], dim=0))
    b = x.shape[0]
    s_real, s_gen = scores[:b], scores[b:]
    d_loss = loss_hinge_disc(s_gen[:, 0:1], s_real[:, 0:1]) + loss_hinge_disc(s_gen[:, 1:2], s_real[:, 1:2])
    grid = GridCellLoss(weight_fn=weight_fn)(out, y)
    g_loss = loss_hinge_gen(s_gen) + 20.0 * grid
    res = {
        "out": out.detach().clone(),
        "scores": scores.detach().clone(),
        "d_loss": d_loss.detach().clone(),
        "grid": grid.detach().clone(),
        "g_loss": g_loss.detach().clone(),
    }
    if training:
        d_params = dict(disc.named_parameters())
        g_params = dict(gen.named_parameters())
        dg = torch.autograd.grad(d_loss, list(d_params.values()), retain_graph=True, allow_unused=True)
        gg = torch.autograd.grad(g_loss, list(g_params.values()), allow_unused=True)
        res["d_grads"] = summarize_grads({k: g for k, g in zip(d_params, dg) if g is not None})
        res["g_grads"] = summarize_grads({k: g for k, g in zip(g_params, gg) if g is not None})
        res["g_state_after"] = {k: v.clone() for k, v in gen.state_dict().items()
                                if k.endswith("._u") or k.endswith("._v") or "running_" in k
                                or "num_batches" in k}
        res["d_state_after"] = {k: v.clone() for k, v in disc.state_dict().items()
                                if k.endswith("._u") or k.endswith("._v") or "running_" in k
                                or "num_batches" in k}
    return res


def block_record():
    """Each building block of the reference on seeded inputs, in train then eval mode (train mode moves the spectral-norm vectors and
    BatchNorm statistics the eval forward then uses): the initial state, and the output and the state after each forward."""
    import_reference()
    from dgmr.common import DBlock, GBlock, LBlock, UpsampleGBlock
    from dgmr.layers import AttentionLayer, ConvGRU

    sd = lambda m: {k: v.clone() for k, v in m.state_dict().items()}  # noqa: E731
    torch.manual_seed(3)
    cases = [
        ("g_block", GBlock(16, 16), torch.rand(2, 16, 8, 8)),
        ("upsample_g_block", UpsampleGBlock(16, 8), torch.rand(2, 16, 8, 8)),
        ("d_block", DBlock(8, 16), torch.rand(2, 8, 8, 8)),
        ("d_block_3d", DBlock(4, 8, conv_type="3d", first_relu=False), torch.rand(2, 4, 6, 8, 8)),
        ("d_block_keep_same_output", DBlock(8, 8, keep_same_output=True), torch.rand(2, 8, 4, 4)),
        ("l_block", LBlock(8, 24), torch.rand(1, 8, 4, 4)),
    ]
    blocks = []
    for name, mod, x in cases:
        rec = {"name": name, "x": x, "state": sd(mod)}     # the eval forward starts from rec["train"]["state_after"]
        for tr in (True, False):
            mod.train(tr)
            with torch.no_grad():
                out = mod(x)
            rec["train" if tr else "eval"] = {"out": out, "state_after": sd(mod)}
        blocks.append(rec)
    att = AttentionLayer(48, 48)
    with torch.no_grad():
        att.gamma.fill_(0.7)
    x = torch.randn(1, 48, 4, 4)
    with torch.no_grad():
        attention = {"state": sd(att), "x": x, "out": att(x)}
    gru = ConvGRU(24 + 8, 8)
    xs, h = [torch.rand(2, 24, 8, 8) for _ in range(3)], torch.rand(2, 8, 8, 8)
    state = sd(gru)
    with torch.no_grad():
        conv_gru = {"state": state, "xs": xs, "h": h, "out": gru(xs, h)}
    return {"blocks": blocks, "attention": attention, "conv_gru": conv_gru}


WRAPPER_CFG = dict(forecast_steps=2, output_shape=128, latent_channels=288, context_channels=48)


def wrapper_losses():
    """The losses the reference's own DGMR.training_step logs for one step on seeded inputs (reference modules, stubbed Lightning:
    baseline/reference_arm.py), for generation_steps 1 and 2."""
    from baseline import reference_arm as R

    os.environ["DGMR_REFERENCE"] = REF
    torch.manual_seed(1)
    x, y = torch.rand(2, 4, 1, 128, 128), torch.rand(2, 2, 1, 128, 128)
    out = {"cfg": WRAPPER_CFG, "init_seed": 0, "data_seed": 1, "step_seed": 2}
    for k in (1, 2):
        model = R.build_dgmr(WRAPPER_CFG, generation_steps=k, dropin=False, anomaly=False, seed=0)
        torch.manual_seed(2)
        out[f"generation_steps={k}"] = {name: float(v) for name, v in R.training_step_fn(model, x, y)().items()}
    for name in [name for name in sys.modules if name == "dgmr" or name.startswith("dgmr.")]:
        del sys.modules[name]
    return out


def main():
    if not os.path.isfile(os.path.join(REF, "dgmr", "dgmr.py")):
        sys.exit("set DGMR_REFERENCE to a checkout of openclimatefix/skillful_nowcasting")
    cfg = C1
    gen, disc = build_reference_gan(cfg, seed=0)
    with torch.no_grad():
        gen.latent_stack.att_block.gamma.fill_(0.5)
    g0 = {k: v.clone() for k, v in gen.state_dict().items()}
    d0 = {k: v.clone() for k, v in disc.state_dict().items()}
    torch.manual_seed(1)
    s, b, t = cfg["output_shape"], cfg["batch"], cfg["forecast_steps"]
    x = torch.rand(b, 4, 1, s, s)
    y = torch.rand(b, t, 1, s, s)
    fix = {"cfg": cfg, "g_checksum": state_checksum(g0), "d_checksum": state_checksum(d0),
           "g_digest": construction_record(g0), "d_digest": construction_record(d0),
           "init_seed": 0, "data_seed": 1, "seed": 2, "gamma": 0.5, "torch_version": str(torch.__version__)}
    fix["eval"] = shrink(run_case(gen, disc, g0, d0, x, y, False, 2))
    fix["train"] = shrink(run_case(gen, disc, g0, d0, x, y, True, 2))
    # RNG draws the reference makes inside that forward, recorded for documentation
    torch.manual_seed(2)
    fix["z"] = torch.normal(torch.zeros(8, s // 32, s // 32, 1), torch.ones(8, s // 32, s // 32, 1))
    fix["idxs"] = torch.randint(low=0, high=4 + t, size=(8,))
    path = os.path.join(HERE, "c1_gan.pt")
    torch.save(fix, path)
    print("wrote", path, os.path.getsize(path) / 1e6, "MB")
    print("eval out sum", fix["eval"]["out"]["sum"], "scores", fix["eval"]["scores"].flatten().tolist())
    print("train out sum", fix["train"]["out"]["sum"], "d_loss", float(fix["train"]["d_loss"]))
    path = os.path.join(HERE, "reference_blocks.pt")
    torch.save(block_record(), path)
    print("wrote", path, os.path.getsize(path) / 1e6, "MB")
    path = os.path.join(HERE, "reference_wrapper_losses.json")
    with open(path, "w") as f:
        json.dump(wrapper_losses(), f, indent=1)
        f.write("\n")
    print("wrote", path)


if __name__ == "__main__":
    main()
