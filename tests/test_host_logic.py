"""Host logic of the drop-in modules (wiring, timestep/frame folding into groups, autograd plumbing, state-dict
contract), exercised WITHOUT a GPU by routing the C-ABI calls to the test-only emulator (tests/emu_backend.py),
and compared with the oracle / golden fixture.  The same comparisons run against the real CUDA library in
tests/test_parity_gpu.py."""
import io

import pytest
import torch

from block_cases import block_cases, run_block_case, run_conv_gru_case
from oracle import dgmr_oracle as O
from parity_util import (C1, GOLDEN, assert_grads_close, build_gan, c1_inputs, compare_grads, module_gan_forward,
                         oracle_gan_forward, rel_err)


@pytest.mark.parametrize("mode", ["eval", "train"])
def test_c1_gan_matches_fixture(emu, mode):
    gen, disc = build_gan(C1, seed=0, gamma=0.5)
    fix = torch.load(GOLDEN)
    x, y = c1_inputs()
    training = mode == "train"
    got = module_gan_forward(gen, disc, x, y, training, seed=fix["seed"], device="cpu")
    tol = 5e-4 if training else 1e-5
    assert rel_err(got["out"], fix[mode]["out"]) < tol
    assert rel_err(got["scores"], fix[mode]["scores"]) < tol * 5
    for k in ("d_loss", "grid", "g_loss"):
        assert rel_err(got[k], fix[mode][k]) < tol * 5, k
    if training:
        for sd, after in ((gen.state_dict(), fix[mode]["g_state_after"]), (disc.state_dict(), fix[mode]["d_state_after"])):
            for k, v in after.items():
                if "num_batches" in k:
                    assert int(sd[k]) == int(v), k
                else:
                    assert rel_err(sd[k], v) < 2e-4, k
        compare_grads(got["d_grads"], fix[mode]["d_grads"], 2e-3, 2e-2, zero_floor=1e-6)
        # G gradients through the whole train-mode net are chaotic at the 1e-2 level even reference-vs-reference
        compare_grads(got["g_grads"], fix[mode]["g_grads"], 5e-2, 2e-1, zero_floor=1e-5)


@pytest.mark.parametrize("case", block_cases(False), ids=lambda c: c[0])
@pytest.mark.parametrize("training", [True, False])
def test_block_forward_backward(emu, case, training):
    """Mirrors the reference's block smoke tests (tests/test_model.py:29-48) but checks values, buffers and grads."""
    run_block_case(case, training, "cpu", 1e-5, 2e-4)


@pytest.mark.parametrize("fused", [True, False])
def test_conv_gru_matches_oracle(emu, fused):
    """ref test shape family: tests/test_model.py:51-81 (scaled down).  fused: read|update gates as one conv and the whole
    recurrence as one autograd node (ops.gru_sequence); False: the per-step wiring."""
    from skillful_nowcasting_b200 import ops
    old = ops.config.gru_sequence
    ops.config.gru_sequence = fused
    try:
        gru, xs, h = run_conv_gru_case("cpu", 1e-5, 2e-4)
        out, new = gru.cell(xs[0].detach(), h)
    finally:
        ops.config.gru_sequence = old
    assert out.shape == (2, 8, 8, 8) and torch.equal(out, new)


def test_state_dict_contract_and_hub_roundtrip(emu, tmp_path):
    """State-dict keys of the reference (SURVEY.md 8b) and save_pretrained / from_pretrained round trip
    (ref: tests/test_model.py:341-399)."""
    import skillful_nowcasting_b200 as B

    smp = B.Sampler(forecast_steps=2, latent_channels=64, context_channels=32)
    keys = set(smp.state_dict().keys())
    for k in ("convGRU1.cell.read_gate_conv.bias", "convGRU1.cell.read_gate_conv.parametrizations.weight.original",
              "convGRU1.cell.output_conv.parametrizations.weight.0._u", "gru_conv_1x1_4.parametrizations.weight.0._v",
              "g1.bn1.running_mean", "g1.bn1.num_batches_tracked", "up_g4.conv_1x1.bias", "bn.weight", "conv_1x1.bias"):
        assert k in keys, k
    assert len(B.Sampler().state_dict()) == 249 and len(B.Discriminator(1).state_dict()) == 162
    ctx = B.ContextConditioningStack(input_channels=1, output_channels=96)
    ctx.save_pretrained(tmp_path / "ctx")
    ctx2 = B.ContextConditioningStack.from_pretrained(tmp_path / "ctx")
    assert ctx2.training is False
    for (ka, va), (kb, vb) in zip(ctx.state_dict().items(), ctx2.state_dict().items()):
        assert ka == kb and torch.equal(va, vb)
    lat = B.LatentConditioningStack(shape=(8, 2, 2), output_channels=288)
    lat.save_pretrained(tmp_path / "lat")
    lat2 = B.LatentConditioningStack.from_pretrained(tmp_path / "lat")
    assert tuple(lat2.shape) == (8, 2, 2)
    d = B.Discriminator(input_channels=1)
    buf = io.BytesIO()
    torch.save(d.state_dict(), buf)
    buf.seek(0)
    B.Discriminator(input_channels=1).load_state_dict(torch.load(buf))


def test_shapes_of_reference_smoke_tests(emu):
    """ref: tests/test_model.py:84-140 (output shapes of the stacks and discriminators), at reduced size."""
    import skillful_nowcasting_b200 as B

    lat = B.LatentConditioningStack(shape=(8, 2, 2), output_channels=288)
    assert lat(torch.rand(1, 4, 1, 64, 64)).shape == (1, 288, 2, 2)
    ctx = B.ContextConditioningStack(input_channels=1, output_channels=96)
    outs = ctx(torch.rand(2, 4, 1, 64, 64))
    assert [tuple(o.shape) for o in outs] == [(2, 12, 16, 16), (2, 24, 8, 8), (2, 48, 4, 4), (2, 96, 2, 2)]


def test_dgmr_training_step_runs_reference_schedule(emu):
    """ref: tests/test_model.py:285-306 (config C1 at reduced width) + the literal schedule of dgmr/dgmr.py:137-218."""
    import skillful_nowcasting_b200 as B

    torch.manual_seed(0)
    model = B.DGMR(forecast_steps=2, output_shape=128, latent_channels=288, context_channels=32, generation_steps=1)
    x, y = torch.rand(2, 4, 1, 128, 128), torch.rand(2, 2, 1, 128, 128)
    g_before = [p.detach().clone() for p in model.generator.parameters()]
    d_before = [p.detach().clone() for p in model.discriminator.parameters()]
    model.training_step((x, y), 0)
    assert set(model.logged) == {"train/d_loss", "train/g_loss", "train/grid_loss"}
    assert all(torch.isfinite(v) and v.dim() == 0 for v in model.logged.values())
    g_changed = sum(not torch.equal(a, b) for a, b in zip(g_before, model.generator.parameters()))
    d_changed = sum(not torch.equal(a, b) for a, b in zip(d_before, model.discriminator.parameters()))
    # parameters that never receive gradients stay put (g*.conv_1x1 w+b, SURVEY Appendix B 11; attention q/k/v/out while gamma == 0),
    # and so do the 8 first_conv_3x3 biases in front of a train-mode BatchNorm: their gradient is identically zero and is not
    # produced at all here (ops._ConvBNRelu), while the reference random-walks them on rounding noise
    assert g_changed >= len(g_before) - 20 and d_changed >= 30, (g_changed, len(g_before), d_changed, len(d_before))
    assert model(x).shape == (2, 2, 1, 128, 128)


def test_gan_step_matches_oracle_step(emu):
    """training.gan_step (minimal schedule, fused Adam on flat buffers, requires_grad toggling) against oracle.gan_step from the same
    state and seeds: losses, all parameters, Adam moments and step counts, mutated buffers.  Recorded fp32 numbers (emulator vs oracle):
    g_m 6.7e-3, g_update 4.2e-3, d_uv 3.3e-3, d_bn 8.0e-3; oracle vs itself with another thread count: 5.3e-3, 3.5e-3, 2.6e-4, 7.7e-3."""
    from parity_util import GAN_STEP_TOL_FP32, compare_gan_step, module_gan_step, oracle_gan_step

    gen, disc = build_gan(C1, seed=0, gamma=0.5)
    g0 = {k: v.clone() for k, v in gen.state_dict().items()}
    d0 = {k: v.clone() for k, v in disc.state_dict().items()}
    x, y = c1_inputs()
    ref = oracle_gan_step(g0, d0, x, y, C1, seed=4)
    got = module_gan_step(gen, disc, x, y, seed=4, device="cpu")
    compare_gan_step(got, ref, g0, d0, GAN_STEP_TOL_FP32)


def test_gan_step_with_two_generation_steps_matches_oracle_step(emu):
    """generation_steps = 2 (ref: dgmr/dgmr.py:171-190: K generator samples per input, grid-cell loss on their mean, every sample scored by
    the discriminator next to the real sequence): the same comparison as above, same fp32 bounds."""
    from parity_util import GAN_STEP_TOL_FP32, compare_gan_step, module_gan_step, oracle_gan_step

    gen, disc = build_gan(C1, seed=0, gamma=0.5)
    g0 = {k: v.clone() for k, v in gen.state_dict().items()}
    d0 = {k: v.clone() for k, v in disc.state_dict().items()}
    x, y = c1_inputs()
    ref = oracle_gan_step(g0, d0, x, y, C1, seed=4, generation_steps=2)
    got = module_gan_step(gen, disc, x, y, seed=4, device="cpu", generation_steps=2)
    compare_gan_step(got, ref, g0, d0, GAN_STEP_TOL_FP32)


def test_packed_weights_keep_their_addresses_across_optimiser_steps(emu):
    """What inference.GraphedGenerator(train_mode=True) relies on: in the 1xTF32 mode every cached packed copy of a generator weight (ordinary,
    channel-padded, dgrad, pre-summed sub-pixel tiles) is refreshed IN PLACE by the optimiser step -- same buffer address before and after,
    tag = the parameter's new version, contents = a fresh pack of the updated weight -- so a captured graph keeps reading live weights."""
    from skillful_nowcasting_b200 import _lib, ops
    from skillful_nowcasting_b200.training import Adam, gan_step

    ops.config._force_upconv = True          # the sub-pixel form (and its packs) on the host emulator too
    try:
        gen, disc = build_gan(C1, seed=0, gamma=0.5)
        gen.train(); disc.train()
        g_opt = Adam(gen.parameters(), lr=5e-5, betas=(0.0, 0.999))
        d_opt = Adam(disc.parameters(), lr=2e-4, betas=(0.0, 0.999))
        x, y = c1_inputs()

        def packs():
            return {(n, key): buf for n, p in gen.named_parameters() for key, (_, buf) in p.__dict__.get("_dgmr_packs", {}).items()}

        torch.manual_seed(1)
        gan_step(gen, disc, g_opt, d_opt, x, y)
        before = {k: (b.data_ptr(), b.clone()) for k, b in packs().items()}
        assert len(before) > 50 and any(isinstance(k[1][2], tuple) and k[1][2][0] == "sub" for k in before)
        torch.manual_seed(2)
        gan_step(gen, disc, g_opt, d_opt, x, y)
        after = packs()
        assert set(after) == set(before)
        be = _lib.backend()
        params = dict(gen.named_parameters())
        changed = 0
        for (n, key), buf in after.items():
            w = params[n]
            assert buf.data_ptr() == before[(n, key)][0], (n, key)
            assert w.__dict__["_dgmr_packs"][key][0] == (w._version, w.data_ptr(), str(w.device)), (n, key)
            changed += int(not torch.equal(buf, before[(n, key)][1]))
            ci0, cin, m = key
            cout, cintot = w.shape[0], w.shape[1]
            fresh = torch.zeros_like(buf)
            if isinstance(m, tuple) and m[0] == "sub":
                be.pack_weight_subpix(w.detach().contiguous(), fresh, cout, cintot, 0, cin, m[1])
            elif isinstance(m, tuple):
                continue                      # channel-padded packs: address and tag checked above
            else:
                be.pack_weight(w.detach().contiguous(), fresh, cout, cintot, ci0, cin, w.numel() // (cout * cintot), m)
            assert torch.equal(buf, fresh), (n, key)
        assert changed > 50                   # the second step did move the weights
    finally:
        ops.config._force_upconv = False


def test_gan_step_with_a_d_phase_generator_runner(emu):
    """gan_step(d_phase_generator=...): the D phase's gradient-free generator forwards go through the supplied runner (on the GPU a CUDA-graph
    replay, inference.GraphedGenerator(train_mode=True); here a plain callable with the same contract: train mode, no autograd, a reused
    output buffer) -- two calls per step, and the step's results are those of the default path bit for bit."""
    from parity_util import module_gan_step

    x, y = c1_inputs()
    results, calls = [], []
    for use_runner in (False, True):
        gen, disc = build_gan(C1, seed=0, gamma=0.5)
        buf = {}

        def runner(images, gen=gen, buf=buf):
            assert gen.training
            with torch.no_grad():
                out = gen(images)
            calls.append(tuple(out.shape))
            buf.setdefault("out", torch.empty_like(out)).copy_(out)     # static output buffer, overwritten by the next call
            return buf["out"]

        results.append(module_gan_step(gen, disc, x, y, seed=4, device="cpu", d_phase_generator=runner if use_runner else None))
    assert len(calls) == 2
    a, b = results
    for k in ("d_loss", "g_loss", "grid_loss"):
        assert torch.equal(a["losses"][k], b["losses"][k]), k
    for part in ("g_state", "d_state"):
        for k in a[part]:
            assert torch.equal(a[part][k], b[part][k]), (part, k)


@pytest.mark.parametrize("which", ["spatial", "temporal"])
@pytest.mark.parametrize("training", [False, True], ids=["eval", "train"])
def test_discriminators_separately(emu, which, training):
    from parity_util import run_discriminator_case

    run_discriminator_case(which, training, "cpu", 2e-4 if not training else 1e-3, tol_grad_l2=1e-2)


def test_packed_weights_die_with_their_parameter(emu):
    """Regression (advisor, round 1): the packed-weight cache was keyed on (data_ptr, version); a new layer whose storage landed on a
    freed layer's address silently ran with the old layer's packed weights.  No clear_pack_cache() between the builds here."""
    from skillful_nowcasting_b200.layers.core import PlainConv

    for i in range(12):
        torch.manual_seed(i)
        m = PlainConv(8, 8, (3, 3))
        x = torch.randn(1, 8, 6, 6)
        ref = torch.nn.functional.conv2d(x, m.weight, m.bias, padding=1)
        assert rel_err(m(x), ref) < 1e-5, i
        with torch.no_grad():          # in-place update without a version bump through autograd is still seen (version counter moves)
            m.weight.mul_(2.0)
        assert rel_err(m(x), torch.nn.functional.conv2d(x, m.weight, m.bias, padding=1)) < 1e-5, i
        del m


def test_adam_checkpoints_like_torch_and_survives_detached_grads(emu):
    """Regression (advisor): Optimizer.state_dict() carried no moments; module.zero_grad() detached the gradients from the flat buffer."""
    from skillful_nowcasting_b200.training import Adam

    torch.manual_seed(0)
    lin, ref = torch.nn.Linear(5, 3), torch.nn.Linear(5, 3)
    ref.load_state_dict(lin.state_dict())
    o, ro = Adam(lin.parameters(), lr=1e-2, betas=(0.0, 0.999)), torch.optim.Adam(ref.parameters(), lr=1e-2, betas=(0.0, 0.999))
    x = torch.randn(4, 5)
    for _ in range(3):
        o.zero_grad(); ro.zero_grad()
        lin(x).pow(2).sum().backward(); ref(x).pow(2).sum().backward()
        o.step(); ro.step()
    assert torch.allclose(lin.weight, ref.weight, atol=1e-7)
    sd, rsd = o.state_dict(), ro.state_dict()
    assert float(sd["state"][0]["step"]) == 3
    for i in (0, 1):
        for k in ("exp_avg", "exp_avg_sq"):
            assert torch.allclose(sd["state"][i][k], rsd["state"][i][k], atol=1e-8), (i, k)
    lin2 = torch.nn.Linear(5, 3)
    lin2.load_state_dict(ref.state_dict())
    o2 = Adam(lin2.parameters(), lr=1e-2, betas=(0.0, 0.999))
    o2.load_state_dict(rsd)                       # a torch.optim.Adam checkpoint resumes here
    lin2.zero_grad(); ref.zero_grad()             # set_to_none: autograd will create fresh .grad tensors
    lin2(x).pow(2).sum().backward(); ref(x).pow(2).sum().backward()
    o2.step(); ro.step()
    assert torch.allclose(lin2.weight, ref.weight, atol=1e-7)
    torch.optim.Adam(ref.parameters(), lr=1e-2).load_state_dict(o2.state_dict())   # and the other way round
    with pytest.raises(RuntimeError):
        o2.add_param_group({"params": [torch.nn.Parameter(torch.zeros(2))]})
        o2.step()


def test_stale_prefetched_sigma_is_dropped(emu):
    """Regression (advisor): a forward that raised between prefetch_sigmas and the consuming conv left a pending 1/sigma behind."""
    from skillful_nowcasting_b200.common import GBlock
    from skillful_nowcasting_b200.layers.core import prefetch_sigmas

    torch.manual_seed(0)
    blk = GBlock(8, 8)
    prefetch_sigmas(blk.sn_calls(1))              # ... and the forward never happens
    with torch.no_grad():
        blk.first_conv_3x3.weight_orig.mul_(3.0)  # weights move on
    y = blk(torch.rand(2, 8, 4, 4))               # must neither assert nor use the stale sigma
    st = O.clone_state({"m." + k: v for k, v in blk.state_dict().items()})
    assert torch.isfinite(y).all()
    prefetch_sigmas(blk.sn_calls(2))              # a stale entry for another G is simply replaced
    blk.run(torch.rand(2, 1, 4, 4, 8), 1)


@pytest.mark.refpkg
@pytest.mark.parametrize("generation_steps", [1, 2])
def test_unmodified_reference_wrapper_runs_on_these_modules(emu, generation_steps):
    """SURVEY 8b / 8d mode (i): the reference's OWN dgmr/dgmr.py (unmodified, from /root/reference or baseline/_ref) constructs and trains
    these modules through the import swap of INTEGRATION.md, and logs the losses the reference itself logs from the same seeds.
    generation_steps = 2: several generator samples per input (ref: dgmr/dgmr.py:171-190; the paper configuration uses 6, BASELINE.json C5)."""
    import os
    import sys

    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    from baseline import reference_arm as R

    cfg = dict(forecast_steps=2, output_shape=128, latent_channels=288, context_channels=48)
    torch.manual_seed(1)
    x, y = torch.rand(2, 4, 1, 128, 128), torch.rand(2, 2, 1, 128, 128)
    logs = {}
    for dropin in (False, True):
        model = R.build_dgmr(cfg, generation_steps=generation_steps, dropin=dropin, anomaly=False, seed=0)
        assert type(model).__module__ == "dgmr.dgmr"
        assert type(model.generator).__module__.startswith("skillful_nowcasting_b200" if dropin else "dgmr.")
        torch.manual_seed(2)
        logs[dropin] = {k: float(v) for k, v in R.training_step_fn(model, x, y)().items()}
    for k in ("train/d_loss", "train/g_loss", "train/grid_loss"):
        a, b = logs[True][k], logs[False][k]
        assert abs(a - b) <= 2e-3 * max(abs(b), 1e-6), (k, a, b)
    for k in [k for k in sys.modules if k == "dgmr" or k.startswith("dgmr.")]:
        del sys.modules[k]


@pytest.mark.parametrize("generation_steps", [1, 2])
def test_gan_step_matches_reference_wrapper_record(emu, generation_steps):
    """training.gan_step on these modules logs the losses the reference's own DGMR.training_step logged on its own modules from the
    same seeds (tests/golden/reference_wrapper_losses.json, written by make_golden.py): same construction, inputs, RNG draws and
    optimiser settings; gan_step only leaves out the wrapper's discarded work, which changes none of the three losses."""
    import json
    import os

    from parity_util import GOLDEN_DIR, module_gan_step

    with open(os.path.join(GOLDEN_DIR, "reference_wrapper_losses.json")) as f:
        rec = json.load(f)
    cfg = rec["cfg"]
    torch.manual_seed(rec["data_seed"])
    x, y = torch.rand(2, 4, 1, 128, 128), torch.rand(2, 2, 1, 128, 128)
    gen, disc = build_gan(dict(cfg, batch=2), seed=rec["init_seed"])
    got = module_gan_step(gen, disc, x, y, seed=rec["step_seed"], device="cpu", generation_steps=generation_steps)["losses"]
    for k, b in rec[f"generation_steps={generation_steps}"].items():
        a = float(got[k.split("/")[1]])
        assert abs(a - b) <= 2e-3 * max(abs(b), 1e-6), (k, a, b)


@pytest.mark.parametrize("training", [True, False], ids=["train", "eval"])
def test_upsample_gblock_subpixel_form(emu, training):
    """UpsampleGBlock with first_conv_3x3 in sub-pixel form (ops.upconv / ops._ConvBNRelu(up2): the four output phases as 2x2-tap
    convolutions of the low-resolution input with pre-summed taps, SURVEY.md section 7) against the oracle's upsample -> 3x3 conv: values,
    buffers and every gradient.  The emulator restates the phase formula, so this pins the host logic (tap sets, weight-gradient
    folding, BatchNorm geometry); the tcgen05 kernels are checked against the same emulator in tests/test_umma_gpu.py."""
    from skillful_nowcasting_b200 import ops

    ops.config._force_upconv = True
    try:
        case = [c for c in block_cases(False) if c[0] == "upg"][0]
        run_block_case(case, training, "cpu", 2e-5, 3e-4)
    finally:
        ops.config._force_upconv = False


def test_save_pretrained_while_parameters_live_in_the_flat_optimiser_buffer(emu, tmp_path):
    """training.Adam turns every parameter into a view of one flat tensor; the stock hub mixin's safetensors writer refuses such views
    ('None is covering the entire storage').  hub.HubMixin saves compact copies: same file format, same keys, same values."""
    import skillful_nowcasting_b200 as B
    from skillful_nowcasting_b200.training import Adam

    torch.manual_seed(0)
    ctx = B.ContextConditioningStack(input_channels=1, output_channels=96)
    Adam(ctx.parameters(), lr=1e-3)          # parameters are now slices of the optimiser's flat buffer
    assert ctx.d1.conv_1x1.bias.untyped_storage().nbytes() > ctx.d1.conv_1x1.bias.numel() * 4
    ctx.save_pretrained(tmp_path / "ctx")
    new = B.ContextConditioningStack.from_pretrained(tmp_path / "ctx")
    for (ka, va), (kb, vb) in zip(ctx.state_dict().items(), new.state_dict().items()):
        assert ka == kb and torch.equal(va, vb)


def test_depth_folded_weight_gradient_matches_direct(emu, monkeypatch):
    """3x3x3 weight gradient with the depth taps folded into the channel axis (ops._Conv.backward: x' = [x(d-1)|x(d)|x(d+1)], a 1x3x3 weight
    gradient with 3*Cin channels, scattered back onto [Cout, Cin, kd, kh, kw]) against the direct form -- same products, same sums."""
    from skillful_nowcasting_b200 import ops

    monkeypatch.setattr(ops, "_tc_wgrad", lambda *a: True)      # take the tensor-core-only branch on the host emulator
    torch.manual_seed(0)
    n, d, h, w, cin, cout = 2, 5, 4, 32, 8, 16
    x, wt, b = torch.randn(n, d, h, w, cin), torch.randn(cout, cin, 3, 3, 3), torch.randn(cout)
    g = None
    res = {}
    for fold in (True, False):
        monkeypatch.setattr(ops.config, "fold_depth_wgrad", fold)
        xs, ws, bs = (t.clone().requires_grad_(True) for t in (x, wt, b))
        y = ops.conv(xs, ws, bs)
        g = torch.randn_like(y) if g is None else g
        res[fold] = torch.autograd.grad(y, [xs, ws, bs], g)
    for a, c in zip(res[True], res[False]):
        assert rel_err(a, c) < 1e-5
