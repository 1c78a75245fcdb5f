"""Batched K-member ensemble forecasts (Generator.sample, DGMR.sample, GraphedGenerator(num_samples=)) and the plain-torch CRPS reference
the GPU tests of ensemble.summarize compare against -- host logic on the ABI emulator, no GPU."""
import pytest
import torch

from ensemble_ref import crps_pairwise, crps_sorted, summarize_ref
from parity_util import C1, build_gan, c1_inputs


@pytest.fixture(scope="module")
def c1_gen():
    gen, _ = build_gan(C1, seed=0, gamma=0.5)
    return gen.eval()


@pytest.mark.parametrize("members_per_pass", [1, 2, 3])
def test_sample_equals_sequential_calls(emu, c1_gen, members_per_pass):
    """sample(x, 3) == stack of 3 eager calls from the same seed, and the CPU RNG ends in the same state."""
    x, _ = c1_inputs()
    torch.manual_seed(7)
    with torch.no_grad():
        seq = torch.stack([c1_gen(x) for _ in range(3)], 1)
    nxt_seq = torch.rand(4)
    torch.manual_seed(7)
    got = c1_gen.sample(x, 3, members_per_pass=members_per_pass)
    nxt = torch.rand(4)
    assert got.shape == (C1["batch"], 3, C1["forecast_steps"], 1, C1["output_shape"], C1["output_shape"])
    assert torch.equal(nxt, nxt_seq)
    torch.testing.assert_close(got, seq, rtol=1e-5, atol=1e-6)
    assert not torch.equal(got[:, 0], got[:, 1])               # each member has its own latent


def test_one_member_pass_issues_the_forward_launches(emu, c1_gen):
    """With one member the sampler runs exactly the single forward's launches (same count; the output permute has no member axis)."""
    from skillful_nowcasting_b200 import _lib

    be = _lib.backend()
    calls = []
    orig = be.permute
    be.permute = lambda *a, **k: (calls.append(len(a[2])), orig(*a, **k))[1]
    x, _ = c1_inputs()
    with torch.no_grad():
        cond = list(c1_gen.conditioning_stack.run(x))
        lat = c1_gen.latent_stack.run(x)
        n0 = len(calls)
        c1_gen.sampler.run(cond, lat)
        n_fwd = len(calls) - n0
        out = torch.empty((x.shape[0], 1, C1["forecast_steps"], 1, C1["output_shape"], C1["output_shape"]))
        n0 = len(calls)
        c1_gen.sampler.run(cond, lat, out=out, member0=0)
    assert len(calls) - n0 == n_fwd and calls[-1] == 7


def test_defaults_and_refusals(emu):
    import skillful_nowcasting_b200 as B
    from skillful_nowcasting_b200.inference import GraphedGenerator

    torch.manual_seed(0)
    m = B.DGMR(forecast_steps=2, output_shape=128, latent_channels=288, context_channels=48, num_samples=2).eval()
    x = torch.rand(1, 4, 1, 128, 128)
    assert m.sample(x).shape == (1, 2, 2, 1, 128, 128)
    assert m.sample(x, 1).shape == (1, 1, 2, 1, 128, 128)
    with pytest.raises(RuntimeError):
        m.generator.sample(x, 0)
    with pytest.raises(RuntimeError):
        m.generator.sample(x, 2, members_per_pass=0)
    m.train()
    with pytest.raises(RuntimeError, match="eval"):
        m.sample(x)
    with pytest.raises(RuntimeError, match="eval"):
        GraphedGenerator(m.generator, x, train_mode=True, num_samples=2)


def test_members_per_pass_keeps_tensor_core_launches_addressable():
    """At C2 widths (latent 768, context 384, 256^2, 18 steps) and B = 8: the derived member count keeps every sampler tensor of a pass
    below 2^31 elements -- walked over the actual modules' shapes here -- and one more member would not."""
    import skillful_nowcasting_b200 as B

    s, T, Bn = B.Sampler(forecast_steps=18, latent_channels=768, context_channels=384), 18, 8
    h = w = 256 // 32
    M = s.members_per_pass(Bn, h, w)
    assert M == 9                                              # floor(2^31 / (18 * 8 * 128^2 * 96))

    def largest(m):
        n = 0
        levels = ((s.convGRU1, s.g1, s.up_g1), (s.convGRU2, s.g2, s.up_g2), (s.convGRU3, s.g3, s.up_g3), (s.convGRU4, s.g4, s.up_g4))
        for lvl, (gru, g, ug) in enumerate(levels):
            r = (h << lvl) * (w << lvl)
            cell = gru.cell
            imgs = T * m * Bn
            n = max(n, imgs * r * cell.input_channels, imgs * r * 2 * cell.output_channels,     # gate x parts (read | update side by side)
                    imgs * r * g.input_channels, imgs * r * g.output_channels,
                    imgs * 4 * r * ug.input_channels, imgs * 4 * r * ug.output_channels)      # up-block convs at twice the resolution
        return n

    assert largest(M) < 2 ** 31 <= largest(M + 1)


def test_crps_hand_computed_and_mae():
    ens = torch.tensor([[0.0, 1.0]], dtype=torch.float64)
    y = torch.zeros(1, dtype=torch.float64)
    # (1/2)(0 + 1) - (1/8)(|0-1| + |1-0|) = 0.25
    assert crps_pairwise(ens, y).item() == pytest.approx(0.25)
    assert crps_sorted(ens, y).item() == pytest.approx(0.25)
    g = torch.Generator().manual_seed(0)
    x, yy = torch.rand(100, 1, generator=g, dtype=torch.float64), torch.rand(100, generator=g, dtype=torch.float64)
    torch.testing.assert_close(crps_pairwise(x, yy), (x[:, 0] - yy).abs(), rtol=0, atol=1e-15)   # K = 1: absolute error


@pytest.mark.parametrize("K", [2, 5, 20, 64])
def test_crps_pairwise_equals_sorted_identity(K):
    g = torch.Generator().manual_seed(K)
    x = torch.randn(300, K, generator=g, dtype=torch.float64)
    x[:, K // 2] = x[:, 0]                                     # ties
    y = torch.randn(300, generator=g, dtype=torch.float64)
    torch.testing.assert_close(crps_sorted(x, y), crps_pairwise(x, y), rtol=1e-12, atol=1e-12)


def test_reference_summary_shapes_and_pooled_scales():
    """Output layouts of the reference; an ensemble whose members all equal the target scores 0 at every scale."""
    y = torch.rand(2, 3, 1, 32, 32, dtype=torch.float64)
    ens = y[:, None].repeat(1, 4, 1, 1, 1, 1)
    r = summarize_ref(ens.float(), (0.5,), y.float())
    assert r["crps"].shape == (2, 3, 1, 5) and r["prob"].shape == (1, 2, 3, 1, 32, 32)
    assert r["crps"].abs().max() < 1e-7


def test_summarize_refuses_cpu_tensors():
    from skillful_nowcasting_b200 import _lib
    from skillful_nowcasting_b200.ensemble import summarize

    old = _lib.set_backend(None)
    try:
        with pytest.raises(RuntimeError, match="CUDA"):
            summarize(torch.rand(1, 2, 1, 1, 16, 16), (0.5,), torch.rand(1, 1, 1, 16, 16))
    finally:
        _lib.set_backend(old)
