"""Batched K-member ensembles on the B200 (Generator.sample, GraphedGenerator(num_samples=)) against sequential eager calls and the CPU
oracle, and the one-pass ensemble statistics kernel (ensemble.summarize) against the plain-torch reference of tests/ensemble_ref.py.

Tolerances (rel = max|a-b| / max|b|): batched against sequential, SIMT 2e-5, 3xTF32 1e-4, 1xTF32 3e-3 -- the last is the run-to-run floor of
the tap-split ConvGRU convolutions' fp32 atomics (DESIGN.md section 5), which the two arms hit at different launch shapes."""
import pytest
import torch

from ensemble_ref import summarize_ref
from parity_util import C1, build_gan, c1_inputs, oracle_gan_forward, rel_err

pytestmark = pytest.mark.gpu

TOL = {"simt": 2e-5, "3xtf32": 1e-4, "tf32": 3e-3}
ORACLE_TOL = {"simt": 2e-5, "3xtf32": 1e-4, "tf32": 1e-3}     # the existing eval-mode forward tolerances (tests/test_parity_gpu.py)


def _set_mode(be, mode):
    from skillful_nowcasting_b200 import ops

    ops.clear_pack_cache()
    ops.config.conv_algo = ops.config.wgrad_algo = 1 if mode == "simt" else 0
    ops.config.precision = 1 if mode == "3xtf32" else 0
    be.set_option("prefer_patch", -1)


@pytest.fixture(scope="module")
def c1_state():
    gen, disc = build_gan(C1, seed=0, gamma=0.5)
    return gen, {k: v.clone() for k, v in gen.state_dict().items()}, {k: v.clone() for k, v in disc.state_dict().items()}


@pytest.mark.parametrize("mode", ["simt", "tf32", "3xtf32"])
def test_sample_matches_sequential_and_oracle(cuda_backend, c1_state, mode):
    from oracle import dgmr_oracle as O

    gen, g0, d0 = c1_state
    gen.load_state_dict(g0)
    gen.cuda().eval()
    _set_mode(cuda_backend, mode)
    x, _ = c1_inputs()
    xc = x.cuda()
    K = 4
    torch.manual_seed(2)
    with torch.no_grad():
        seq = torch.stack([gen(xc) for _ in range(K)], 1)
    torch.manual_seed(2)
    zs = [torch.normal(torch.zeros(8, 4, 4, 1), torch.ones(8, 4, 4, 1)) for _ in range(K)]   # the draws sample() consumes
    torch.manual_seed(2)
    got = gen.sample(xc, K)
    torch.manual_seed(2)
    chunked = gen.sample(xc, K, members_per_pass=3)          # passes of 3 + 1
    assert rel_err(got, seq) < TOL[mode], rel_err(got, seq)
    assert rel_err(chunked, got) < TOL[mode], rel_err(chunked, got)
    s = C1["output_shape"]
    for k in range(K):
        ref = O.generator(O.clone_state(g0), x, C1["forecast_steps"], (8, s // 32, s // 32), False, z=zs[k])
        assert rel_err(got[:, k], ref) < ORACLE_TOL[mode], (k, rel_err(got[:, k], ref))
    gen.cpu()


def test_graphed_ensemble_replays_sample(cuda_backend, c1_state):
    from skillful_nowcasting_b200.inference import GraphedGenerator

    gen, g0, _ = c1_state
    gen.load_state_dict(g0)
    gen.cuda().eval()
    _set_mode(cuda_backend, "tf32")
    x, _ = c1_inputs()
    xc = x.cuda()
    runner = GraphedGenerator(gen, xc, num_samples=4)
    n0 = cuda_backend.launches
    torch.manual_seed(2)
    out_g = runner(xc).clone()
    assert cuda_backend.launches == n0, "a graph replay must not issue C-ABI launches from the host"
    torch.manual_seed(2)
    out_e = gen.sample(xc, 4)
    assert out_g.shape == out_e.shape and rel_err(out_g, out_e) < TOL["tf32"]
    torch.manual_seed(5)                        # a second replay takes the next K draws in the reference's order
    runner(xc)
    torch.manual_seed(5)
    assert torch.equal(runner.z, gen.latent_stack.sample_z(xc, 4))
    gen.cpu()


def test_full_size_ensemble_in_several_passes_stays_on_tensor_cores(cuda_backend):
    """C2 widths (latent 768, context 384), 256^2, T = 18, B = 2, K = 20 in passes of 8 + 8 + 4 against 20 sequential eager calls (1xTF32);
    every convolution launch of the batched passes is served by the tensor-core kernels whenever its per-group shape is."""
    import skillful_nowcasting_b200 as B
    from skillful_nowcasting_b200 import ops

    _set_mode(cuda_backend, "tf32")
    torch.manual_seed(0)
    gen = B.Generator(B.ContextConditioningStack(input_channels=1, output_channels=384),
                      B.LatentConditioningStack(shape=(8, 8, 8), output_channels=768),
                      B.Sampler(forecast_steps=18, latent_channels=768, context_channels=384)).cuda().eval()
    x = torch.rand(2, 4, 1, 256, 256, device="cuda")
    K = 20
    assert gen.sampler.members_per_pass(2, 8, 8) == 37
    torch.manual_seed(3)
    with torch.no_grad():
        seq = torch.stack([gen(x) for _ in range(K)], 1)
    seen = []
    be = cuda_backend
    orig_conv, orig_up = ops._conv_launch, ops._upconv_fwd

    def conv_rec(x_, wp, bias, scale, res, y, n, d, h, wd, c, cout, kd, kh, kw, G, act, y_is_zero=False):
        seen.append((be.conv_umma_supported(n, d, h, wd, c, cout, kd, kh, kw), be.conv_umma_supported(G, d, h, wd, c, cout, kd, kh, kw),
                     ("conv", n, h, wd, c, cout, kd, kh, kw, G)))
        return orig_conv(x_, wp, bias, scale, res, y, n, d, h, wd, c, cout, kd, kh, kw, G, act, y_is_zero)

    def up_rec(x_, w, bias, scale, res, G, act):
        n, _, h, wd, c = x_.shape
        seen.append((be.upconv_supported(n, h, wd, c, w.shape[0]), be.upconv_supported(G, h, wd, c, w.shape[0]), ("upconv", n, h, wd, c, G)))
        return orig_up(x_, w, bias, scale, res, G, act)

    ops._conv_launch, ops._upconv_fwd = conv_rec, up_rec
    try:
        torch.manual_seed(3)
        got = gen.sample(x, K, members_per_pass=8)
    finally:
        ops._conv_launch, ops._upconv_fwd = orig_conv, orig_up
    left = [s[2] for s in seen if s[1] and not s[0]]
    assert not left, f"launches that left the tensor-core kernels because of their size: {left[:5]}"
    assert any(s[2][1] == 18 * 8 * 2 for s in seen)           # the passes did run at T*M*B images
    assert rel_err(got, seq) < TOL["tf32"], rel_err(got, seq)


CASES = [(K, C, S) for K in (1, 2, 6, 20, 33, 64) for C, S in ((1, 128), (2, 256))]


@pytest.mark.parametrize("K,C,S", CASES, ids=[f"K{k}-C{c}-{s}" for k, c, s in CASES])
def test_summarize_matches_reference(cuda_backend, K, C, S):
    from skillful_nowcasting_b200.ensemble import summarize

    g = torch.Generator(device="cuda").manual_seed(K * 100 + C)
    B_, T = 2, 3
    ens = torch.rand((B_, K, T, C, S, S), generator=g, device="cuda") * 4.0
    ens[:, :, :, :, :8, :8] = torch.round(ens[:, :, :, :, :8, :8])            # ties, and exact threshold hits
    target = torch.rand((B_, T, C, S, S), generator=g, device="cuda") * 4.0
    thr = (1.0, float(ens[0, 0, 0, 0, 20, 20]), 2.5)                           # 1.0 and a member value are hit exactly
    got = summarize(ens, thr, target)
    ref = summarize_ref(ens, thr, target)
    assert torch.equal(got["prob"], ref["prob"])
    assert ((got["mean"].double() - ref["mean"]).abs().max() / ref["mean"].abs().max()).item() <= 1e-6
    for s in range(5):
        e = ((got["crps"][..., s].double() - ref["crps"][..., s]).abs().max() / ref["crps"][..., s].abs().max()).item()
        assert e <= 1e-5, (s, e)
    again = summarize(ens, thr, target)
    for k in ("mean", "prob", "crps"):
        assert torch.equal(again[k], got[k]), k


def test_summarize_without_target_reads_no_target(cuda_backend):
    from skillful_nowcasting_b200.ensemble import summarize

    ens = torch.rand((1, 5, 2, 1, 40, 24), device="cuda")                      # no target: any H, W
    seen = []
    orig = cuda_backend._call
    cuda_backend._call = lambda name, *a, **k: (seen.append(a), orig(name, *a, **k))[1]
    try:
        out = summarize(ens, (0.5,))
    finally:
        cuda_backend._call = orig
    assert out["crps"] is None and seen[-1][1] is None                        # the target pointer is NULL
    ref = summarize_ref(ens, (0.5,))
    assert torch.equal(out["prob"], ref["prob"])
    assert ((out["mean"].double() - ref["mean"]).abs().max() / ref["mean"].abs().max()).item() <= 1e-6
    with pytest.raises(RuntimeError, match="multiples of 16"):
        summarize(ens, (), torch.rand((1, 2, 1, 40, 24), device="cuda"))
    with pytest.raises(RuntimeError, match="K = 65"):
        summarize(torch.rand((1, 65, 1, 1, 16, 16), device="cuda"))
