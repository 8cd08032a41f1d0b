"""Whole-model parity on the GPU, through the reference-facing nn.Module API
(which calls the C-ABI): golden fixtures of the reference, the oracle at the
BASELINE.json shapes, and size-independent properties at full size.

Tolerance (north_star / SURVEY §8d): max|y-ref| <= 1e-3 * max|ref| per sample
and rel-L2 <= 1e-3 against the reference's fp32 forward."""
import pytest
import torch

import sudo_rm_rf_b200 as P
from oracle import sudormrf_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL = 1e-3


CLASSES = {"improved": P.SuDORMRF, "groupcomm": P.GroupCommSudoRmRf, "causal": P.CausalSuDORMRF,
           "original": P.OriginalSuDORMRF}


def build(variant, kw, sd):
    m = CLASSES[variant](**kw)
    m.load_state_dict(sd)
    return m.to(DEV).eval()


def test_native_library_is_loaded():
    """The product path must be the CUDA extension (no eager fallback)."""
    from sudo_rm_rf_b200 import _native
    _native.lib()
    maps = open("/proc/self/maps").read()
    assert "libsudormrf_b200.so" in maps


def test_golden_fixtures(golden):
    meta, sd, x, outs, taps = golden
    m = build(meta["variant"], meta["kwargs"], sd)
    with torch.no_grad():
        y = m(x.to(DEV))
    assert y.shape == outs["output"].shape and y.dtype == torch.float32 and y.is_cuda
    e = O.parity_errors(y, outs["output"])
    assert max(e) < TOL, e
    assert max(e) < 1e-4, e          # the fp32 path should be far inside the budget
    if "mc_uniform" in outs:
        with torch.no_grad():
            ymc = m.separate(x.to(DEV), mixture_consistency=True)
        assert max(O.parity_errors(ymc, outs["mc_uniform"])) < TOL
        got = P.mixture_consistency.apply(y, x.to(DEV))
        assert max(O.parity_errors(got, outs["mc_uniform"])) < TOL
        got = P.mixture_consistency.apply(y, x.to(DEV), "magsq")
        assert max(O.parity_errors(got, outs["mc_magsq"])) < TOL


FULL = [
    # BASELINE.json configs (SURVEY §8 table), batch reduced so the CPU oracle finishes in seconds
    ("cfg1_improved_u8_512", "improved",
     dict(out_channels=256, in_channels=512, num_blocks=8, upsampling_depth=5,
          enc_kernel_size=21, enc_num_basis=512, num_sources=2), 1, 32000),
    ("cfg2_improved_u16_512", "improved",
     dict(out_channels=256, in_channels=512, num_blocks=16, upsampling_depth=5,
          enc_kernel_size=21, enc_num_basis=512, num_sources=2), 2, 32079),
    ("cfg4_groupcomm_u8_512", "groupcomm",
     dict(out_channels=256, in_channels=512, num_blocks=8, upsampling_depth=5,
          enc_kernel_size=21, enc_num_basis=512, num_sources=2, group_size=16), 2, 32000),
    ("cfg3_improved_u36_2048_short", "improved",
     dict(out_channels=512, in_channels=512, num_blocks=36, upsampling_depth=6,
          enc_kernel_size=21, enc_num_basis=2048, num_sources=2), 1, 8000),
    # full-length cfg 3 (L=3200 -> level lengths 3200..100: the kernel variants the benchmark dispatches)
    ("cfg3_improved_u36_2048", "improved",
     dict(out_channels=512, in_channels=512, num_blocks=36, upsampling_depth=6,
          enc_kernel_size=21, enc_num_basis=2048, num_sources=2), 1, 32000),
    # cfg 5: WHAMR! model, 4 s @ 16 kHz (mask GEMM M=8192, decoder GEMM K=8192, L=6400)
    ("cfg5_improved_u36_4096_16k", "improved",
     dict(out_channels=512, in_channels=512, num_blocks=36, upsampling_depth=6,
          enc_kernel_size=21, enc_num_basis=4096, num_sources=2), 1, 64000),
    # SURVEY 8d odd lengths on the benchmark model
    ("cfg2_improved_u16_512_T31999", "improved",
     dict(out_channels=256, in_channels=512, num_blocks=16, upsampling_depth=5,
          enc_kernel_size=21, enc_num_basis=512, num_sources=2), 1, 31999),
    ("cfg2_improved_u16_512_T56000", "improved",
     dict(out_channels=256, in_channels=512, num_blocks=16, upsampling_depth=5,
          enc_kernel_size=21, enc_num_basis=512, num_sources=2), 2, 56000),
    ("cfg4_groupcomm_u8_512_T31999", "groupcomm",
     dict(out_channels=256, in_channels=512, num_blocks=8, upsampling_depth=5,
          enc_kernel_size=21, enc_num_basis=512, num_sources=2, group_size=16), 1, 31999),
    # SURVEY 8f.3 sibling variant: CausalSuDORMRF with its constructor defaults (causal_improved_sudormrf_v3.py:121-129)
    # and the stereo / depth-5 geometry of its __main__ block (:235-243), odd length
    ("causal_default_u16_512", "causal",
     dict(in_audio_channels=1, out_channels=128, in_channels=512, num_blocks=16, upsampling_depth=4,
          enc_kernel_size=21, enc_num_basis=512, num_sources=2), 2, 32000),
    ("causal_stereo_u4_512_T44099", "causal",
     dict(in_audio_channels=2, out_channels=256, in_channels=512, num_blocks=4, upsampling_depth=5,
          enc_kernel_size=21, enc_num_basis=512, num_sources=2), 1, 44099),
    # SURVEY 8f.3 sibling variant: the ORIGINAL SuDoRM-RF with its constructor defaults (sudormrf.py:186-193; tensor-core
    # GEMMs with per-channel PReLU on the operand loads, reshape_before_masks, Toeplitz mask GEMM M = 1024 / K = 512) ...
    ("original_default_u16_512", "original",
     dict(out_channels=128, in_channels=512, num_blocks=16, upsampling_depth=4,
          enc_kernel_size=21, enc_num_basis=512, num_sources=2), 2, 32000),
    # ... and a three-source model without the reshape layer (out_channels == enc_num_basis), depth 5, odd length
    ("original_u4_256_3src_T32079", "original",
     dict(out_channels=256, in_channels=512, num_blocks=4, upsampling_depth=5,
          enc_kernel_size=21, enc_num_basis=256, num_sources=3), 1, 32079),
]
DEFAULT_TOO = ("cfg2_improved_u16_512", "cfg3_improved_u36_2048", "cfg5_improved_u36_4096_16k",
               "original_default_u16_512")


@pytest.mark.parametrize("name,variant,kw,B,T", FULL, ids=[f[0] for f in FULL])
@pytest.mark.parametrize("weights", ["perturbed", "default"])
def test_full_size_vs_oracle(name, variant, kw, B, T, weights):
    if weights == "default" and name not in DEFAULT_TOO:
        pytest.skip("default-init weights checked on cfg 2 / 3 / 5 only")
    cfg = O.Config(variant=variant, **kw)
    sd = O.make_state_dict(cfg, seed=21, perturbed=(weights == "perturbed"))
    g = torch.Generator().manual_seed(1)
    x = torch.randn(B, kw.get("in_audio_channels", 1), T, generator=g)
    x = (x - x.mean(-1, keepdim=True)) / (x.std(-1, keepdim=True) + 1e-9)   # README.md:101-103
    ref = O.forward(cfg, sd, x)
    m = build(variant, kw, sd)
    with torch.no_grad():
        y = m(x.to(DEV))
    assert y.shape == ref.shape
    e = O.parity_errors(y, ref)
    print(name, weights, "rel_max %.3e rel_l2 %.3e" % e)
    assert max(e) < TOL, e


def test_properties_at_benchmark_size():
    """Size-independent checks at the cfg-2 benchmark shape (B=32 x 4 s @ 8 kHz)."""
    kw = dict(out_channels=256, in_channels=512, num_blocks=16, upsampling_depth=5,
              enc_kernel_size=21, enc_num_basis=512, num_sources=2)
    cfg = O.Config(variant="improved", **kw)
    sd = O.make_state_dict(cfg, seed=5)
    m = build("improved", kw, sd)
    g = torch.Generator().manual_seed(2)
    x = torch.rand(32, 1, 32000, generator=g).to(DEV)      # the reference's bench input
    with torch.no_grad():
        y = m(x)
        assert y.shape == (32, 2, 32000) and torch.isfinite(y).all()
        # (1) samples are independent: a sample run alone gives the same estimate
        y1 = m(x[5:6])
        assert max(O.parity_errors(y1, y[5:6])) < 1e-5
        # (2) batch-permutation equivariance
        perm = torch.randperm(32, generator=g).to(DEV)
        yp = m(x[perm])
        assert max(O.parity_errors(yp, y[perm])) < 1e-5
        # (3) mixture consistency: corrected estimates sum to the mixture
        ymc = m.separate(x, mixture_consistency=True)
        assert torch.allclose(ymc.sum(1, keepdim=True), x, atol=1e-4)
        assert max(O.parity_errors(ymc, P.mixture_consistency.apply(y, x))) < 1e-6
        # (4) implicit padding == explicit zero padding (improved_sudormrf.py:303-314)
        xo = x[:2, :, :31999]
        yo = m(xo)
        xz = torch.zeros(2, 1, 32000, device=DEV)      # same padded length -> same GlobLN statistics
        xz[..., :31999] = xo
        yz = m(xz)
        assert yo.shape[-1] == 31999
        assert max(O.parity_errors(yo, yz[..., :31999])) < 1e-5
        # (5) spot check one sample of the big batch against the oracle
        ref = O.forward(cfg, sd, x[7:8].cpu())
        assert max(O.parity_errors(y[7:8], ref)) < TOL


def test_depth1_model_with_unaligned_frame_count():
    """upsampling_depth=1 allows L % 4 != 0: big channel counts then run on the FFMA kernels."""
    kw = dict(out_channels=128, in_channels=128, num_blocks=2, upsampling_depth=1,
              enc_kernel_size=21, enc_num_basis=64, num_sources=2)
    cfg = O.Config(variant="improved", **kw)
    sd = O.make_state_dict(cfg, seed=8)
    m = build("improved", kw, sd)
    x = torch.randn(2, 1, 1290, generator=torch.Generator().manual_seed(0))     # Tp = 1300 -> L = 130
    with torch.no_grad():
        y = m(x.to(DEV))
    assert max(O.parity_errors(y, O.forward(cfg, sd, x))) < 1e-4


def test_host_entry_and_dtype_handling():
    kw = dict(out_channels=32, in_channels=64, num_blocks=2, upsampling_depth=4,
              enc_kernel_size=21, enc_num_basis=48, num_sources=2)
    cfg = O.Config(variant="improved", **kw)
    sd = O.make_state_dict(cfg, seed=3)
    m = build("improved", kw, sd)
    x = torch.randn(3, 1, 4001, generator=torch.Generator().manual_seed(0))
    ref = O.forward(cfg, sd, x)
    hx = x.pin_memory()
    hy = m.forward_host(hx)                  # 1st call: eager
    torch.cuda.synchronize()
    assert max(O.parity_errors(hy, ref)) < 1e-4
    # 2nd call captures a CUDA graph of (H2D, forward, D2H); later calls replay it with new buffer contents
    for seed in (11, 12, 13):
        xn = torch.randn(3, 1, 4001, generator=torch.Generator().manual_seed(seed))
        hx.copy_(xn)
        m.forward_host(hx, hy)
        torch.cuda.synchronize()
        assert max(O.parity_errors(hy, O.forward(cfg, sd, xn))) < 1e-4
    hx.copy_(x)
    # pageable buffers take the eager path
    hp = m.forward_host(x.clone(), torch.empty(3, 2, 4001))
    torch.cuda.synchronize()
    assert max(O.parity_errors(hp, ref)) < 1e-4
    with torch.no_grad():
        y64 = m(x.double().to(DEV))          # any float dtype is cast to fp32 (reference :312)
        y16 = m(x.half().to(DEV))
    assert y64.dtype == torch.float32
    assert max(O.parity_errors(y64, ref)) < 1e-4
    assert max(O.parity_errors(y16, O.forward(cfg, sd, x.half().float()))) < 1e-4
    # weights updated in place are re-packed
    with torch.no_grad():
        m.bottleneck.bias.add_(0.5)
        y2 = m(x.to(DEV))
    sd2 = dict(sd)
    sd2["bottleneck.bias"] = sd["bottleneck.bias"] + 0.5
    assert max(O.parity_errors(y2, O.forward(cfg, sd2, x))) < 1e-4
    m.forward_host(hx, hy)                   # ... and invalidate the captured host graph
    torch.cuda.synchronize()
    assert max(O.parity_errors(hy, O.forward(cfg, sd2, x))) < 1e-4


def test_training_mode_with_grad_raises_and_eval_runs():
    m = P.SuDORMRF(16, 32, 1, 2, 21, 16, 2).to(DEV)
    x = torch.randn(1, 1, 400, device=DEV)
    m.train()
    with pytest.raises(RuntimeError, match="inference"):
        m(x)
    m.eval()
    y = m(x)                                  # simple_whamr_evaluation.py:145 calls without no_grad
    assert not y.requires_grad


def test_cuda_graph_capture_replays():
    kw = dict(out_channels=32, in_channels=64, num_blocks=2, upsampling_depth=4,
              enc_kernel_size=21, enc_num_basis=48, num_sources=2)
    cfg = O.Config(variant="improved", **kw)
    m = build("improved", kw, O.make_state_dict(cfg, seed=3))
    x = torch.randn(2, 1, 4000, device=DEV)
    with torch.no_grad():
        want = m(x).clone()
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            m(x)
        torch.cuda.current_stream().wait_stream(s)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            y = m(x)
        x.copy_(torch.randn_like(x))
        g.replay()
        want2 = m(x)
    torch.cuda.synchronize()
    assert max(O.parity_errors(y, want2)) < 1e-6
    assert max(O.parity_errors(want, want2)) > 1e-3


def test_data_parallel_wrapper_single_device():
    """nn.DataParallel(model) keeps working (run_improved_sudormrf.py:118)."""
    kw = dict(out_channels=32, in_channels=64, num_blocks=1, upsampling_depth=3,
              enc_kernel_size=21, enc_num_basis=32, num_sources=2)
    cfg = O.Config(variant="improved", **kw)
    sd = O.make_state_dict(cfg, seed=4)
    m = torch.nn.DataParallel(build("improved", kw, sd)).cuda().eval()
    x = torch.randn(4, 1, 1000, generator=torch.Generator().manual_seed(0))
    with torch.no_grad():
        y = m(x.cuda())
    assert max(O.parity_errors(y, O.forward(cfg, sd, x))) < 1e-4


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_data_parallel_two_devices():
    """nn.DataParallel over 2 GPUs: one host thread per device calls forward on a replica whose
    parameters are freshly broadcast tensors (run_improved_sudormrf.py:118)."""
    kw = dict(out_channels=128, in_channels=256, num_blocks=2, upsampling_depth=4,
              enc_kernel_size=21, enc_num_basis=128, num_sources=2)
    cfg = O.Config(variant="improved", **kw)
    sd = O.make_state_dict(cfg, seed=4)
    m = torch.nn.DataParallel(build("improved", kw, sd), device_ids=[0, 1]).eval()
    x = torch.randn(6, 1, 3000, generator=torch.Generator().manual_seed(0))
    ref = O.forward(cfg, sd, x)
    with torch.no_grad():
        for _ in range(3):                      # replicas are rebuilt on every call
            y = m(x.cuda(0))
            assert y.device.index == 0 and max(O.parity_errors(y, ref)) < 1e-4


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_model_on_second_device():
    kw = dict(out_channels=128, in_channels=256, num_blocks=1, upsampling_depth=3,
              enc_kernel_size=21, enc_num_basis=128, num_sources=2)
    cfg = O.Config(variant="improved", **kw)
    sd = O.make_state_dict(cfg, seed=6)
    m = P.SuDORMRF(**kw)
    m.load_state_dict(sd)
    m = m.to("cuda:1").eval()
    x = torch.randn(2, 1, 2000, generator=torch.Generator().manual_seed(1))
    with torch.no_grad():
        y = m(x.to("cuda:1"))                   # current device stays cuda:0
    assert y.device.index == 1 and max(O.parity_errors(y, O.forward(cfg, sd, x))) < 1e-4
    with pytest.raises(RuntimeError):
        m(x.to("cuda:0"))                       # parameters and input on different devices


def test_validation_loop_of_the_reference_runner():
    """The validation half of dnn/experiments/run_improved_sudormrf.py:189-208 on synthetic tensors: model under
    nn.DataParallel (:118), eval + no_grad, per-utterance normalisation, PermInvariantSISDR with improvement
    (:82-85), with this repo's metric kernel (same constructor as the reference's loss class).  The reference's
    own PermInvariantSISDR on the oracle's estimates of these batches is stored in golden/reference_sisdr.npz
    (golden/make_golden_reference.py), and the per-utterance values must agree with it."""
    import os
    import numpy as np
    kw = dict(out_channels=64, in_channels=128, num_blocks=2, upsampling_depth=4,
              enc_kernel_size=21, enc_num_basis=64, num_sources=2)
    cfg = O.Config(variant="improved", **kw)
    sd = O.make_state_dict(cfg, seed=9)
    model = torch.nn.DataParallel(build("improved", kw, sd)).cuda()
    from sudo_rm_rf_b200 import sisdr as b200_sisdr
    losses = {"b200": b200_sisdr.PermInvariantSISDR(batch_size=4, n_sources=2, zero_mean=True, backward_loss=False,
                                                 improvement=True, return_individual_results=True)}
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_sisdr.npz"))
    reference_loss = torch.from_numpy(z["runner_val/loss"]).reshape(2, 4)
    g = torch.Generator().manual_seed(3)
    acc = {k: [] for k in losses}
    model.eval()
    with torch.no_grad():
        for bi in range(2):                                                  # two "batches"
            clean = torch.randn(4, 2, 8000, generator=g)
            m1wavs = clean.sum(1).cuda()
            m1wavs = (m1wavs - m1wavs.mean(-1, keepdim=True)) / (m1wavs.std(-1, keepdim=True) + 1e-9)
            rec = model(m1wavs.unsqueeze(1))
            ref = O.forward(cfg, sd, m1wavs.unsqueeze(1).cpu())
            assert max(O.parity_errors(rec, ref)) < 1e-4
            for name, fn in losses.items():
                l = fn(rec, clean.cuda(), initial_mixtures=m1wavs.unsqueeze(1))
                acc[name] += l.tolist()
                want = O.pit_sisdr(ref, clean, m1wavs.unsqueeze(1).cpu(), zero_mean=True, improvement=True)[0]
                assert torch.allclose(l.cpu().float(), want.float(), atol=2e-3), (name, l, want)
                assert torch.allclose(l.cpu().float(), reference_loss[bi].float(), atol=2e-3), (name, l, reference_loss[bi])
    assert all(len(v) == 8 for v in acc.values())


def test_pickle_and_deepcopy_after_forward():
    """torch.save(model) / copy.deepcopy(model) after forward / forward_host do not drag the workspace or the
    captured CUDA graphs along (README.md:75 whole-module checkpoints)."""
    import copy
    import io
    kw = dict(out_channels=32, in_channels=64, num_blocks=1, upsampling_depth=3,
              enc_kernel_size=21, enc_num_basis=32, num_sources=2)
    cfg = O.Config(variant="improved", **kw)
    sd = O.make_state_dict(cfg, seed=4)
    m = build("improved", kw, sd)
    hx = torch.randn(2, 1, 2000).pin_memory()
    for _ in range(3):
        hy = m.forward_host(hx)
    torch.cuda.synchronize()
    assert "_b200_cache" in m.__dict__
    buf = io.BytesIO()
    torch.save(m, buf)
    assert buf.tell() < 4 * sum(p.numel() for p in m.parameters()) + (1 << 20)
    buf.seek(0)
    m2 = torch.load(buf, weights_only=False)
    m3 = copy.deepcopy(m)
    for mm in (m2, m3):
        assert "_b200_cache" not in mm.__dict__
        with torch.no_grad():
            y = mm(hx.cuda())
        assert max(O.parity_errors(y, hy)) < 1e-6


def test_two_streams_share_one_model():
    """Calls arriving on different streams are serialised on the shared workspace."""
    kw = dict(out_channels=64, in_channels=128, num_blocks=2, upsampling_depth=4,
              enc_kernel_size=21, enc_num_basis=64, num_sources=2)
    cfg = O.Config(variant="improved", **kw)
    m = build("improved", kw, O.make_state_dict(cfg, seed=3))
    xs = [torch.randn(4, 1, 16000, device=DEV) for _ in range(4)]
    with torch.no_grad():
        want = [m(x).clone() for x in xs]
        torch.cuda.synchronize()
        streams = [torch.cuda.Stream() for _ in range(2)]
        got = []
        for i, x in enumerate(xs):
            with torch.cuda.stream(streams[i % 2]):
                got.append(m(x))
        torch.cuda.synchronize()
    for a, b in zip(got, want):
        assert torch.equal(a, b)


def test_replaced_parameter_and_submodule_are_noticed():
    """The cached parameter list is validated by object identity along the whole module path."""
    kw = dict(out_channels=32, in_channels=64, num_blocks=2, upsampling_depth=3,
              enc_kernel_size=21, enc_num_basis=32, num_sources=2)
    cfg = O.Config(variant="improved", **kw)
    sd = O.make_state_dict(cfg, seed=4)
    m = build("improved", kw, sd)
    x = torch.randn(2, 1, 1500, generator=torch.Generator().manual_seed(0))
    with torch.no_grad():
        m(x.to(DEV))
        # a middle Parameter object is replaced (not updated in place)
        new_b = torch.nn.Parameter(sd["sm.0.res_conv.bias"].to(DEV) + 1.0)
        m.sm[0].res_conv.bias = new_b
        sd2 = dict(sd)
        sd2["sm.0.res_conv.bias"] = sd["sm.0.res_conv.bias"] + 1.0
        assert max(O.parity_errors(m(x.to(DEV)), O.forward(cfg, sd2, x))) < 1e-4
        # a whole sub-module is replaced
        blk = P.improved_sudormrf.UConvBlock(32, 64, 3).to(DEV)
        m.sm[1] = blk
        sd3 = {k: v for k, v in sd2.items() if not k.startswith("sm.1.")}
        sd3.update({"sm.1." + k: v.detach().cpu() for k, v in blk.state_dict().items()})
        assert max(O.parity_errors(m(x.to(DEV)), O.forward(cfg, sd3, x))) < 1e-4


def test_mixture_consistency_on_multichannel_model_raises():
    m = P.GroupCommSudoRmRf(in_audio_channels=2, out_channels=32, in_channels=64, num_blocks=1,
                            upsampling_depth=2, enc_kernel_size=11, enc_num_basis=32, num_sources=2,
                            group_size=4).to(DEV).eval()
    x = torch.randn(1, 2, 800, device=DEV)
    with torch.no_grad():
        assert m(x).shape == (1, 4, 800)
        with pytest.raises(RuntimeError, match="mono"):
            m.separate(x)                       # default mixture_consistency=True


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_data_parallel_two_devices_sees_new_weights():
    """load_state_dict between two DataParallel forwards: the replicas' parameters are fresh broadcast tensors
    (version 0, recycled addresses), so replicas re-pack on every call."""
    kw = dict(out_channels=128, in_channels=256, num_blocks=2, upsampling_depth=4,
              enc_kernel_size=21, enc_num_basis=128, num_sources=2)
    cfg = O.Config(variant="improved", **kw)
    sd_a = O.make_state_dict(cfg, seed=4)
    sd_b = O.make_state_dict(cfg, seed=5)
    base = build("improved", kw, sd_a)
    m = torch.nn.DataParallel(base, device_ids=[0, 1]).eval()
    x = torch.randn(6, 1, 3000, generator=torch.Generator().manual_seed(0))
    with torch.no_grad():
        for sd in (sd_a, sd_b, sd_a, sd_b):
            base.load_state_dict(sd)
            y = m(x.cuda(0))
            assert max(O.parity_errors(y, O.forward(cfg, sd, x))) < 1e-4


def test_original_model_api():
    """The original SuDoRM-RF (sudormrf.py) behind its own import path: README-style call, mixture consistency,
    separate(normalize=True), forward_host with a CUDA graph, lengths that need padding and lengths that do not."""
    kw = dict(out_channels=32, in_channels=64, num_blocks=2, upsampling_depth=4,
              enc_kernel_size=21, enc_num_basis=48, num_sources=2)
    cfg = O.Config(variant="original", **kw)
    sd = O.make_state_dict(cfg, seed=3)
    m = build("original", kw, sd)
    assert m.lcm == 80
    for T in (4001, 4000, 77):                 # 4000 is a multiple of lcm(10, 16) = 80: the reference does not pad it
        x = torch.randn(3, 1, T, generator=torch.Generator().manual_seed(T))
        ref = O.forward(cfg, sd, x)
        with torch.no_grad():
            y = m(x.to(DEV))
            ymc = m.separate(x.to(DEV), mixture_consistency=True)
        assert y.shape == (3, 2, T)
        assert max(O.parity_errors(y, ref)) < 1e-4
        assert max(O.parity_errors(ymc, O.mixture_consistency(ref, x))) < 1e-4
    x = torch.randn(3, 1, 4001, generator=torch.Generator().manual_seed(5)) * 3 + 0.5
    with torch.no_grad():
        got = m.separate(x.to(DEV), normalize=True)
    assert max(O.parity_errors(got, O.separate(cfg, sd, x.squeeze(1)))) < 1e-4
    hx = x.pin_memory()
    hy = m.forward_host(hx)
    for _ in range(2):                         # eager, capture, replay
        m.forward_host(hx, hy)
    torch.cuda.synchronize()
    assert max(O.parity_errors(hy, O.forward(cfg, sd, x))) < 1e-4
    m.train()
    with pytest.raises(RuntimeError, match="inference"):
        m(x.to(DEV))


@pytest.mark.parametrize("depth,T", [(1, 1290), (2, 1300), (3, 1324)])
def test_original_model_shallow_depths_with_unaligned_frame_counts(depth, T):
    """upsampling_depth 1 / 2 / 3 with lcm padding gives frame counts that are odd / even-but-not-a-multiple-of-4 /
    a multiple of 4 only (L = 129 / 130 / 132): the scalar and float2 paths of every kernel the original model uses."""
    kw = dict(out_channels=64, in_channels=128, num_blocks=2, upsampling_depth=depth,
              enc_kernel_size=21, enc_num_basis=64, num_sources=2)
    cfg = O.Config(variant="original", **kw)
    sd = O.make_state_dict(cfg, seed=8)
    m = build("original", kw, sd)
    x = torch.randn(2, 1, T, generator=torch.Generator().manual_seed(0))
    with torch.no_grad():
        y = m(x.to(DEV))
    assert max(O.parity_errors(y, O.forward(cfg, sd, x))) < 1e-4
