"""RAFT optical flow (SURVEY §8 rows a6, a7): oracle vs reference goldens (CPU), RAFT helper kernels
and the full sm_100a path vs oracle + goldens (GPU). Flow tolerance: 1e-3 relative (rel-L2 and
max-abs / max|flow|) after the full 20-iteration recurrence."""
import argparse

import pytest
import torch
import torch.nn.functional as F

from fgt_b200 import synth
from oracle import raft_oracle as RO
from tests.util import REL_TOL, assert_close, load_golden

ARGS = dict(small=False, mixed_precision=False, alternate_corr=False)


@pytest.mark.parametrize("name", ["raft_small_i6", "raft_small_i20"])
def test_raft_oracle_small(name):
    g = load_golden(name)
    m = g["meta"]
    sd = synth.raft_state_dict(seed=m["seed"])
    im1, im2 = synth.raft_inputs(seed=m["seed"] + 1, H=m["H"], W=m["W"])
    with torch.no_grad():
        lo, up = RO.raft_forward(sd, im1, im2, iters=m["iters"])
    assert_close(lo, g["lo"], 2e-5, name + " low-res flow")
    assert_close(up, g["up"], 2e-5, name + " upsampled flow")


def test_raft_state_dict_contract_and_dataparallel_roundtrip():
    """The driver wraps the model in DataParallel to load 'module.'-prefixed keys, then unwraps
    (tool/video_inpainting.py:186-197)."""
    from fgt_b200.raft_model import RAFT
    sd = synth.raft_state_dict(seed=3)
    dp = torch.nn.DataParallel(RAFT(argparse.Namespace(**ARGS)))
    dp.load_state_dict({"module." + k: v for k, v in sd.items()})
    model = dp.module
    got = model.state_dict()
    assert set(got.keys()) == set(sd.keys()) and len(got) == 179
    for k, v in sd.items():
        assert torch.equal(got[k].cpu(), v), k   # DataParallel moves the module to cuda:0 when a GPU is present
    with pytest.raises(RuntimeError):
        model(*synth.raft_inputs(seed=0, H=64, W=64), iters=1, test_mode=True)  # CPU tensors: no fallback
    with pytest.raises(ValueError):
        RAFT(argparse.Namespace(small=True, mixed_precision=False, alternate_corr=False))


def _gpu_model(seed):
    from fgt_b200.raft_model import RAFT
    sd = synth.raft_state_dict(seed=seed)
    m = RAFT(argparse.Namespace(**ARGS))
    m.load_state_dict(sd)
    return m.cuda().eval(), sd


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["raft_small_i6", "raft_small_i20"])
def test_raft_gpu_small(name):
    g = load_golden(name)
    m = g["meta"]
    model, sd = _gpu_model(m["seed"])
    im1, im2 = synth.raft_inputs(seed=m["seed"] + 1, H=m["H"], W=m["W"])
    with torch.no_grad():
        lo, up = model(im1.cuda(), im2.cuda(), iters=m["iters"], test_mode=True)
    assert tuple(lo.shape) == (1, 2, m["H"] // 8, m["W"] // 8) and tuple(up.shape) == (1, 2, m["H"], m["W"])
    assert_close(lo, g["lo"], REL_TOL, name + " low vs reference golden")
    assert_close(up, g["up"], REL_TOL, name + " up vs reference golden")
    with torch.no_grad():
        olo, oup = RO.raft_forward(sd, im1, im2, iters=m["iters"])
    assert_close(lo, olo, REL_TOL, name + " low vs oracle")
    assert_close(up, oup, REL_TOL, name + " up vs oracle")


@pytest.mark.gpu
def test_raft_gpu_batch3_vs_oracle_and_single():
    """n=3 pairs in one call (one GEMM per layer over all pairs) against the oracle on the batch and
    against three single-pair calls (instance-norm partial sums are split differently, hence 1e-4 rather than
    bit equality); with a per-pair flow_init."""
    model, sd = _gpu_model(3)
    im1, im2 = synth.raft_inputs(seed=13, H=128, W=160, n=3)  # >= 16x16 at 1/8: no 1-pixel pyramid level
    with torch.no_grad():
        lo, up = model(im1.cuda(), im2.cuda(), iters=5, test_mode=True)
        olo, oup = RO.raft_forward(sd, im1, im2, iters=5)
    assert tuple(lo.shape) == (3, 2, 16, 20) and tuple(up.shape) == (3, 2, 128, 160)
    assert_close(lo, olo, REL_TOL, "batch low vs oracle")
    assert_close(up, oup, REL_TOL, "batch up vs oracle")
    with torch.no_grad():
        for i in range(3):
            lo1, up1 = model(im1[i:i + 1].cuda(), im2[i:i + 1].cuda(), iters=5, test_mode=True)
            assert_close(lo[i:i + 1], lo1, 1e-4, f"batch vs single pair {i}")
            assert_close(up[i:i + 1], up1, 1e-4, f"batch vs single pair {i} (up)")
        # warm start: flow_init shifts coords1 only (raft.py:121-122); zero init equals no init
        z0, zu = model(im1.cuda(), im2.cuda(), iters=2, flow_init=torch.zeros(3, 2, 16, 20).cuda(), test_mode=True)
        n0, nu = model(im1.cuda(), im2.cuda(), iters=2, test_mode=True)
    assert torch.equal(zu, nu)


@pytest.mark.gpu
def test_raft_gpu_full_480x864():
    """BASELINE config 3 geometry (the driver feeds RAFT 480x864 for 240x432 clips)."""
    g = load_golden("raft_full_i20")
    m = g["meta"]
    model, _ = _gpu_model(m["seed"])
    im1, im2 = synth.raft_inputs(seed=m["seed"] + 1, H=m["H"], W=m["W"])
    with torch.no_grad():
        lo, up = model(im1.cuda(), im2.cuda(), iters=m["iters"], test_mode=True)
    assert_close(lo, g["lo"], REL_TOL, "raft_full low")
    assert_close(up.reshape(-1).cpu()[torch.from_numpy(g["up_idx"])], g["up_val"], REL_TOL, "raft_full up samples")
    # non-test mode returns every iteration's upsampled flow; the last equals test-mode's
    with torch.no_grad():
        seq = model(im1.cuda(), im2.cuda(), iters=3, test_mode=False)
        lo3, up3 = model(im1.cuda(), im2.cuda(), iters=3, test_mode=True)
    assert len(seq) == 3 and torch.equal(seq[-1], up3)


@pytest.mark.gpu
def test_raft_gpu_720p():
    """BASELINE config 5 geometry: at imgH >= 350 the driver feeds RAFT the working resolution itself (720x1280 ->
    90x160 features, 14 400^2 all-pairs correlation = 829 MB at level 0)."""
    g = load_golden("raft_720p_i20")
    m = g["meta"]
    model, _ = _gpu_model(m["seed"])
    im1, im2 = synth.raft_inputs(seed=m["seed"] + 1, H=m["H"], W=m["W"])
    with torch.no_grad():
        lo, up = model(im1.cuda(), im2.cuda(), iters=m["iters"], test_mode=True)
    assert tuple(up.shape) == (1, 2, 720, 1280)
    assert_close(lo, g["lo"], REL_TOL, "raft_720p low")
    assert_close(up.reshape(-1).cpu()[torch.from_numpy(g["up_idx"])], g["up_val"], REL_TOL, "raft_720p up samples")


@pytest.mark.gpu
def test_raft_helper_kernels():
    from fgt_b200 import lib
    dev = torch.device("cuda:0")
    torch.manual_seed(5)
    # instance-norm statistics + normalise/relu/residual
    n, hh, ww, C = 2, 30, 46, 96
    x = torch.randn(n, hh, ww, C, device=dev) * 3 + 1.5
    res = torch.relu(torch.randn(n, hh, ww, C, device=dev))
    stats = torch.empty(n * C * 2, dtype=torch.float64, device=dev)
    out = torch.empty_like(x)
    osp = lib.empty_split(x.shape, dev)
    lib.chan_stats(x, n, hh * ww, C, stats)
    lib.instnorm_act(x, stats, n, hh * ww, C, relu=True, res=res, out=out, out_split=osp)
    torch.cuda.synchronize()
    ref = F.relu(F.relu(F.instance_norm(x.permute(0, 3, 1, 2).double())) + res.permute(0, 3, 1, 2).double())
    assert_close(out.permute(0, 3, 1, 2), ref, 1e-4, "instnorm_act")
    assert_close(lib.from_split(osp).permute(0, 3, 1, 2), ref, 1e-4, "instnorm_act split")
    # pyramid pooling (odd sizes floor like F.avg_pool2d)
    v = torch.randn(50, 15, 27, device=dev)
    p = torch.empty(50, 7, 13, device=dev)
    lib.avgpool2(v, 50, 15, 27, p)
    torch.cuda.synchronize()
    assert_close(p, F.avg_pool2d(v[:, None].double(), 2, stride=2)[:, 0], 1e-5, "avgpool2")
    # correlation lookup vs the reference-style grid_sample restatement (incl. out-of-range coords)
    h, w = 16, 24  # coarsest level 2x3 (a 1-pixel level would divide by zero in the reference sampler)
    npx = h * w
    lv0 = torch.randn(npx, h, w, device=dev)
    pyr = [lv0]
    for _ in range(3):
        pyr.append(F.avg_pool2d(pyr[-1][:, None], 2, stride=2)[:, 0].contiguous())
    coords = torch.stack([torch.rand(npx, device=dev) * (w + 8) - 4, torch.rand(npx, device=dev) * (h + 8) - 4], -1)
    look = torch.zeros(2, npx, 384, dtype=torch.bfloat16, device=dev)
    lib.corr_lookup(pyr, coords.contiguous(), npx, 4, look)
    torch.cuda.synchronize()
    c4 = coords.t().reshape(1, 2, h, w).cpu()
    ref = RO.corr_lookup([t[:, None].cpu() for t in pyr], c4)  # [1, 324, h, w]
    got = lib.from_split(look)[:, :324].reshape(h, w, 324).permute(2, 0, 1)[None]
    assert_close(got, ref, 1e-4, "corr_lookup")
    # convex upsampling
    mask = torch.randn(npx, 576, device=dev)
    flow = torch.randn(2, h, w, device=dev)
    up = torch.empty(2, 8 * h, 8 * w, device=dev)
    lib.convex_upsample(mask, flow, h, w, up)
    torch.cuda.synchronize()
    ref = RO.upsample_flow(flow[None].cpu(), mask.t().reshape(1, 576, h, w).cpu())
    assert_close(up[None], ref, 1e-4, "convex_upsample")
