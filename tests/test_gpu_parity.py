"""GPU parity tests: the CUDA path through the C ABI vs the oracle / the fixtures recorded from the reference.

Tolerances (BASELINE.json north_star): fp32 mode — corner offsets within 1e-3 px, warp sampling indices
bit-exact; bf16 mode — offsets within 0.05 px, covariance within 1 % relative.
"""
import numpy as np
import pytest
import torch

from conftest import unpack_masks
from cuahn_vio_b200 import synthetic as S
from oracle import uahn_oracle as O

pytestmark = pytest.mark.gpu

FP32_PX = 1e-3
BF16_PX = 0.05
BF16_COV_REL = 0.01


@pytest.fixture(scope="module")
def wfile():
    from cuahn_vio_b200 import build, weights
    build.build()
    return weights.synthetic_weights_file(0)


@pytest.fixture(scope="module")
def api():
    from cuahn_vio_b200 import api
    return api


def _masks_for(n, seed0=20240 + 10 ** 6):
    return [S.torch_dropout_masks(seed0 + i) for i in range(n)]


def _pack(api, masks_list):
    return np.stack([api.pack_keep_masks(m) for m in masks_list])


def _oracle_batch(prev, curr, sd, masks_list, priors, show_error, btr=3):
    return O.forward_batch(prev, curr, sd, masks_list, priors, show_error, btr)


# ---------------------------------------------------------------------------------------------------------
def test_stage_dlt_matches_reference(api, wfile, golden_stages):
    """The DLT solve of head_kernels.cu: the closed form of the fixed source rectangle."""
    g = golden_stages
    with api.Uahn(wfile, "prior1", max_batch=64) as net:
        Hg = net.stage_dlt(g["dlt_offsets"].reshape(-1, 8))
        assert np.abs(Hg - g["dlt_H"]).max() < 2e-4           # fp32 torch.inverse noise (cond ~1.8e5)
        assert np.abs(Hg[0] - np.eye(3)).max() < 1e-6         # DLT(p, p) = I
        rng = np.random.default_rng(3)
        off = ((rng.random((64, 4, 2)) * 2 - 1) * 30).astype(np.float32)
        Hd = net.stage_dlt(off.reshape(-1, 8))
        pts0 = O.origin_4pt().unsqueeze(0).double()
        for i in range(64):
            # fp64 torch reference of the same solve: the kernel accumulates in fp64
            Hr = O.dlt_solve(pts0, pts0 + torch.from_numpy(off[i:i + 1]).double())[0].numpy()
            assert np.abs(Hd[i] - Hr).max() / max(1.0, np.abs(Hr).max()) < 1e-6
            # and it must map the corners onto corners + offsets
            p = Hd[i].astype(np.float64) @ np.concatenate([S.ORIGIN_4PT.T, np.ones((1, 4))])
            assert np.abs((p[:2] / p[2]).T - (S.ORIGIN_4PT + off[i])).max() < 2e-3


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_stage_warp_indices_bit_exact(api, wfile, golden_stages, precision):
    """fp32 handle: the exact coordinate chain.  bf16 handle: the product path's fast coordinates with the exact fallback
    near integer boundaries (image_kernels.cu CM_FAST) — the indices must be just as bit-exact; its bilinear weights may
    move by 3e-4 px, i.e. 3e-4 x the local grey-level step in value."""
    g = golden_stages
    vtol = 2e-6 if precision == "fp32" else 4e-4
    with api.Uahn(wfile, "prior1", precision=precision, max_batch=32) as net:
        img = np.repeat(g["warp_src_u8"][None], 4, 0)
        out, ix, iy = net.stage_warp(img, g["warp_H"])
        assert np.array_equal(ix, g["warp_ix"]) and np.array_equal(iy, g["warp_iy"])   # fixtures from the reference
        assert np.abs(out - g["warp_out"]).max() < vtol
        # random homographies incl. large ones that leave the image; oracle computed here
        rng = np.random.default_rng(11)
        Hs = []
        NH = 32      # 2.3 M coordinates: the shared-reciprocal division fast path and (large H) the IEEE fallback
        for t in range(NH):
            disp = (rng.random((4, 2)) * 2 - 1) * (20 if t < 24 else 150)
            Hs.append(S.dlt_numpy(S.ORIGIN_4PT.astype(np.float64), S.ORIGIN_4PT + disp).astype(np.float32))
        Hs = np.stack(Hs)
        img8 = np.repeat(g["warp_src_u8"][None], NH, 0)
        out, ix, iy = net.stage_warp(img8, Hs)
        src = O.u8_to_unit(g["warp_src_u8"])
        mism = 0
        for t in range(NH):
            Ht = torch.from_numpy(Hs[t])
            rix, riy, _, _ = O.sample_indices(Ht)
            inside = (rix.numpy() >= -1) & (rix.numpy() <= 320) & (riy.numpy() >= -1) & (riy.numpy() <= 224)
            mism += int((ix[t][inside] != rix.numpy()[inside]).sum() + (iy[t][inside] != riy.numpy()[inside]).sum())
            assert np.abs(out[t] - O.warp_image(src, Ht)[0, 0].numpy()).max() < vtol
        assert mism == 0
        # integer translations: every sample sits exactly on a pixel (the fast path's worst case: all fallbacks)
        Ht = np.stack([np.eye(3, dtype=np.float32)] * 3)
        Ht[1, 0, 2], Ht[1, 1, 2] = 5.0, -3.0
        Ht[2, 0, 2], Ht[2, 1, 2] = -17.0, 40.0
        out, ix, iy = net.stage_warp(img8[:3], Ht)
        for t in range(3):
            rix, riy, _, _ = O.sample_indices(torch.from_numpy(Ht[t]))
            inside = (rix.numpy() >= -1) & (rix.numpy() <= 320) & (riy.numpy() >= -1) & (riy.numpy() <= 224)
            assert np.array_equal(ix[t][inside], rix.numpy()[inside]) and np.array_equal(iy[t][inside], riy.numpy()[inside])
            assert np.abs(out[t] - O.warp_image(src, torch.from_numpy(Ht[t]))[0, 0].numpy()).max() < vtol


def test_warp_identity_and_outside(api, wfile):
    with api.Uahn(wfile, "prior1", max_batch=2) as net:
        rng = np.random.default_rng(0)
        img = rng.integers(0, 256, (2, 224, 320), dtype=np.uint8)
        far = np.eye(3, dtype=np.float32); far[0, 2] = 1000.0
        out, _, _ = net.stage_warp(img, np.stack([np.eye(3, dtype=np.float32), far]))
        assert np.abs(out[0] - img[0].astype(np.float32) / np.float32(255)).max() < 1e-4
        assert np.abs(out[1]).max() == 0.0


@pytest.mark.parametrize("variant,show", [("prior3", True), ("full", True), ("prior2", False), ("prior1", False)])
def test_e2e_fp32_vs_oracle(api, wfile, synth_sd, variant, show):
    n = 4
    prev, curr, gt, prior = S.synthetic_batch(n, start=100)
    masks = _masks_for(n)
    btr = {"prior3": 3, "prior2": 2, "prior1": 1, "full": 3}[variant]
    pr = None if variant == "full" else prior
    om, oc, oe = _oracle_batch(prev, curr, synth_sd, masks, pr, show, btr)
    with api.Uahn(wfile, variant, show_error=show, precision="fp32", max_batch=n) as net:
        m, c, e = net.infer_batch(prev, curr, pr, keep_masks=_pack(api, masks), want_error=show)
        assert np.abs(m - om).max() < FP32_PX, np.abs(m - om).max()
        assert np.abs(c - oc).max() <= 2e-4 * np.abs(oc).max()
        # symmetric up to fp32 rounding, like the reference's own H·V·Hᵀ (Eigen::Map reads it transposed)
        assert np.abs(c - np.swapaxes(c, 1, 2)).max() <= 1e-6 * np.abs(c).max()
        if show:
            # 255-scaled grey levels; the max sits on the warped image border (value jump x 1e-4 px of H noise)
            assert np.abs(e - oe).max() < 0.25 and np.abs(e - oe).mean() < 1e-3
        # stage taps vs the oracle's taps for pair 0
        t = O.Taps()
        O.forward(O.u8_to_unit(prev[0]), O.u8_to_unit(curr[0]), synth_sd, masks[0],
                  None if pr is None else torch.from_numpy(pr[0]).view(1, 1, 4, 2), show, btr, taps=t)
        for b in (1, 2, 3):
            if b in t.d:
                assert np.abs(net.debug_read(f"d{b}", (n, 8))[0] - t.d[b].numpy()).max() < 2e-4
                assert np.abs(net.debug_read(f"H{b}", (n, 3, 3))[0] - t.H[b][0].numpy()).max() < 2e-4
                assert np.abs(net.debug_read(f"x{b}", (n,) + tuple(t.x_in[b].shape[1:]))[0] - t.x_in[b][0].numpy()).max() < 2e-4   # image gradient x H noise
        f4 = net.debug_read("feat4", (n, 256, 4, 5))[0]
        ref4 = t.feat[4][0].numpy()
        assert np.abs(f4 - ref4).max() < 1e-4 * max(1.0, np.abs(ref4).max())
        assert np.abs(net.debug_read("mcmean", (n, 16, 8))[0] - t.mc_mean.reshape(16, 8).numpy()).max() < 2e-4


def test_e2e_fp32_vs_reference_fixtures(api, wfile, golden_e2e):
    g = golden_e2e
    masks = np.stack([api.pack_keep_masks(unpack_masks(g, i)) for i in range(3)])
    for variant in ("prior3", "full"):
        with api.Uahn(wfile, variant, show_error=True, precision="fp32", max_batch=3) as net:
            m, c, e = net.infer_batch(g["prev"], g["curr"], g["prior"] if variant == "prior3" else None,
                                      keep_masks=masks, want_error=True)
            for i in range(3):
                assert np.abs(m[i] - g[f"flow_{variant}_{i}"]).max() < FP32_PX
                assert np.abs(c[i] - g[f"cov_{variant}_{i}"]).max() < 2e-4 * np.abs(g[f"cov_{variant}_{i}"]).max()
                assert abs(float(e[i].astype(np.float64).sum()) - float(g[f"errsum_{variant}_{i}"])) < 1e-4 * float(g[f"errsum_{variant}_{i}"])
            assert np.abs(e[0] - g[f"err_{variant}_0"]).max() < 0.25


def test_batch_equals_loop_and_is_deterministic(api, wfile):
    n = 6
    prev, curr, _, prior = S.synthetic_batch(n, start=300)
    with api.Uahn(wfile, "prior3", precision="fp32", max_batch=n) as net:
        m, c, _ = net.infer_batch(prev, curr, prior, seed=5, first_pair=40)
        m2, c2, _ = net.infer_batch(prev, curr, prior, seed=5, first_pair=40)
        assert np.array_equal(m, m2) and np.array_equal(c, c2)
        for i in range(n):
            mi, ci, _ = net.infer_batch(prev[i:i + 1], curr[i:i + 1], prior[i:i + 1], seed=5, first_pair=40 + i)
            assert np.array_equal(mi[0], m[i]) and np.array_equal(ci[0], c[i])
        m3, _, _ = net.infer_batch(prev, curr, prior, seed=6, first_pair=40)
        assert not np.array_equal(m, m3)     # MC dropout really is stochastic in the seed


def test_pipelined_submissions_match_blocking_call(api, wfile):
    import torch as _t
    n = 4
    prev, curr, _, prior = S.synthetic_batch(3 * n, start=800)
    with api.Uahn(wfile, "prior3", precision="bf16", max_batch=n) as net:
        ref = [net.infer_batch(prev[i * n:(i + 1) * n], curr[i * n:(i + 1) * n], prior[i * n:(i + 1) * n], seed=2,
                               first_pair=10 * i) for i in range(3)]
        pin = lambda a: _t.from_numpy(np.ascontiguousarray(a)).pin_memory()
        hp, hc, hq = pin(prev), pin(curr), pin(prior.reshape(-1, 8))
        outs = [(_t.empty(n, 8).pin_memory(), _t.empty(n, 64).pin_memory()) for _ in range(3)]
        for i in range(3):       # three submissions in flight over two staging sets
            net.submit_batch_ptrs(n, hp[i * n:].data_ptr(), hc[i * n:].data_ptr(), hq[i * n:].data_ptr(),
                                  outs[i][0].data_ptr(), outs[i][1].data_ptr(), seed=2, first_pair=10 * i)
        net.wait()
        for i in range(3):
            assert np.array_equal(outs[i][0].numpy(), ref[i][0])
            assert np.array_equal(outs[i][1].numpy().reshape(n, 8, 8), ref[i][1])


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_philox_and_explicit_masks_agree(api, wfile, precision):
    """In-kernel Philox masks == the same masks replayed as explicit bytes (bf16: fused masked-A GEMM producer;
    fp32: mc_expand), for a batch that leaves the last 128-row GEMM tile partly empty."""
    n = 5
    prev, curr, _, prior = S.synthetic_batch(n, start=900)
    packed = np.stack([api.philox_keep_masks(77, 11 + i) for i in range(n)])
    with api.Uahn(wfile, "prior3", precision=precision, max_batch=n) as net:
        m0, c0, _ = net.infer_batch(prev, curr, prior, seed=77, first_pair=11)
        m1, c1, _ = net.infer_batch(prev, curr, prior, keep_masks=packed)
        assert np.array_equal(m0, m1) and np.array_equal(c0, c1)


def test_fused_mc_gemm_matches_expand_path(api, wfile):
    """bf16, n >= 64: the masked-A GEMM producer (keep bits, no materialised masks) vs the expand + GEMM path that small
    batches take; Philox masks and explicit masks; a batch that leaves the last 128-row tile partly empty."""
    n = 70
    prev, curr, _, prior = S.tiled_batch(n, unique=6)
    packed = np.stack([api.philox_keep_masks(5, 100 + i) for i in range(n)])
    with api.Uahn(wfile, "prior3", precision="bf16", max_batch=n) as net:
        m_big, c_big, _ = net.infer_batch(prev, curr, prior, seed=5, first_pair=100)          # fused, Philox bits
        m_exp, c_exp, _ = net.infer_batch(prev, curr, prior, keep_masks=packed)               # fused, explicit masks
        assert np.array_equal(m_big, m_exp) and np.array_equal(c_big, c_exp)
        # expand + plain GEMM path, 12 pairs at a time (9..63 pairs: above the latency-path kernels, whose split-K FC8 sums in
        # another order and would move the cascade by bf16 flips; below the fused MC GEMM)
        for lo in (0, 32, 58):
            m6, c6, _ = net.infer_batch(prev[lo:lo + 12], curr[lo:lo + 12], prior[lo:lo + 12], seed=5, first_pair=100 + lo)
            assert np.abs(m6 - m_big[lo:lo + 12]).max() < 2e-3, np.abs(m6 - m_big[lo:lo + 12]).max()
            assert np.abs(c6 - c_big[lo:lo + 12]).max() <= 2e-3 * np.abs(c6).max()


def test_latency_path_mc_kernel_is_the_expand_path_bit_for_bit(api, wfile):
    """<= 8 pairs, bf16: dropout expansion + first MC-head layer of both heads in one CUDA-core kernel vs the three launches
    it replaces (mc_expand + 2 x mc_fc1_small): the same bf16 values in the same summation order."""
    import os
    n = 5
    prev, curr, _, prior = S.synthetic_batch(n, start=1200)
    packed = np.stack([api.philox_keep_masks(21, 300 + i) for i in range(n)])
    res = {}
    for fused in (True, False):
        if not fused:
            os.environ["UAHN_NO_MC_SMALL_FUSED"] = "1"
        try:
            with api.Uahn(wfile, "prior3", precision="bf16", max_batch=n) as net:
                res[fused] = (net.infer_batch(prev, curr, prior, seed=21, first_pair=300)[:2],
                              net.infer_batch(prev, curr, prior, keep_masks=packed)[:2])
        finally:
            os.environ.pop("UAHN_NO_MC_SMALL_FUSED", None)
    for a, b in zip(res[True], res[False]):
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    assert np.array_equal(res[True][0][0], res[True][1][0])           # Philox == the same masks replayed explicitly


def test_sequence_submission_matches_pairwise_call(api, wfile):
    """uahn_submit_sequence: pair i = (frames[i], frames[i+1]), every frame uploaded once."""
    import torch as _t
    nf = 6
    frames, gt, prior = S.synthetic_sequence(nf, seed=77)
    assert np.abs(gt).max() < 16 and np.abs(gt).max() > 0.05           # a smooth walk, not a static scene
    with api.Uahn(wfile, "prior3", precision="bf16", max_batch=nf - 1) as net:
        ref_m, ref_c, _ = net.infer_batch(frames[:-1], frames[1:], prior, seed=4, first_pair=3)
        pin = lambda a: _t.from_numpy(np.ascontiguousarray(a)).pin_memory()
        hf, hq = pin(frames), pin(prior.reshape(-1, 8))
        outs = [(_t.empty(nf - 1, 8).pin_memory(), _t.empty(nf - 1, 64).pin_memory()) for _ in range(3)]
        for m, c in outs:       # three submissions in flight over two staging sets
            net.submit_sequence_ptrs(nf, hf.data_ptr(), hq.data_ptr(), m.data_ptr(), c.data_ptr(), seed=4, first_pair=3)
        net.wait()
        for m, c in outs:
            assert np.array_equal(m.numpy(), ref_m) and np.array_equal(c.numpy().reshape(nf - 1, 8, 8), ref_c)
        with pytest.raises(api.UahnError):           # one frame is not a pair (HomographyNet.cpp:155-158)
            net.submit_sequence_ptrs(1, hf.data_ptr(), hq.data_ptr(), outs[0][0].data_ptr(), outs[0][1].data_ptr())
        # the network, seeded with the noisy prior, must land closer to the ground truth than chance would
        assert np.isfinite(ref_m).all()


def test_philox_masks_replayed_through_oracle(api, wfile, synth_sd):
    n = 2
    prev, curr, _, prior = S.synthetic_batch(n, start=500)
    with api.Uahn(wfile, "prior3", precision="fp32", max_batch=n) as net:
        m, c, _ = net.infer_batch(prev, curr, prior, seed=1234, first_pair=7)
    masks = []
    for i in range(n):
        k = api.philox_keep_masks(1234, 7 + i).astype(np.float32) * np.float32(1.0 / 0.95)
        masks.append(tuple(torch.from_numpy(np.ascontiguousarray(a)) for a in
                           (k[0, :, :5120], k[0, :, 5120:], k[1, :, :5120], k[1, :, 5120:])))
    om, oc, _ = _oracle_batch(prev, curr, synth_sd, masks, prior, False)
    assert np.abs(m - om).max() < FP32_PX and np.abs(c - oc).max() < 2e-4 * np.abs(oc).max()


def test_streaming_call_surface(api, wfile):
    prev, curr, _, prior = S.synthetic_batch(3, start=700)
    frames = [prev[0], curr[0], curr[1]]
    with api.Uahn(wfile, "prior3", show_error=True, precision="fp32", max_batch=1) as net:
        net.load_image(frames[0], 1.0)
        with pytest.raises(api.UahnError):           # HomographyNet.cpp:155-158
            net.infer(prior[0].reshape(8))
        assert net.latest_inference_time == -1.0
        net.load_image(frames[1], 2.0)
        assert net.img_counter == 2 and net.latest_inference_time == 2.0
        m, c, e = net.infer(prior[0].reshape(8), seed=9, pair_index=0, want_error=True)
        mb, cb, eb = net.infer_batch(frames[0][None], frames[1][None], prior[:1], seed=9, first_pair=0, want_error=True)
        assert np.array_equal(m.astype(np.float32), mb[0]) and np.array_equal(c.astype(np.float32), cb[0])
        assert np.array_equal(e, np.clip(eb[0], 0, 255).astype(np.uint8))
        net.load_image(frames[2], 3.0)               # prev <- curr slot flip
        m2, _, _ = net.infer(prior[1].reshape(8), seed=9, pair_index=1)
        mb2, _, _ = net.infer_batch(frames[1][None], frames[2][None], prior[1:2], seed=9, first_pair=1)
        assert np.array_equal(m2.astype(np.float32), mb2[0])
    # CUDA-graph replay (third call onwards) must reproduce the eager results and honour per-call seeds
    for precision in ("fp32", "bf16"):
        with api.Uahn(wfile, "prior3", show_error=True, precision=precision, max_batch=1) as net:
            net.load_image(frames[0], 1.0)
            net.load_image(frames[1], 2.0)
            ref = [net.infer(prior[0].reshape(8), seed=3, pair_index=i, want_error=(i % 2 == 0)) for i in range(2)]   # eager
            l0 = net.launch_count
            again = [net.infer(prior[0].reshape(8), seed=3, pair_index=i, want_error=(i % 2 == 0)) for i in range(2)]  # graphs
            assert net.launch_count - l0 >= 2 * 20            # replays are counted as the kernels they contain
            for (m0, c0, e0), (m1, c1, e1) in zip(ref, again):
                assert np.array_equal(m0, m1) and np.array_equal(c0, c1)
                assert (e0 is None and e1 is None) or np.array_equal(e0, e1)
            m5, _, _ = net.infer(prior[0].reshape(8), seed=3, pair_index=5)
            assert not np.array_equal(m5, ref[0][0])
            net.load_image(frames[2], 3.0)                     # other ring slot -> its own graph
            mg, _, _ = net.infer(prior[1].reshape(8), seed=3, pair_index=1)
            mb, _, _ = net.infer_batch(frames[1][None], frames[2][None], prior[1:2], seed=3, first_pair=1)
            assert np.array_equal(mg.astype(np.float32), mb[0])
    hn = api.HomographyNet(wfile, use_prior=True, precision="fp32")
    hn.load_current_img(frames[0], 0.1)
    hn.network_inference(prior[0].reshape(8), 0)     # prints, leaves outputs untouched
    assert np.all(hn.get_pred_mean() == 0)
    hn.load_current_img(frames[1], 0.2)
    hn.network_inference(prior[0].reshape(8), 0)
    assert np.abs(hn.get_pred_mean()).max() > 0 and hn.get_latest_inference_time() == 0.2


def test_error_paths(api, wfile):
    with api.Uahn(wfile, "prior3", precision="fp32", max_batch=2) as net:
        prev, curr, _, prior = S.synthetic_batch(3, start=0)
        with pytest.raises(api.UahnError):
            net.infer_batch(prev, curr, prior)              # n > max_batch
        with pytest.raises(api.UahnError):
            net.infer_batch(prev[:1], curr[:1], None)       # prior variant without prior
        with pytest.raises(api.UahnError):
            net.load_image(np.zeros((100, 100), np.uint8))


# ---- per-layer conv parity (fp32 SIMT and bf16 tcgen05 implicit GEMM) ---------------------------------------
LAYERS = [  # name, Cin, Hin, Win, Cout, k, stride   (model_to_trace.py:93-113, 210-216)
    ("block_1_1", 2, 28, 40, 128, 7, 2), ("block_1_2", 128, 14, 20, 128, 5, 2), ("block_1_3", 128, 7, 10, 256, 3, 2),
    ("block_2_1", 2, 56, 80, 64, 7, 2), ("block_2_2", 64, 28, 40, 128, 5, 2), ("block_2_4", 256, 7, 10, 256, 3, 2),
    ("block_3_0", 2, 112, 160, 16, 7, 1), ("block_3_1", 16, 112, 160, 32, 5, 2), ("block_3_2", 32, 56, 80, 64, 3, 2),
    ("block_4_0", 2, 224, 320, 8, 7, 1), ("block_4_1", 8, 224, 320, 16, 5, 2), ("block_4_2", 16, 112, 160, 32, 3, 2),
    ("block_4_3", 32, 56, 80, 64, 3, 2), ("block_4_4", 64, 28, 40, 128, 3, 2), ("block_4_5", 128, 14, 20, 256, 3, 2),
]


def _bf16_round(t: torch.Tensor) -> torch.Tensor:
    return t.to(torch.bfloat16).to(torch.float32)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_conv_layers_vs_torch(api, wfile, synth_sd, precision):
    n = 3     # odd batch: exercises the partial last M tile
    g = torch.Generator().manual_seed(4)
    with api.Uahn(wfile, "full", precision=precision, max_batch=n) as net:
        for name, cin, hin, win, cout, k, s in LAYERS:
            x = torch.rand(n, cin, hin, win, generator=g) * 2 - 0.5
            pre = "model_last_block_list.0." if name.startswith("block_4") else "model_part1."
            w, b = synth_sd[pre + name + ".0.weight"], synth_sd[pre + name + ".0.bias"]
            if precision == "bf16":
                x = _bf16_round(x)
                w = _bf16_round(w)
            ref = torch.nn.functional.leaky_relu(
                torch.nn.functional.conv2d(x.double(), w.double(), b.double(), stride=s, padding=(k - 1) // 2), 0.1).float()
            out = net.stage_conv(name, x.numpy(), tuple(ref.shape[1:]))
            err = np.abs(out - ref.numpy()).max()
            scale = max(1.0, float(ref.abs().max()))
            tol = 2e-5 * scale if precision == "fp32" else 6e-3 * scale    # bf16: output rounding 2^-9
            assert err < tol, (name, precision, err, scale)


SMALL_M_LAYERS = [  # the layers the latency path runs as split-K over a cluster (conv_small_m.cu): M = 20 or 70 rows per pair
    ("block_1_2", 128, 14, 20, 128, 5, 2), ("block_1_3", 128, 7, 10, 256, 3, 2), ("block_2_3", 128, 14, 20, 256, 3, 2),
    ("block_2_4", 256, 7, 10, 256, 3, 2), ("block_3_4", 128, 14, 20, 256, 3, 2), ("block_3_5", 256, 7, 10, 256, 3, 2),
    ("block_4_5", 128, 14, 20, 256, 3, 2), ("block_4_6", 256, 7, 10, 256, 3, 2),
]


def test_small_m_split_k_layers_vs_torch_and_batch_independent(api, wfile, synth_sd):
    """bf16 latency path: every deep layer by name at 1 and 2 pairs (and 8 for the 4x5 layers) against torch fp64 on the
    bf16-rounded operands; a 2-pair call is bit for bit two 1-pair calls (the K split never depends on the batch)."""
    g = torch.Generator().manual_seed(11)
    with api.Uahn(wfile, "full", precision="bf16", max_batch=8) as net:
        for name, cin, hin, win, cout, k, s in SMALL_M_LAYERS:
            pre = "model_last_block_list.0." if name.startswith("block_4") else "model_part1."
            w, b = _bf16_round(synth_sd[pre + name + ".0.weight"]), synth_sd[pre + name + ".0.bias"]
            ho, wo = (hin + 2 * ((k - 1) // 2) - k) // s + 1, (win + 2 * ((k - 1) // 2) - k) // s + 1
            for n in (1, 2, 8):
                x = _bf16_round(torch.rand(n, cin, hin, win, generator=g) * 2 - 0.5)
                ref = torch.nn.functional.leaky_relu(
                    torch.nn.functional.conv2d(x.double(), w.double(), b.double(), stride=s, padding=(k - 1) // 2), 0.1).float()
                l0 = net.launch_count
                out = net.stage_conv(name, x.numpy(), (cout, ho, wo))
                assert net.launch_count - l0 == 1
                scale = max(1.0, float(ref.abs().max()))
                assert np.abs(out - ref.numpy()).max() < 6e-3 * scale, (name, n)
                if n == 2:
                    for i in range(2):
                        one = net.stage_conv(name, x[i:i + 1].numpy(), (cout, ho, wo))
                        assert np.array_equal(one[0], out[i]), (name, i)


def test_fused_front_matches_per_layer_kernels(api, wfile):
    """Blocks 3/4: the fused conv0+conv1 kernel vs the two separate tcgen05 kernels (same bf16 intermediate)."""
    import os
    n = 3
    prev, curr, _, prior = S.synthetic_batch(n, start=600)
    outs = {}
    for fuse in (True, False):
        if not fuse:
            os.environ["UAHN_NO_FUSE"] = "1"
        try:
            with api.Uahn(wfile, "prior3", precision="bf16", max_batch=n) as net:
                m, c, _ = net.infer_batch(prev, curr, prior, seed=4)
                outs[fuse] = (m, c, net.debug_read("act:block_3_1", (n, 32, 56, 80)),
                              net.debug_read("act:block_4_1", (n, 16, 112, 160)))
        finally:
            os.environ.pop("UAHN_NO_FUSE", None)
    # block 3's input is identical in both runs; block 4's differs in a few bf16 values because H3 moved by ~1e-2 px
    for k, max_frac in ((2, 0.005), (3, 0.3)):
        a, b = outs[True][k], outs[False][k]
        scale = max(1.0, float(np.abs(b).max()))
        assert np.abs(a - b).max() <= 2.0 ** -7 * scale        # one bf16 ulp at the top of the range
        assert np.mean(a != b) < max_frac
    # both paths sit inside the bf16 budget around the oracle; between themselves they differ by bf16 flips that the
    # cascade (H3 -> warp -> block 4) amplifies
    assert np.abs(outs[True][0] - outs[False][0]).max() < BF16_PX


def test_texture_warp_matches_shared_memory_warp(api, wfile):
    """bf16, more than 8 pairs: the texture-gather warp kernel (taps by tld4 from the cell array) against the shared-memory
    kernel on the same inputs — identity (every sample on the integer grid: exact chain), far-outside and partly-outside
    homographies (clamp into the zero margin) and ordinary ones; all three pooling factors."""
    import os
    n = 12
    prev, curr, _, prior = S.synthetic_batch(n, start=640)
    prior = prior.copy()
    prior[0] = 0.0                                   # identity
    prior[1] = 400.0                                 # every sample outside the image
    prior[2] = np.array([[-30, -25], [28, -31], [-27, 30], [31, 26]], np.float32)    # zoom: all four borders leave the image
    prior[3, :, 0] += 21.0                           # pure shift: the left border samples the zero padding
    outs = {}
    for tex, env in ((True, None), (False, "UAHN_NO_TEX_WARP")):
        if env:
            os.environ[env] = "1"
        try:
            with api.Uahn(wfile, "prior3", precision="bf16", max_batch=n) as net:
                m, c, _ = net.infer_batch(prev, curr, prior, seed=4)
                outs[tex] = (m, c, net.debug_read("x2", (n, 2, 56, 80)), net.debug_read("x3", (n, 2, 112, 160)),
                             net.debug_read("x4", (n, 2, 224, 320)))
        finally:
            if env:
                os.environ.pop(env, None)
    # x2 sees the same H in both runs: the two kernels may differ by the rounding of a tap sum (b / 255 per tap against
    # one scaling of the integer sum), i.e. by one bf16 ulp in a few pixels.  x3 / x4 follow H2 / H3, which those flips move
    # by ~1e-3 px.
    for k, max_frac in ((2, 0.02), (3, 0.3), (4, 0.3)):
        a, b = outs[True][k], outs[False][k]
        assert np.array_equal(a[:, 0], b[:, 0])                # previous-frame channel: exact integer sums in both
        assert np.abs(a - b).max() <= 2.0 ** -8                # one bf16 ulp below 1.0
        assert np.mean(a != b) < max_frac
    assert np.abs(outs[True][2][1, 1]).max() == 0.0            # far outside: zeros
    assert np.abs(outs[True][0] - outs[False][0]).max() < BF16_PX


def test_texture_warp_sees_every_refill_of_the_cell_array(api, wfile):
    """The cell array is rewritten by every batch call and read through the (non-coherent) texture path, with programmatic
    dependent launch between the kernels: alternate two input sets through one handle — every call must reproduce the first
    result of its set bit for bit (a stale texture line or a fill / gather overlap would not)."""
    n = 40
    sets = [S.synthetic_batch(n, start=700), S.synthetic_batch(n, start=760)]
    with api.Uahn(wfile, "prior3", precision="bf16", max_batch=n) as net:
        first = {}
        for it in range(8):
            k = it & 1
            prev, curr, _, prior = sets[k]
            m, c, _ = net.infer_batch(prev, curr, prior, seed=9)
            x4 = net.debug_read("x4", (n, 2, 224, 320))
            if k not in first:
                first[k] = (m.copy(), c.copy(), x4.copy())
            else:
                assert np.array_equal(m, first[k][0]) and np.array_equal(c, first[k][1]) and np.array_equal(x4, first[k][2]), it
        assert not np.array_equal(first[0][2], first[1][2])


def test_cta_pair_deep_layers_match_single_cta_kernels(api, wfile):
    """Deep conv layers (Cin % 64 == 0) at a batch large enough for the CTA-pair kernels (tcgen05.mma.cta_group::2, half
    of each B stage per CTA) vs the one-CTA im2col kernels: the same accumulation order, so every activation and output
    is bit-identical.  1090 pairs -> 171 M tiles in the last layers: the odd count leaves the peer CTA of the last
    unit with a tile entirely past the end of M."""
    import os
    n = 1090
    prev, curr, _, prior = S.tiled_batch(n, unique=8)
    outs = {}
    for pair in (True, False):
        if not pair:
            os.environ["UAHN_NO_IGEMM_PAIR"] = "1"
        try:
            with api.Uahn(wfile, "prior3", precision="bf16", max_batch=n) as net:
                m, c, _ = net.infer_batch(prev, curr, prior, seed=8)
                outs[pair] = (m, c, net.debug_read("feat4", (n, 256, 4, 5)), net.debug_read("act:block_2_2", (n, 128, 14, 20)))
        finally:
            os.environ.pop("UAHN_NO_IGEMM_PAIR", None)
    for a, b in zip(outs[True], outs[False]):
        assert np.array_equal(a, b)
    assert np.isfinite(outs[True][0]).all() and np.abs(outs[True][2]).max() > 0


def test_edge_inputs_fp32_vs_oracle(api, wfile, synth_sd):
    """Degenerate frames and a prior that throws the warp (mostly) outside the image: black, saturated, identical
    frames, a 250-px shift; n == max_batch and n < max_batch through the same handle."""
    prev, curr, _, prior = S.synthetic_batch(2, start=950)
    z = np.zeros((224, 320), np.uint8)
    frames_p = np.stack([z, z + 255, prev[0], prev[1], prev[1]])
    frames_c = np.stack([z, z + 255, prev[0], curr[1], curr[1]])
    pri = np.zeros((5, 4, 2), np.float32)
    pri[3] = prior[1] + np.float32(250.0)          # warp window almost entirely outside the frame
    pri[4] = prior[1]
    masks = _masks_for(5)
    om, oc, oe = _oracle_batch(frames_p, frames_c, synth_sd, masks, pri, True)
    assert np.isfinite(om).all() and np.isfinite(oc).all()
    with api.Uahn(wfile, "prior3", show_error=True, precision="fp32", max_batch=5) as net:
        m, c, e = net.infer_batch(frames_p, frames_c, pri, keep_masks=_pack(api, masks), want_error=True)   # n == max_batch
        assert np.isfinite(m).all() and np.isfinite(c).all()
        assert np.abs(m - om).max() < FP32_PX, np.abs(m - om).max()
        assert np.abs(c - oc).max() <= 5e-4 * np.abs(oc).max()
        assert np.abs(e - oe).max() < 0.05          # grey levels of 255: the <= 1e-4 px difference of H_total times the image gradient
        m1, c1, _ = net.infer_batch(frames_p[3:4], frames_c[3:4], pri[3:4], keep_masks=_pack(api, masks[3:4]))   # n < max_batch
        assert np.array_equal(m1[0], m[3]) and np.array_equal(c1[0], c[3])
        with pytest.raises(api.UahnError):
            net.infer_batch(frames_p[:0], frames_c[:0], pri[:0])                                            # empty batch


@pytest.mark.parametrize("variant", ["prior3", "full"])
def test_e2e_bf16_vs_oracle(api, wfile, synth_sd, variant):
    n = 5
    prev, curr, gt, prior = S.synthetic_batch(n, start=200)
    masks = _masks_for(n)
    pr = None if variant == "full" else prior
    om, oc, oe = _oracle_batch(prev, curr, synth_sd, masks, pr, True)
    with api.Uahn(wfile, variant, show_error=True, precision="bf16", max_batch=n) as net:
        m, c, e = net.infer_batch(prev, curr, pr, keep_masks=_pack(api, masks), want_error=True)
        assert np.abs(m - om).max() < BF16_PX, np.abs(m - om).max()
        diag = np.abs(np.diagonal(oc, axis1=1, axis2=2)).max()
        assert np.abs(c - oc).max() <= BF16_COV_REL * diag, np.abs(c - oc).max() / diag
        assert np.abs(e - oe).mean() < 0.25      # grey levels of 255; follows the <=0.05 px homography difference
