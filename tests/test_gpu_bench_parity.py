"""GPU parity at the configurations bench.py measures (VERDICT r01 "Next round" #1): the kernels that only run at large
batch — CTA-pair im2col implicit GEMM (>= 1 tile per SM), fused masked-A MC GEMM (n >= 64), its CTA-pair form
(n >= 256), the CTA-pair fused block fronts — against the ORACLE directly, not against sibling kernels.

Tolerances (BASELINE.json north_star), per pair and per element:
  * bf16: corner offsets within 0.05 px;
  * bf16: covariance within 1 % relative, element by element over the four 2x2 diagonal blocks, each element measured
    against the scale of ITS OWN pair and block: |dC_jk| <= 0.01 * sqrt(C_jj * C_kk) (for the diagonal entries that is
    exactly |dC_jj| <= 0.01 * C_jj; an off-diagonal entry of a near-axis-aligned block is ~0 and has no scale of its own);
  * entries outside the diagonal blocks are exactly 0 on both sides (model_to_trace.py:313-317).
Synthetic weights (the checkpoint is not shipped) — the tolerances have to be re-validated on the real file.
"""
import numpy as np
import pytest
import torch

from cuahn_vio_b200 import synthetic as S
from oracle import uahn_oracle as O

pytestmark = pytest.mark.gpu

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


def philox_masks_for_oracle(api, seed, pair):
    """The in-kernel Philox masks of (seed, pair), exported by the library and shaped for the oracle."""
    k = api.philox_keep_masks(seed, pair).astype(np.float32) * np.float32(1.0 / 0.95)
    return tuple(torch.from_numpy(np.ascontiguousarray(a)) for a in
                 (k[0, :, :5120], k[0, :, 5120:], k[1, :, :5120], k[1, :, 5120:]))


def check_pairs(m, c, om, oc, what):
    """Per-pair, per-element bf16 budget; returns (max px error, max relative covariance error) for the log."""
    px = np.abs(m - om).max(axis=1)
    assert px.max() < BF16_PX, (what, "offset", float(px.max()), int(px.argmax()))
    worst = 0.0
    off_block = np.ones((8, 8), bool)
    for i in range(4):
        s = slice(2 * i, 2 * i + 2)
        off_block[s, s] = False
        d = np.sqrt(np.abs(oc[:, 2 * i, 2 * i] * oc[:, 2 * i + 1, 2 * i + 1]))          # block scale for the off-diagonal
        scale = np.stack([np.stack([np.abs(oc[:, 2 * i, 2 * i]), d], 1), np.stack([d, np.abs(oc[:, 2 * i + 1, 2 * i + 1])], 1)], 1)
        rel = np.abs(c[:, s, s] - oc[:, s, s]) / scale
        worst = max(worst, float(rel.max()))
        assert rel.max() <= BF16_COV_REL, (what, "cov block", i, float(rel.max()), int(rel.reshape(len(m), -1).max(1).argmax()))
    assert np.all(c[:, off_block] == 0) and np.all(oc[:, off_block] == 0)
    return float(px.max()), worst


def test_bf16_256_pairs_one_call_vs_oracle(api, wfile, synth_sd):
    """BASELINE config 3: 3-block UAHN, 256 pairs in ONE infer_batch, bf16, Philox masks replayed through the oracle."""
    n, seed, first = 256, 4242, 1000
    prev, curr, _, prior = S.synthetic_batch(n, start=2000)
    with api.Uahn(wfile, "prior3", precision="bf16", max_batch=n) as net:
        m, c, _ = net.infer_batch(prev, curr, prior, seed=seed, first_pair=first)
        # the fused block fronts at this batch, against torch on the kernel's own inputs (pairs 0, 100, 255)
        for blk, pre, l0, l1, s1 in ((3, O.P1, "block_3_0", "block_3_1", (32, 56, 80)), (4, O.P4, "block_4_0", "block_4_1", (16, 112, 160))):
            x = net.debug_read(f"x{blk}", (n, 2, 224 >> (4 - blk), 320 >> (4 - blk)))
            a = net.debug_read(f"act:{l1}", (n,) + s1)
            for i in (0, 100, 255):
                xi = torch.from_numpy(x[i:i + 1]).double()
                w0, b0 = synth_sd[pre + l0 + ".0.weight"], synth_sd[pre + l0 + ".0.bias"]
                w1, b1 = synth_sd[pre + l1 + ".0.weight"], synth_sd[pre + l1 + ".0.bias"]
                bf = lambda t: t.to(torch.bfloat16).double()
                h0 = torch.nn.functional.leaky_relu(torch.nn.functional.conv2d(xi, bf(w0), b0.double(), padding=3), 0.1)
                h0 = bf(h0.float())                                     # the on-chip intermediate is bf16
                ref = torch.nn.functional.leaky_relu(torch.nn.functional.conv2d(h0, bf(w1), b1.double(), stride=2, padding=2), 0.1)[0].numpy()
                scale = max(1.0, float(np.abs(ref).max()))
                # bf16 output rounding (2^-9) + rounding flips of the bf16 intermediate
                assert np.abs(a[i] - ref).max() < 8e-3 * scale, (l1, i, float(np.abs(a[i] - ref).max()), scale)
    masks = [philox_masks_for_oracle(api, seed, first + i) for i in range(n)]
    om, oc, _ = O.forward_batch(prev, curr, synth_sd, masks, prior, False)
    px, rel = check_pairs(m, c, om, oc, "256 pairs")
    print(f"\n[parity] bf16 prior3 256 pairs vs oracle: max |offset| err {px:.4f} px, max cov rel err {rel:.4f}")


def test_bf16_1024_pair_call_sampled_vs_oracle(api, wfile, synth_sd):
    """The exact kernels of the BENCH line (1024 pairs per call): 64 pairs sampled across the batch vs the oracle."""
    n, seed, first = 1024, 99, 5000
    uniq = 128
    prev, curr, _, prior = S.synthetic_batch(uniq, start=3000)
    idx = np.arange(n) % uniq
    with api.Uahn(wfile, "prior3", precision="bf16", max_batch=n) as net:
        m, c, _ = net.infer_batch(prev[idx], curr[idx], prior[idx], seed=seed, first_pair=first)
    sample = np.unique(np.concatenate([np.arange(0, n, 17), [n - 1, n - 2, 511, 512]]))[:64]
    masks = [philox_masks_for_oracle(api, seed, first + int(i)) for i in sample]
    om, oc, _ = O.forward_batch(prev[idx[sample]], curr[idx[sample]], synth_sd, masks, prior[idx[sample]], False)
    px, rel = check_pairs(m[sample], c[sample], om, oc, "1024-pair call")
    print(f"\n[parity] bf16 prior3 1024-pair call, 64 sampled pairs vs oracle: max |offset| err {px:.4f} px, max cov rel err {rel:.4f}")
    # pairs that repeat the same images but draw different masks: means close, not identical (MC dropout is live)
    assert not np.array_equal(m[0], m[uniq]) and np.abs(m[0] - m[uniq]).max() < 0.5


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_full_cascade_show_error_72_pairs_vs_oracle(api, wfile, synth_sd, precision):
    """`full` + show_error above the 64-pair switch to the fused MC GEMM (bf16) — both precisions, vs the oracle."""
    n, seed, first = 72, 31, 200
    prev, curr, _, _ = S.synthetic_batch(n, start=4000, max_disp=6.0)      # no prior: block 1 has to find it
    with api.Uahn(wfile, "full", show_error=True, precision=precision, max_batch=n) as net:
        m, c, e = net.infer_batch(prev, curr, None, seed=seed, first_pair=first, want_error=True)
    masks = [philox_masks_for_oracle(api, seed, first + i) for i in range(n)]
    om, oc, oe = O.forward_batch(prev, curr, synth_sd, masks, None, True)
    if precision == "bf16":
        px, rel = check_pairs(m, c, om, oc, "full 72 pairs")
        assert np.abs(e - oe).mean() < 0.25                  # grey levels of 255; follows the <= 0.05 px homography difference
    else:
        px = float(np.abs(m - om).max())
        rel = float((np.abs(c - oc).max(axis=(1, 2)) / np.abs(oc).max(axis=(1, 2))).max())
        assert px < 1e-3 and rel < 5e-4, (px, rel)
        assert np.abs(e - oe).max() < 0.25 and np.abs(e - oe).mean() < 1e-3
    print(f"\n[parity] {precision} full+showError 72 pairs vs oracle: max |offset| err {px:.5f} px, max cov rel err {rel:.5f}")


# every conv layer that runs as its own kernel in the bf16 product path (the four block-front layers run fused and are
# checked at 256 pairs above), by name, at a batch where the CTA-pair kernels are selected (>= 1 tile per SM)
BIG_BATCH_LAYERS = [  # name, Cin, Hin, Win, Cout, k, stride   (model_to_trace.py:93-113, 210-216)
    ("block_1_1", 2, 28, 40, 128, 7, 2), ("block_1_2", 128, 14, 20, 128, 5, 2), ("block_1_3", 128, 7, 10, 256, 3, 2),
    ("block_2_1", 2, 56, 80, 64, 7, 2), ("block_2_2", 64, 28, 40, 128, 5, 2), ("block_2_3", 128, 14, 20, 256, 3, 2),
    ("block_2_4", 256, 7, 10, 256, 3, 2),
    ("block_3_2", 32, 56, 80, 64, 3, 2), ("block_3_3", 64, 28, 40, 128, 3, 2), ("block_3_4", 128, 14, 20, 256, 3, 2),
    ("block_3_5", 256, 7, 10, 256, 3, 2),
    ("block_4_2", 16, 112, 160, 32, 3, 2), ("block_4_3", 32, 56, 80, 64, 3, 2), ("block_4_4", 64, 28, 40, 128, 3, 2),
    ("block_4_5", 128, 14, 20, 256, 3, 2), ("block_4_6", 256, 7, 10, 256, 3, 2),
]


def test_conv_layers_by_name_at_large_batch_vs_torch_fp64(api, wfile, synth_sd):
    nmax = 1100   # 1100 x 20 / 128 = 172 M tiles in the last layers: >= 148, odd unit count at the end
    g = torch.Generator().manual_seed(9)
    worst = {}
    with api.Uahn(wfile, "full", precision="bf16", max_batch=nmax) as net:
        for name, cin, hin, win, cout, k, s in BIG_BATCH_LAYERS:
            n = nmax if hin <= 28 else 301      # the large-image layers have thousands of tiles at any batch
            x = (torch.rand(n, cin, hin, win, generator=g) * 2 - 0.5).to(torch.bfloat16).float()
            pre = O.P4 if name.startswith("block_4") else O.P1
            w, b = synth_sd[pre + name + ".0.weight"].to(torch.bfloat16).float(), synth_sd[pre + name + ".0.bias"]
            ho, wo = (hin + 2 * ((k - 1) // 2) - k) // s + 1, (win + 2 * ((k - 1) // 2) - k) // s + 1
            out = net.stage_conv(name, x.numpy(), (cout, ho, wo))
            # fp64 torch on a spread of images (first, last, the odd tail, the middle): the whole batch would take minutes
            sel = [0, 1, n // 2, n - 2, n - 1] if hin > 14 else list(range(0, n, 7)) + [n - 1]
            ref = torch.nn.functional.leaky_relu(
                torch.nn.functional.conv2d(x[sel].double(), w.double(), b.double(), stride=s, padding=(k - 1) // 2), 0.1).float().numpy()
            scale = max(1.0, float(np.abs(ref).max()))
            err = float(np.abs(out[sel] - ref).max())
            worst[name] = err / scale
            assert err < 6e-3 * scale, (name, err, scale)            # bf16 output rounding 2^-9
            assert np.isfinite(out).all()
    print("\n[parity] conv layers at n=1100/301 vs torch fp64, max err / scale:", {k: round(v, 5) for k, v in worst.items()})


def test_stage_transfer_matches_reference_fixture(api, wfile, golden_stages):
    """transfer_mean_var_single alone (model_to_trace.py:18-38) against the vectors the reference itself produced."""
    g = golden_stages
    with api.Uahn(wfile, "prior1", max_batch=8) as net:
        flow, cov = net.stage_transfer(g["tr_var"], g["tr_H"], g["tr_pts"])
        p2 = g["tr_p2"][0]                                             # [3, 4] projected, perspective-normalised points
        ref_flow = (p2[:2].T - S.ORIGIN_4PT).reshape(8)
        assert np.abs(flow[0] - ref_flow).max() < 2e-4                 # fp32, coordinates up to 320
        for i in range(4):
            blk = cov[0, 2 * i:2 * i + 2, 2 * i:2 * i + 2]
            ref = g["tr_cov"][0, i]
            assert np.abs(blk - ref).max() <= 2e-6 * np.abs(ref).max(), (i, blk, ref)
        mask = np.kron(np.eye(4), np.ones((2, 2))) == 0
        assert np.all(cov[0][mask] == 0)
        # H = I: the covariance is diag(var) and the flow is the offset itself (SURVEY §8c analytic KAT)
        var = np.array([[0.5, 1.5, 2.0, 0.25, 1.0, 1.0, 3.0, 0.75]], np.float32)
        mu = np.array([[1.0, -2.0, 0.5, 0.25, -3.0, 4.0, 0.0, 0.0]], np.float32)
        flow, cov = net.stage_transfer(var, np.eye(3, dtype=np.float32)[None], S.ORIGIN_4PT.reshape(1, 8) + mu)
        assert np.array_equal(flow, mu) and np.array_equal(cov[0], np.diag(var[0]))


def test_corrupt_weight_files_are_reported_not_fatal(api, wfile, tmp_path):
    """ADVICE r01: a truncated or corrupt file must come back as an error code, not as an exception across the C ABI."""
    raw = open(wfile, "rb").read()
    cases = {"truncated": raw[: len(raw) // 2], "huge_dim": raw[:12] + raw[12:].replace(b"\x80\x00\x00\x00", b"\xff\xff\xff\x7f", 1),
             "bad_magic": b"NOTUAHN1" + raw[8:], "count": raw[:8] + b"\xff\xff\xff\xff" + raw[12:]}
    for name, data in cases.items():
        p = tmp_path / f"{name}.bin"
        p.write_bytes(data)
        with pytest.raises(api.UahnError) as ei:
            api.Uahn(str(p), "prior3", precision="fp32", max_batch=1)
        assert "(-3)" in str(ei.value), (name, str(ei.value))          # UAHN_ERR_WEIGHTS
    with api.Uahn(wfile, "prior3", precision="fp32", max_batch=1):      # the process is still healthy
        pass


def test_device_entry_rejects_error_map_without_show_error(api, wfile):
    t = torch.zeros(224 * 320, dtype=torch.uint8, device="cuda")
    o = torch.zeros(224 * 320, dtype=torch.float32, device="cuda")
    with api.Uahn(wfile, "prior3", show_error=False, precision="bf16", max_batch=1) as net:
        with pytest.raises(api.UahnError):
            net.infer_batch_ptrs(1, t.data_ptr(), t.data_ptr(), o.data_ptr(), o.data_ptr(), o.data_ptr(), err=o.data_ptr())


def test_torchscript_export_reproduces_reference_fixtures(api, tmp_path, golden_e2e, synth_sd):
    """Row f4: a user holding only the reference-style `.pt` (HomographyNet.cpp:89) converts it and gets the reference's
    own outputs; the handle takes the variant from the file (UAHN_VARIANT_AUTO)."""
    from conftest import unpack_masks
    from cuahn_vio_b200 import weights
    pt = str(tmp_path / "traced_model_3_blocks_using_prior.pt")
    O.trace(synth_sd, "prior3").save(pt)
    path = str(tmp_path / "traced_model_3_blocks_using_prior.bin")
    weights.export_torchscript(pt, path)
    g = golden_e2e
    masks = np.stack([api.pack_keep_masks(unpack_masks(g, i)) for i in range(3)])
    with api.Uahn(path, "auto", show_error=None, precision="fp32", max_batch=3) as net:
        assert net.variant == "prior3" and net.show_error is False
        m, c, _ = net.infer_batch(g["prev"], g["curr"], g["prior"], keep_masks=masks)
        for i in range(3):
            assert np.abs(m[i] - g[f"flow_prior3_{i}"]).max() < 1e-3
            assert np.abs(c[i] - g[f"cov_prior3_{i}"]).max() < 2e-4 * np.abs(g[f"cov_prior3_{i}"]).max()
    with pytest.raises(api.UahnError):                                  # a bare state_dict export has no variant record
        api.Uahn(weights.synthetic_weights_file(0), "auto", precision="fp32", max_batch=1)


def test_fresh_masks_on_every_default_call(api, wfile):
    """ADVICE r01: with no rng the forward must draw new MC-dropout masks on every call (model_to_trace.py:266-273)."""
    prev, curr, _, prior = S.synthetic_batch(1, start=60)
    with api.Uahn(wfile, "prior3", precision="fp32", max_batch=1) as net:
        net.load_image(prev[0], 0.0)
        net.load_image(curr[0], 0.1)
        a = [net.infer(prior[0].reshape(8))[0] for _ in range(4)]       # eager x2, then graph replays
        assert all(not np.array_equal(a[0], x) for x in a[1:]) and not np.array_equal(a[2], a[3])
        b = [net.infer(prior[0].reshape(8), seed=3, pair_index=7)[0] for _ in range(2)]
        assert np.array_equal(b[0], b[1])                               # an explicit key replays


def test_handles_on_two_devices_in_one_process(api, wfile):
    """ADVICE r01 (medium): shared-memory opt-ins and SM counts are cached per device."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    prev, curr, _, prior = S.synthetic_batch(3, start=70)
    outs = []
    for dev in (1, 0):                                                  # the second device first
        for precision in ("bf16", "fp32"):
            with api.Uahn(wfile, "prior3", show_error=True, precision=precision, device=dev, max_batch=3) as net:
                outs.append((precision, net.infer_batch(prev, curr, prior, seed=1, want_error=True)))
    for (p0, a), (p1, b) in zip(outs[:2], outs[2:]):
        assert p0 == p1 and all(np.array_equal(x, y) for x, y in zip(a, b))


def test_fast_coordinate_path_indices_bit_exact_over_18M_coordinates(api, wfile, golden_stages):
    """The bf16 product path's warp (CM_FAST: 3 FMAs + MUFU.RCP coordinates, exact chain only near integer boundaries)
    against the reference's index arithmetic over 256 random homographies in the benchmark's displacement range."""
    g = golden_stages
    rng = np.random.default_rng(2024)
    n = 256
    Hs = np.stack([S.dlt_numpy(S.ORIGIN_4PT.astype(np.float64), S.ORIGIN_4PT + (rng.random((4, 2)) * 2 - 1) * 20).astype(np.float32)
                   for _ in range(n)])
    img = np.repeat(g["warp_src_u8"][None], n, 0)
    with api.Uahn(wfile, "prior1", precision="bf16", max_batch=n) as net:
        _, ix, iy = net.stage_warp(img, Hs)
    mism = checked = 0
    for t in range(n):
        rix, riy, _, _ = O.sample_indices(torch.from_numpy(Hs[t]))
        rix, riy = rix.numpy(), riy.numpy()
        inside = (rix >= -1) & (rix <= 320) & (riy >= -1) & (riy <= 224)
        mism += int((ix[t][inside] != rix[inside]).sum() + (iy[t][inside] != riy[inside]).sum())
        checked += 2 * int(inside.sum())
    assert mism == 0 and checked > 30_000_000, (mism, checked)


def test_every_kernel_selection_boundary_vs_oracle(api, wfile, synth_sd):
    """Kernel selection switches with the batch size (latency-path kernels <= 8 pairs, expand-path MC head 9..63, fused MC
    GEMM from 64, CTA-pair MC GEMM from 256, CTA-pair deep layers once a layer has a tile per SM): first, middle and last
    pair of a call on both sides of every switch, bf16 vs the oracle."""
    sizes = (1, 2, 8, 9, 63, 64, 65, 255, 256, 257, 1023)
    uniq = 24
    prev, curr, _, prior = S.synthetic_batch(uniq, start=5000)
    oracle_cache = {}
    worst_px = worst_cov = 0.0
    with api.Uahn(wfile, "prior3", precision="bf16", max_batch=max(sizes)) as net:
        for n in sizes:
            idx = np.arange(n) % uniq
            seed, first = 600 + n, 10 * n
            m, c, _ = net.infer_batch(prev[idx], curr[idx], prior[idx], seed=seed, first_pair=first)
            assert np.isfinite(m).all() and np.isfinite(c).all(), n
            pick = sorted({0, n // 2, n - 1})
            masks = [philox_masks_for_oracle(api, seed, first + i) for i in pick]
            sel = idx[pick]
            om, oc, _ = O.forward_batch(prev[sel], curr[sel], synth_sd, masks, prior[sel], False)
            px, rel = check_pairs(m[pick], c[pick], om, oc, f"n={n}")
            worst_px, worst_cov = max(worst_px, px), max(worst_cov, rel)
    print(f"\n[parity] bf16 prior3 at batch sizes {sizes}: max |offset| err {worst_px:.4f} px, max cov rel err {worst_cov:.4f}")
