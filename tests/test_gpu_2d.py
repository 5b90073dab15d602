"""GPU parity, 2-D path: libhipr_b200 (through the C ABI) against the oracle on seeded inputs.
Gates (SURVEY.md 8d): literal gather bit-exact; score maps rtol 1e-5."""
import hashlib
import os

import numpy as np
import pytest

from conftest import smooth_image

pytestmark = pytest.mark.gpu
GOLD = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_vectors.npz"))

RTOL = 1e-5          # north_star: similarity maps within 1e-5 relative
ATOL_F32 = 2e-6      # float32 storage of a [0,1] score; float64 runs use ATOL_F64
ATOL_F64 = 1e-12


def _cuda(torch, a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.mark.parametrize("shape", [(11, 11), (12, 40), (37, 53), (64, 64), (75, 130)])
@pytest.mark.parametrize("params", [(11, 9), (7, 5), (5, 3), (15, 12)])
def test_line_profile_2d_bit_exact_f64(torch_cuda, oracle, shape, params):
    import neighbor2d
    P, R = params
    rng = np.random.default_rng(1)
    a = rng.random((shape[0] + P - 1, shape[1] + P - 1))
    got = neighbor2d.line_profile_2d_v2(a, P, R)
    want = oracle.line_profile_2d_v2(a, P, R)
    assert got.dtype == np.float64 and got.shape == want.shape
    assert np.array_equal(got, want)


def test_line_profile_2d_vs_compiled_reference(torch_cuda):
    """Against the output of the unmodified reference stencil, stored in tests/golden/reference_vectors.npz."""
    import neighbor2d
    img = GOLD["img2d"]
    lp = neighbor2d.line_profile_2d_v2(np.pad(img / img.max(), 5, mode="edge"), 11, 9)
    assert np.array_equal(lp[:3, :4], GOLD["lp2d_corner"])
    assert hashlib.sha256(lp.tobytes()).digest() == GOLD["lp2d_sha256"].tobytes()


def test_line_profile_2d_f32_device(torch_cuda, oracle):
    import hipr_b200
    a = np.random.default_rng(3).random((70, 91)).astype(np.float32)
    got = hipr_b200.line_profile_2d(_cuda(torch_cuda, a), 11, 9).cpu().numpy()
    want = oracle.line_profile_2d_v2(a.astype(np.float64), 11, 9).astype(np.float32)
    assert np.array_equal(got, want)


def test_line_profile_2d_host_bands_pinned_and_pageable(torch_cuda, oracle):
    """hipr_line_profile_2d_host: several row bands (32 MiB of output each), pageable output through the staging ring,
    page-locked output directly, a caller's `out`; all bit-identical to the oracle and to the device operator."""
    import hipr_b200
    a = np.random.default_rng(11).random((330, 610))
    want = oracle.line_profile_2d_v2(a, 11, 9)                       # (320, 600, 9, 11): 152 MB = 5 bands
    got = hipr_b200.line_profile_2d_host(a, 11, 9)
    assert got.dtype == np.float64 and np.array_equal(got, want)
    pinned = hipr_b200.line_profile_2d_host(a, 11, 9, pinned=True)
    assert np.array_equal(pinned, want)
    out = np.full(want.shape, -1.0)
    assert hipr_b200.line_profile_2d_host(a, 11, 9, out=out) is out and np.array_equal(out, want)
    dev = hipr_b200.line_profile_2d(_cuda(torch_cuda, a), 11, 9).cpu().numpy()
    assert np.array_equal(dev, want)
    with pytest.raises(ValueError):
        hipr_b200.line_profile_2d_host(a, 11, 9, out=np.empty((3, 3)))
    with pytest.raises(TypeError):
        hipr_b200.line_profile_2d_host(a.astype(np.float32), 11, 9)


def test_line_profile_2d_noncontiguous_and_special_values(torch_cuda, oracle):
    import neighbor2d
    a = np.random.default_rng(4).random((60, 90))[::2, ::3]          # strided view, as a memoryview accepts
    a = a.copy(); a[3, 4] = np.nan; a[7, 7] = np.inf; a[9, 1] = -0.0
    view = np.asfortranarray(a)
    got = neighbor2d.line_profile_2d_v2(view, 11, 9)
    want = oracle.line_profile_2d_v2(np.ascontiguousarray(a), 11, 9)
    assert np.array_equal(got, want, equal_nan=True)
    assert np.array_equal(np.signbit(got), np.signbit(want))


@pytest.mark.parametrize("flavour", ["F1", "F2", "F3"])
@pytest.mark.parametrize("shape", [(1, 1), (5, 7), (32, 32), (33, 65), (97, 130)])
def test_lne2d_f64(torch_cuda, oracle, flavour, shape):
    import hipr_b200
    img = smooth_image(shape, 5).astype(np.float64)
    got = hipr_b200.lne2d(_cuda(torch_cuda, img), flavour).cpu().numpy()
    want = oracle.lne2d(img, flavour)
    np.testing.assert_allclose(got, want, rtol=RTOL, atol=ATOL_F64, equal_nan=True)


@pytest.mark.parametrize("flavour", ["F1", "F2", "F3"])
def test_lne2d_f32(torch_cuda, oracle, flavour):
    import hipr_b200
    img = smooth_image((150, 201), 6)
    got = hipr_b200.lne2d(_cuda(torch_cuda, img), flavour).cpu().numpy()
    want = oracle.lne2d(img.astype(np.float64), flavour)
    assert got.dtype == np.float32
    np.testing.assert_allclose(got, want, rtol=RTOL, atol=ATOL_F32)


def test_lne2d_padded_equals_unpadded(torch_cuda):
    import hipr_b200
    img = smooth_image((80, 90), 7)
    a = hipr_b200.lne2d(_cuda(torch_cuda, img), "F1").cpu().numpy()
    b = hipr_b200.lne2d(_cuda(torch_cuda, np.pad(img, 5, mode="edge")), "F1", padded=True).cpu().numpy()
    assert np.array_equal(a, b)


@pytest.mark.parametrize("params", [(7, 5), (5, 3), (15, 12), (11, 4), (9, 16)])
@pytest.mark.parametrize("flavour", ["F1", "F2", "F3"])
def test_lne2d_generic_parameters(torch_cuda, oracle, params, flavour):
    import hipr_b200
    P, R = params
    img = smooth_image((41, 57), 8).astype(np.float64)
    got = hipr_b200.lne2d(_cuda(torch_cuda, img), flavour, P, R).cpu().numpy()
    want = oracle.lne2d(img, flavour, P, R)
    np.testing.assert_allclose(got, want, rtol=RTOL, atol=ATOL_F64, equal_nan=True)


@pytest.mark.parametrize("flavour", ["F1", "F2", "F3"])
def test_lne2d_flat_and_nan_inputs(torch_cuda, oracle, flavour):
    """Degenerate lines: flat regions give 0/0 = NaN in F1/F2 and are clamped by 1e-8 in F3;
    NaN samples are zeroed by nan_to_num in F1/F2 and propagate in F3."""
    import hipr_b200
    img = smooth_image((48, 48), 9).astype(np.float64)
    img[10:30, 10:30] = 0.25          # flat block
    img[40, 5] = np.nan
    got = hipr_b200.lne2d(_cuda(torch_cuda, img), flavour).cpu().numpy()
    want = oracle.lne2d(img, flavour)
    assert np.array_equal(np.isnan(got), np.isnan(want))
    np.testing.assert_allclose(got, want, rtol=RTOL, atol=ATOL_F64, equal_nan=True)


def test_lne2d_scale_invariance(torch_cuda):
    """F1 is invariant to a power-of-two rescale of the image (exact in floating point)."""
    import hipr_b200
    img = smooth_image((64, 64), 10)
    a = hipr_b200.lne2d(_cuda(torch_cuda, img), "F1").cpu().numpy()
    b = hipr_b200.lne2d(_cuda(torch_cuda, img * 8.0), "F1").cpu().numpy()
    assert np.array_equal(a, b)


@pytest.mark.parametrize("shape", [(40, 36, 95), (67, 129, 95), (33, 31, 63), (16, 16, 8), (9, 5, 130)])
def test_channel_sum(torch_cuda, shape):
    import hipr_b200
    cube = (np.random.default_rng(11).random(shape) * 0.5).astype(np.float32)
    want = cube.astype(np.float64).sum(axis=2)
    for dt, tol in ((torch_cuda.float64, 1e-14), (torch_cuda.float32, 6e-8)):
        got = hipr_b200.channel_sum(_cuda(torch_cuda, cube), normalize=False, dtype=dt).cpu().numpy()
        np.testing.assert_allclose(got, want, rtol=tol, atol=0)
        gotn = hipr_b200.channel_sum(_cuda(torch_cuda, cube), normalize=True, dtype=dt).cpu().numpy()
        np.testing.assert_allclose(gotn, want / want.max(), rtol=2 * tol + 1e-15, atol=0)
        assert gotn.max() == 1.0


def test_channel_sum_calibration(torch_cuda):
    import hipr_b200
    rng = np.random.default_rng(12)
    cube = rng.random((30, 41, 95)).astype(np.float32)
    cal = (0.5 + rng.random((30, 41, 95))).astype(np.float32)
    got = hipr_b200.channel_sum(_cuda(torch_cuda, cube), _cuda(torch_cuda, cal), normalize=False,
                                dtype=torch_cuda.float64).cpu().numpy()
    want = (cube.astype(np.float64) / cal.astype(np.float64)).sum(axis=2)
    np.testing.assert_allclose(got, want, rtol=1e-14)


ATOL_FUSED = 5e-7   # fused kernel: same arithmetic as the fixed-point stencil, window-local quantisation
ATOL_FIXED = 5e-7   # fixed-point stencil: float32 arithmetic on exact differences, float32 score in [0, 1] (4 ulp at 1.0)
ATOL_F32_SUM = 1e-5  # float32 SUM IMAGE: its 6e-8 rounding is amplified by value/line-range (DESIGN.md)


@pytest.mark.parametrize("flavour", ["F1", "F2", "F3"])
@pytest.mark.parametrize("mode", ["fixed", "float32", "float64"])
def test_neighbor2d_score_pipeline(torch_cuda, oracle, flavour, mode):
    """The whole 2-D path on a synthetic FOV: cube -> sum -> /max -> pad -> stencil -> epilogue.
    Default mode = float64 sums + fixed-point stencil: meets rtol 1e-5 with atol 2e-7."""
    import hipr_b200
    from hipr_b200 import synth
    cube, _, _ = synth.make_fov(96, 160, 95, fov_index=3)
    cube_np = cube.numpy()
    dt = {"fixed": None, "float32": torch_cuda.float32, "float64": torch_cuda.float64}[mode]
    got = hipr_b200.neighbor2d_score(cube.cuda(), flavour, dtype=dt).cpu().numpy()
    want = oracle.neighbor2d_score(cube_np, flavour)
    atol = {"fixed": ATOL_FIXED, "float32": ATOL_F32_SUM, "float64": ATOL_F64}[mode]
    np.testing.assert_allclose(got, want, rtol=RTOL, atol=atol)


@pytest.mark.parametrize("flavour", ["F1", "F2", "F3"])
@pytest.mark.parametrize("shape", [(1, 1), (7, 3), (32, 32), (45, 77), (130, 97)])
def test_lne2d_fixed_point(torch_cuda, oracle, flavour, shape):
    """Fixed-point stencil on a float64 image against the float64 oracle of image / max."""
    import hipr_b200
    img = smooth_image(shape, 21).astype(np.float64) + 0.1
    got = hipr_b200.lne2d_fixed(_cuda(torch_cuda, img), flavour).cpu().numpy()
    want = oracle.lne2d(img / img.max(), flavour)
    np.testing.assert_allclose(got, want, rtol=RTOL, atol=ATOL_FIXED, equal_nan=True)


def test_lne2d_fixed_point_flat_regions_and_custom_table(torch_cuda, oracle):
    import hipr_b200
    img = smooth_image((64, 64), 22).astype(np.float64) + 0.1
    img[20:45, 20:45] = 0.7
    for flavour in ("F1", "F2", "F3"):
        got = hipr_b200.lne2d_fixed(_cuda(torch_cuda, img), flavour).cpu().numpy()
        want = oracle.lne2d(img / img.max(), flavour)
        assert np.array_equal(np.isnan(got), np.isnan(want))
        np.testing.assert_allclose(got, want, rtol=RTOL, atol=ATOL_FIXED, equal_nan=True)
    flat = np.full((20, 20), 3.0)
    got = hipr_b200.lne2d_fixed(_cuda(torch_cuda, flat), "F3").cpu().numpy()
    np.testing.assert_allclose(got, oracle.lne2d(flat / 3.0, "F3"), atol=1e-12)
    assert np.isnan(hipr_b200.lne2d_fixed(_cuda(torch_cuda, flat), "F1").cpu().numpy()).all()


def test_neighbor2d_score_vs_compiled_reference(torch_cuda):
    """Against the score the reference path (compiled reference stencil) computed, stored in
    tests/golden/reference_vectors.npz."""
    import hipr_b200
    cube = torch_cuda.from_numpy(GOLD["cube"])
    want = GOLD["cube_score_F1"]
    got = hipr_b200.neighbor2d_score(cube.cuda(), "F1", dtype=torch_cuda.float64).cpu().numpy()
    np.testing.assert_allclose(got, want, rtol=RTOL, atol=ATOL_F64)
    got = hipr_b200.neighbor2d_score(cube.cuda(), "F1").cpu().numpy()
    np.testing.assert_allclose(got, want, rtol=RTOL, atol=ATOL_FIXED)


def test_neighbor2d_score_batch_and_sum(torch_cuda, oracle):
    import hipr_b200
    from hipr_b200 import synth
    cubes = torch_cuda.stack([synth.make_fov(48, 64, 95, fov_index=i)[0] for i in range(3)])
    score, s = hipr_b200.neighbor2d_score(cubes.cuda(), "F1", return_sum=True)
    assert score.shape == (3, 48, 64) and s.shape == (3, 48, 64)
    for i in range(3):
        want_s, _ = oracle.prologue(cubes[i].numpy())
        np.testing.assert_allclose(s[i].cpu().numpy(), want_s / want_s.max(), rtol=2e-7)
        np.testing.assert_allclose(score[i].cpu().numpy(), oracle.neighbor2d_score(cubes[i].numpy(), "F1"),
                                   rtol=RTOL, atol=ATOL_FIXED)


def test_host_entry_point(torch_cuda, oracle):
    """hipr_neighbor2d_host: numpy in, numpy out, copies inside, banded H2D pipeline."""
    import hipr_b200
    from hipr_b200 import synth
    cube = synth.make_fov(200, 333, 95, fov_index=8)[0].numpy()
    score, s = hipr_b200.neighbor2d_score_host(cube, "F1", return_sum=True)
    want_s, _ = oracle.prologue(cube)
    np.testing.assert_allclose(s, want_s / want_s.max(), rtol=2e-7)
    np.testing.assert_allclose(score, oracle.neighbor2d_score(cube, "F1"), rtol=RTOL, atol=ATOL_FIXED)
    pinned = hipr_b200.pinned_empty(cube.shape, np.float32)
    pinned[...] = cube
    score2 = hipr_b200.neighbor2d_score_host(pinned, "F1")
    assert np.array_equal(score, score2)


def test_rejects_cpu_tensors_and_bad_arguments(torch_cuda):
    import hipr_b200
    with pytest.raises(ValueError):
        hipr_b200.lne2d(torch_cuda.zeros(20, 20), "F1")              # CPU tensor: no CPU path
    x = torch_cuda.zeros(20, 20, device="cuda")
    with pytest.raises(ValueError):
        hipr_b200.lne2d(x, "F9")
    with pytest.raises(ValueError):
        hipr_b200.lne2d(x, "F1", 10, 9)                              # even patch
    with pytest.raises(TypeError):
        hipr_b200.lne2d(x.to(torch_cuda.float16), "F1")
    with pytest.raises(ValueError):
        hipr_b200.lne2d(torch_cuda.zeros(8, 8, device="cuda"), "F1", padded=True)   # smaller than patch


def test_mosaic_slabs_equal_unsplit_single_gpu(torch_cuda, oracle):
    """Config 5 on one GPU: row slabs + 5-row halos + the GLOBAL range give exactly the unsplit
    score (what sharding.MosaicSlab computes after its halo exchange and range all-reduce)."""
    import hipr_b200
    from hipr_b200 import ops, sharding, synth
    cube = synth.make_fov(96, 128, 95, fov_index=11)[0].cuda()
    s, mk = ops.channel_sum(cube, None, normalize=False, dtype=torch_cuda.float64, return_max=True)
    whole = ops.lne2d_fixed(s, "F1", range_keys=mk)
    vmax, vmin = mk.values()
    world = 3
    for rank in range(world):
        r0, r1 = sharding.slab_bounds(96, rank, world)
        s_slab, mk_slab = ops.channel_sum(cube[r0:r1], None, normalize=False, dtype=torch_cuda.float64, return_max=True)
        assert torch_cuda.equal(s_slab, s[r0:r1])
        lmax, lmin = mk_slab.values()
        assert float(lmax) <= float(vmax) and float(lmin) >= float(vmin)
        nt, nb = (0 if rank == 0 else 5), (0 if rank == world - 1 else 5)
        ext = s[r0 - nt: r1 + nb].contiguous()
        got = ops.lne2d_fixed(ext, "F1", range_keys=ops.MaxKey.from_values(vmax, vmin))[nt: ext.shape[0] - nb]
        assert torch_cuda.equal(got, whole[r0:r1])
    np.testing.assert_allclose(whole.cpu().numpy(), oracle.neighbor2d_score(cube.cpu().numpy(), "F1"), rtol=RTOL, atol=ATOL_FIXED)


@pytest.mark.parametrize("flavour", ["F1", "F2"])
@pytest.mark.parametrize("shape", [(8, 128), (64, 256), (96, 160), (200, 132), (37, 388), (300, 1024), (11, 4)])
def test_fused_kernel(torch_cuda, oracle, flavour, shape):
    """One-launch cube -> score (csrc/fused2d.cu) against the oracle; bands, strips, partial strips,
    partial row blocks and images smaller than a strip."""
    import hipr_b200
    from hipr_b200 import ops, synth
    cube = synth.make_fov(shape[0], shape[1], 95, fov_index=17)[0]
    got = ops.neighbor2d_fused(cube.cuda(), flavour)
    assert got is not None
    want = oracle.neighbor2d_score(cube.numpy(), flavour)
    np.testing.assert_allclose(got.cpu().numpy(), want, rtol=RTOL, atol=ATOL_FUSED)


def test_fused_kernel_sum_output_and_fallback(torch_cuda, oracle):
    import hipr_b200
    from hipr_b200 import ops, synth
    cube = synth.make_fov(130, 260, 95, fov_index=18)[0]
    score, s, mk = ops.neighbor2d_fused(cube.cuda(), "F1", return_sum=True)
    want_s, _ = oracle.prologue(cube.numpy())
    np.testing.assert_allclose(s.cpu().numpy(), want_s, rtol=1e-14)
    vmax, vmin = mk.values()
    assert float(vmax) == s.max().item() and float(vmin) == s.min().item()
    np.testing.assert_allclose(score.cpu().numpy(), oracle.neighbor2d_score(cube.numpy(), "F1"), rtol=RTOL, atol=ATOL_FUSED)
    # outside the envelope: odd width, F3, other channel counts still work through neighbor2d_score
    assert ops.neighbor2d_fused(cube[:, :259].contiguous().cuda(), "F1") is None
    assert ops.neighbor2d_fused(cube.cuda(), "F3") is None
    for c in (cube[:, :259].contiguous(), cube[:40, :64, :63].contiguous(), cube[:40, :64, :8].contiguous()):
        got = hipr_b200.neighbor2d_score(c.cuda(), "F1").cpu().numpy()
        np.testing.assert_allclose(got, oracle.neighbor2d_score(c.numpy(), "F1"), rtol=RTOL, atol=ATOL_FIXED)


def test_fused_kernel_flat_image(torch_cuda):
    from hipr_b200 import ops
    cube = torch_cuda.full((40, 128, 95), 0.25, device="cuda")
    assert torch_cuda.isnan(ops.neighbor2d_fused(cube, "F1")).all()


@pytest.mark.parametrize("C", [95, 63, 32, 130, 300])
def test_channel_sum_ring_wraps(torch_cuda, C):
    """Enough chunks per CTA that every stage of the bulk-copy ring is reused several times, for
    the stage/group geometries the channel count selects (chansum.cu: stages % groups == 0)."""
    import hipr_b200
    rng = np.random.default_rng(C)
    npix = 148 * 128 * 9 + 77          # ~9 chunks per CTA + a ragged tail
    cube = rng.random((npix, C), dtype=np.float32)
    want = cube.astype(np.float64).sum(axis=1)
    got = hipr_b200.channel_sum(_cuda(torch_cuda, cube), normalize=False, dtype=torch_cuda.float64).cpu().numpy()
    np.testing.assert_allclose(got, want, rtol=1e-14, atol=0)


def test_channel_sum_calibration_bulk_path(torch_cuda, oracle):
    """Flat-field divide fused into the bulk-copy kernel (two streams per stage), ring wrapped."""
    import hipr_b200
    rng = np.random.default_rng(77)
    shape = (420, 512, 95)
    cube = rng.random(shape, dtype=np.float32)
    cal = (0.5 + rng.random(shape, dtype=np.float32)).astype(np.float32)
    got, mk = hipr_b200.channel_sum(_cuda(torch_cuda, cube), _cuda(torch_cuda, cal), normalize=False,
                                    dtype=torch_cuda.float64, return_max=True)
    want = (cube.astype(np.float64) / cal.astype(np.float64)).sum(axis=2)
    # the quotient is a float32 reciprocal + exact float64 product + float32 correction (hipr_common.cuh,
    # sum_channels_div): within ~2e-14 of numpy's correctly rounded float64 divide
    np.testing.assert_allclose(got.cpu().numpy(), want, rtol=1e-13)
    np.testing.assert_allclose(float(mk.value()), want.max(), rtol=1e-13)
    # and through the pipeline entry point with calibration= (two-kernel path)
    small = (slice(0, 64), slice(0, 96))
    score = hipr_b200.neighbor2d_score(_cuda(torch_cuda, cube[small]), "F1", calibration=_cuda(torch_cuda, cal[small]))
    want_score = oracle.neighbor2d_score(cube[small], "F1", calibration=cal[small])
    np.testing.assert_allclose(score.cpu().numpy(), want_score, rtol=RTOL, atol=ATOL_FIXED)


def _raw_cube(bits, shape=(96, 128, 95), fov=2):
    """Raw detector counts with the structure of the synthetic FOV."""
    from hipr_b200 import synth
    cube = synth.make_fov(shape[0], shape[1], shape[2], fov_index=fov)[0].numpy()
    top = (1 << bits) - 1
    u = np.clip(np.round(cube / cube.max() * top * 0.9), 0, top)
    return u.astype(np.uint16 if bits > 8 else np.uint8)


@pytest.mark.parametrize("bits,scale", [(16, 65535.0), (12, 4095.0), (8, 255.0)])
def test_channel_sum_raw_counts(torch_cuda, bits, scale):
    """Raw uint16 / uint8 counts: every sample becomes float32(count) / float32(scale) (bioformats' rescale)
    before the float64 channel sum -- the sums of the rescaled float32 cube, to the last bits."""
    import hipr_b200
    u = _raw_cube(bits, (37 * 4, 131, 95))                       # 19,388 px: bulk chunks + a ragged tail
    f = u.astype(np.float32) / np.float32(scale)
    want = f.astype(np.float64).sum(axis=2)
    got, mk = hipr_b200.channel_sum_raw(torch_cuda.from_numpy(u).cuda(), scale, return_max=True)
    np.testing.assert_allclose(got.cpu().numpy(), want, rtol=1e-15, atol=0)
    same, _ = hipr_b200.channel_sum(torch_cuda.from_numpy(f).cuda(), normalize=False, dtype=torch_cuda.float64, return_max=True)
    assert torch_cuda.equal(got, same)                           # bit-identical to the float32 path
    assert float(mk.value()) == got.max().item()


def test_neighbor2d_host_raw_counts(torch_cuda, oracle):
    """hipr_neighbor2d_host_raw on uint16 counts == the oracle on the rescaled float32 cube."""
    import hipr_b200
    u = _raw_cube(16)
    f = u.astype(np.float32) / np.float32(65535.0)
    want = oracle.neighbor2d_score(f, "F1")
    got = hipr_b200.neighbor2d_score_host_raw(u, 65535.0, "F1")
    np.testing.assert_allclose(got, want, rtol=RTOL, atol=ATOL_FIXED)
    assert np.array_equal(got, hipr_b200.neighbor2d_score_host(f, "F1"))      # same sums -> same score, bit for bit
    with pytest.raises(TypeError):
        hipr_b200.neighbor2d_score_host_raw(f, 65535.0)
    with pytest.raises(ValueError):
        hipr_b200.neighbor2d_score_host_raw(u, 0.0)


def test_host_entry_point_pageable_equals_pinned(torch_cuda):
    """A numpy array (pageable: copied through the page-locked staging ring by host threads) and a page-locked
    array (direct DMA) give the same score, bit for bit; several bands, so the ring wraps."""
    import hipr_b200
    from hipr_b200 import ops, synth
    cube = synth.make_fov(1000, 1024, 95, fov_index=4)[0].numpy()          # 389 MB: 12 bands of 32 MiB
    pinned = ops.pinned_empty(cube.shape, np.float32)
    pinned[...] = cube
    a = hipr_b200.neighbor2d_score_host(cube, "F1")
    b = hipr_b200.neighbor2d_score_host(pinned, "F1")
    assert np.array_equal(a, b)
    dev = hipr_b200.neighbor2d_score(torch_cuda.from_numpy(cube).cuda(), "F1").cpu().numpy()
    assert np.array_equal(a, dev)                                          # and the same as the device-resident call


@pytest.mark.parametrize("flavour", ["F1", "F2", "F3"])
def test_score_strict_relative_parity(torch_cuda, oracle, flavour):
    """north_star's gate as written: 1e-5 RELATIVE, no absolute term, over a whole 512^2 FOV.  The fixed-point
    stencil alone cannot give it (a pixel that is almost the minimum of its lines keeps the grid's absolute error);
    the pixels it marks as ill-conditioned are recomputed in float64 (lne2d_refine_kernel)."""
    import hipr_b200
    from hipr_b200 import synth
    cube, _, _ = synth.make_fov(512, 512, 95, fov_index=5)
    want = oracle.neighbor2d_score(cube.numpy(), flavour)
    for got in (hipr_b200.neighbor2d_score(cube.cuda(), flavour).cpu().numpy(),
                hipr_b200.neighbor2d_score_host(cube.numpy(), flavour)):
        assert (got >= 0).all(), "a refinement sentinel survived"
        np.testing.assert_allclose(got, want, rtol=1e-5, atol=0)
        assert np.array_equal(got == 0, want == 0)


def test_fov_handle_one_upload_for_score_and_spectra(torch_cuda, oracle):
    """hipr_fov_*: the cube is uploaded once; score and per-cell spectra equal the two host entry points bit for bit
    and the oracle within the gates; int64 labels, more cells than the first capacity guess, release."""
    import hipr_b200
    from hipr_b200 import synth
    cube, labels, _ = synth.make_fov(200, 176, 95, fov_index=8, drop_fraction=0.1)
    cube_np, lab_np = cube.numpy(), labels.numpy()
    with hipr_b200.Fov(cube_np) as fov:
        for fl in ("F1", "F2", "F3"):
            got = fov.score(fl)
            assert np.array_equal(got, hipr_b200.neighbor2d_score_host(cube_np, fl))
            np.testing.assert_allclose(got, oracle.neighbor2d_score(cube_np, fl), rtol=1e-5, atol=0)
        score, s = fov.score("F1", return_sum=True)
        want_s = cube_np.astype(np.float64).sum(axis=2)
        np.testing.assert_allclose(s, want_s / want_s.max(), rtol=1e-6)
        for lab_in in (lab_np, lab_np.astype(np.int64)):
            l1, a1, v1, n1 = fov.cell_spectra(lab_in)
            l2, a2, v2, n2 = hipr_b200.cell_spectra_host(cube_np, lab_in)
            assert np.array_equal(l1, l2) and np.array_equal(a1, a2)
            np.testing.assert_allclose(v1, v2, rtol=1e-12)
            wl, wa, wavg, wnorm = oracle.cell_spectra(lab_in, cube_np)
            assert np.array_equal(l1, wl) and np.array_equal(a1, wa)
            np.testing.assert_allclose(v1, wavg, rtol=1e-5)
            np.testing.assert_allclose(n1, wnorm, rtol=1e-5)
        general = fov.score("F1", patch_size=7, phi_range=5)          # outside the fixed-point fast path
        np.testing.assert_allclose(general, oracle.lne2d(want_s / want_s.max(), "F1", 7, 5), rtol=1e-5, atol=1e-6)
        assert all(p for p in fov.device_arrays())
    with pytest.raises(ValueError):
        fov.score("F1")                                               # released
    many = np.arange(1, 200 * 176 + 1, dtype=np.int32).reshape(200, 176)    # 35,200 one-pixel cells > first capacity
    with hipr_b200.Fov(cube_np) as fov:
        l, a, v, _ = fov.cell_spectra(many)
        assert l.size == many.size and (a == 1).all()
        np.testing.assert_allclose(v, cube_np.reshape(-1, 95).astype(np.float64), rtol=1e-12)
    with pytest.raises(TypeError):
        hipr_b200.Fov(cube_np.astype(np.float64))
