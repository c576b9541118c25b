"""GPU parity tests (run on the B200 box): the CUDA kernels, called through the C-ABI, against
the oracle on the same seeded inputs, against the committed golden fixtures from the
reference's JAX file, and -- at BASELINE.json's full 4K size -- against the full oracle on
one frame plus size-independent properties.  Tolerance: 1e-5 relative (tests/util.py);
cell indices bit-exact."""
import os

import numpy as np
import pytest
import torch

import oracle
from hdrnet_b200 import _lib, hdrnet_ops, layers
from util import RTOL, assert_parity, load_golden, rand_case, rel_err

pytestmark = pytest.mark.gpu

VARIANTS = {"auto": _lib.VARIANT_AUTO, "generic": _lib.VARIANT_GENERIC, "tma": _lib.VARIANT_TMA,
            "tex": _lib.VARIANT_TEX, "tex_async": _lib.VARIANT_TEX_ASYNC}
ROW_KERNELS = ("tma", "tex", "tex_async")


def cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def run_apply(grid, guide, inp, has_offset, variant="auto"):
    out = hdrnet_ops.bilateral_slice_apply(cuda(grid), cuda(guide), cuda(inp), has_offset,
                                           variant=VARIANTS[variant])
    torch.cuda.synchronize()
    return out.cpu().numpy()


def run_slice(grid, guide, variant="auto"):
    out = hdrnet_ops.bilateral_slice(cuda(grid), cuda(guide), variant=VARIANTS[variant])
    torch.cuda.synchronize()
    return out.cpu().numpy()


def checker():
    """Compiled reference loops when present, else the C restatement."""
    return oracle.best()


# ---- golden fixtures from the reference's jax/bilateral_slice.py ---------------------------
@pytest.mark.parametrize("name", ["ops_test_extents", "jax_tf2_extents", "interpolate_kat_0",
                                  "interpolate_kat_1", "interpolate_kat_2", "edge_guides",
                                  "edge_gd1", "wide_rows", "signed_random"])
def test_matches_reference_jax_golden(name):
    g = load_golden(name)
    assert_parity(run_slice(g["grid"], g["guide"]), g["slice"], what=f"{name}: slice")
    gh, gw, gd = g["grid"].shape[1:4]
    idx = hdrnet_ops.slice_indices(cuda(g["guide"]), (gh, gw, gd)).cpu().numpy()
    assert np.array_equal(idx, g["indices"]), f"{name}: cell indices must be bit-exact"
    if "apply_offset" in g:
        for v in ("auto", "generic"):
            assert_parity(run_apply(g["grid"], g["guide"], g["input"], True, v), g["apply_offset"],
                          what=f"{name}: apply+offset [{v}]")
    if "apply_nooffset" in g:
        assert_parity(run_apply(g["grid"], g["guide"], g["input"], False), g["apply_nooffset"],
                      what=f"{name}: apply")


def test_wide_rows_golden_through_tma_kernel():
    g = load_golden("wide_rows")
    assert_parity(run_apply(g["grid"], g["guide"], g["input"], True, "tma"), g["apply_offset"],
                  what="wide_rows [tma]")


@pytest.mark.parametrize("val", [0, 1, 2])
def test_interpolate_known_answer(val):
    """hdrnet/test/ops_test.py:61-86, tolerance 5e-4 there."""
    g = load_golden(f"interpolate_kat_{val}")
    out = run_slice(g["grid"], g["guide"])
    assert np.abs(out - val).max() < 5e-4


# ---- seeded parity against the oracle, every variant ----------------------------------------
SHAPES = [
    # B, H, W, gh, gw, gd
    (1, 40, 3840, 16, 16, 8),   # 4K rows: the z-bucketed kernel's home shape (5 x cells / segment)
    (2, 11, 2048, 8, 8, 8),     # 2 segments, 4-5 x cells each
    (1, 6, 1920, 16, 16, 4),    # few depth buckets
    (1, 5, 4000, 16, 12, 15),   # gd + 1 = 16 depth buckets, ragged segments
    (3, 30, 25, 16, 12, 8),     # hdrnet_ops_test.py:91-100 (W % 4 != 0 -> generic only)
    (3, 8, 5, 6, 3, 7),         # hdrnet_ops_test.py:185-195
    (4, 48, 64, 16, 12, 8),     # hdrnet_ops_jax_tf2_test.py:28-34, reduced
    (2, 33, 128, 16, 16, 8),    # narrowest width AUTO sends to the TMA kernel
    (1, 5, 4, 2, 2, 2),         # a single quad per row
    (2, 7, 1028, 5, 7, 3),      # two segments per row, ragged second segment
    (1, 300, 1920, 16, 16, 8),  # 1080p rows: more rows than CTAs
    (2, 16, 4032, 32, 32, 16),  # 12 MP width, largest grid of the sweep (1 CTA / SM)
    (1, 9, 512, 1, 1, 1),       # degenerate 1x1x1 grid
]


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("variant", ["auto", "generic", "tma", "tex", "tex_async"])
def test_slice_apply_matches_oracle(shape, variant):
    B, H, W, gh, gw, gd = shape
    if variant in ROW_KERNELS and W % 4 != 0:
        pytest.skip("TMA kernels need W % 4 == 0")
    grid, guide, inp = rand_case(1234, B, H, W, gh, gw, gd, signed=True)
    expected = checker().bilateral_slice_apply(grid, guide, inp, True)
    try:
        got = run_apply(grid, guide, inp, True, variant)
    except ValueError as e:
        if variant == "tex_async" and gw * gd * 48 >= 24 * 1024 and "cannot run these shapes" in str(e):
            pytest.skip("issuer-warp kernel: two slab rows + a 3-stage ring exceed two CTAs' shared memory")
        raise
    assert_parity(got, expected, what=f"{shape} [{variant}]")


@pytest.mark.parametrize("n_in,n_out,has_offset", [(3, 3, False), (3, 4, True), (1, 1, True),
                                                   (4, 2, True), (2, 5, False), (3, 9, True)])
def test_slice_apply_general_channels(n_in, n_out, has_offset):
    """ops_test.py:345-365 (has_offset False -> gc/n_in outputs) and the GaussianPyrNN
    n_out = 9 case (models.py:221-223)."""
    grid, guide, inp = rand_case(7, 2, 21, 36, 5, 4, 6, n_in, n_out, has_offset, signed=True)
    expected = checker().bilateral_slice_apply(grid, guide, inp, has_offset)
    got = run_apply(grid, guide, inp, has_offset)
    assert got.shape == (2, 21, 36, n_out)
    assert_parity(got, expected)


@pytest.mark.parametrize("n_in,n_out,has_offset,W", [(3, 3, False, 1000), (3, 4, True, 1026), (2, 5, False, 777),
                                                      (3, 3, True, 1023), (3, 9, True, 640), (1, 1, True, 65)])
def test_any_shape_row_kernel_matches_oracle(n_in, n_out, has_offset, W):
    """What AUTO runs where the TMA kernels' contract does not hold (has_offset False, other channel
    counts, odd widths; ops_test.py:345-365, hdrnet_ops_test.py:91-100, models.py:221-223): the
    any-shape row kernel (y-pre-blended slab in shared memory, plain loads) against the oracle,
    and against the one-thread-per-pixel kernel it replaces; grid-row pairs change inside a CTA's rows."""
    grid, guide, inp = rand_case(23, 2, 157, W, 7, 9, 5, n_in, n_out, has_offset, signed=True)
    guide[0, :, ::7] = 1.6
    guide[1, :, 3::11] = -0.4
    expected = checker().bilateral_slice_apply(grid, guide, inp, has_offset)
    got = run_apply(grid, guide, inp, has_offset)
    assert_parity(got, expected, what=f"any-shape rows {n_in}->{n_out} offset={has_offset} W={W}")
    assert_parity(got, run_apply(grid, guide, inp, has_offset, "generic"), rtol=2e-6, what="vs per-pixel kernel")
    sl = run_slice(grid, guide)                                             # un-fused slice, gc = n_out * J
    assert_parity(sl, checker().bilateral_slice(grid, guide), what="any-shape slice")


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("variant", ["auto", "generic", "tma"])
def test_slice_matches_oracle(shape, variant):
    B, H, W, gh, gw, gd = shape
    if variant == "tma" and W % 4 != 0:
        pytest.skip("TMA kernel needs W % 4 == 0")
    rng = np.random.RandomState(3)
    grid = rng.randn(B, gh, gw, gd, 12).astype(np.float32)
    guide = rng.rand(B, H, W).astype(np.float32)
    assert_parity(run_slice(grid, guide, variant), checker().bilateral_slice(grid, guide),
                  what=f"{shape} [{variant}]")


def test_slice_other_channel_counts_use_generic_kernel():
    """hdrnet_ops_jax_tf2_test.py:28-34 uses gc = 2; the TMA kernel is specialised for gc = 12."""
    rng = np.random.RandomState(4)
    grid = rng.randn(2, 16, 12, 8, 2).astype(np.float32)
    guide = rng.rand(2, 48, 640).astype(np.float32)
    assert_parity(run_slice(grid, guide), checker().bilateral_slice(grid, guide))
    with pytest.raises(ValueError):
        run_slice(grid, guide, "tma")


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_cell_indices_bit_exact(shape):
    B, H, W, gh, gw, gd = shape
    rng = np.random.RandomState(5)
    guide = rng.rand(B, H, W).astype(np.float32)
    # exercise the cell boundaries: guide * gd - 0.5 exactly integral, and just around it
    k = (np.arange(guide.size) % (gd + 1)).reshape(guide.shape).astype(np.float32)
    edge = ((k + 0.5) / gd).astype(np.float32)
    guide = np.where(rng.rand(*guide.shape) < 0.3, edge, guide).astype(np.float32)
    guide = np.where(rng.rand(*guide.shape) < 0.1, np.nextafter(edge, np.float32(0)), guide)
    got = hdrnet_ops.slice_indices(cuda(guide), (gh, gw, gd)).cpu().numpy()
    assert np.array_equal(got, oracle.port().slice_indices(guide, gh, gw, gd))


def test_guide_outside_unit_range_clamps_like_reference():
    grid, guide, inp = rand_case(17, 1, 16, 256, 4, 4, 8, signed=True)
    guide[0, :, ::3] = -0.75
    guide[0, :, 1::3] = 1.5
    guide[0, 0, :4] = [0.0, 1.0, 100.0, -100.0]
    expected = checker().bilateral_slice_apply(grid, guide, inp, True)
    for v in ("generic", "tma"):
        assert_parity(run_apply(grid, guide, inp, True, v), expected, what=v)
    grid, guide, inp = rand_case(18, 1, 9, 1920, 8, 16, 8, signed=True)
    guide[0, :, ::3] = -0.75
    guide[0, :, 1::3] = 1.5
    guide[0, 0, :4] = [0.0, 1.0, 100.0, -100.0]
    expected = checker().bilateral_slice_apply(grid, guide, inp, True)
    for v in ROW_KERNELS:
        assert_parity(run_apply(grid, guide, inp, True, v), expected, what=v)


def test_row_kernels_are_bitwise_equal():
    """Same per-pixel arithmetic whatever path a corner chunk travels (shared memory / texture) and
    whatever the control flow (block-synchronous / issuer warp, per-pixel / per-quad indices):
    results must be identical bits."""
    grid, guide, inp = rand_case(77, 2, 64, 3840, 16, 16, 8, signed=True)
    a = run_apply(grid, guide, inp, True, "tma")
    assert np.array_equal(a, run_apply(grid, guide, inp, True, "tex"))
    assert np.array_equal(a, run_apply(grid, guide, inp, True, "tex_async"))
    # smooth (image-like) guide: long runs of equal depth cells; and a constant guide
    yy, xx = np.mgrid[0:64, 0:3840]
    guide2 = np.stack([(0.5 + 0.5 * np.sin(xx / 700.0 + yy / 30.0)).astype(np.float32)] * 2)
    const = np.full_like(guide, 0.3)
    for gu in (guide2, const):
        a = run_apply(grid, gu, inp, True, "tma")
        assert np.array_equal(a, run_apply(grid, gu, inp, True, "tex_async"))


def _knob_shas(env, *args):
    """{case: sha256} of the seeded cases of tests/knob_runner.py, computed in a process of its own
    (the library reads its tuning record once per process)."""
    import subprocess, sys
    e = {k: v for k, v in os.environ.items() if not k.startswith("HDRNET_")}
    e.update(env)
    runner = os.path.join(os.path.dirname(os.path.abspath(__file__)), "knob_runner.py")
    out = subprocess.run([sys.executable, runner, *map(str, args)], env=e, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout + out.stderr
    return dict(l.split()[1:3] for l in out.stdout.splitlines() if l.startswith("SHA256"))


@pytest.mark.parametrize("env", [dict(HDRNET_ASYNC_THREADS="512"), dict(HDRNET_ASYNC_SLAB="0"),
                                 dict(HDRNET_ASYNC_SLAB="1"), dict(HDRNET_ASYNC_SLAB="1", HDRNET_TEX_CHUNKS="4"),
                                 dict(HDRNET_ASYNC_THREADS="512", HDRNET_TEX_CHUNKS="4")],
                         ids=lambda e: ",".join(f"{k[7:].lower()}={v}" for k, v in e.items()))
def test_issuer_warp_kernel_knobs_are_bitwise_equal(env):
    """Both CTA shapes of the issuer-warp form, slab rows from the pre-pass or from the slab warp
    inside the kernel, and 4 / 5 of a pixel's 12 corner chunks on the texture pipe: identical bits; also on narrow x cells (W < 4 gw: per-pixel indices), many rows
    per CTA, a ragged last segment and out-of-range guides."""
    import hashlib
    import knob_runner
    got = _knob_shas(env, "apply", _lib.VARIANT_TEX_ASYNC)
    for k, (seed, B, H, W, gh, gw, gd, edge) in enumerate(knob_runner.APPLY_CASES):
        grid, guide, inp = rand_case(seed, B, H, W, gh, gw, gd, signed=True)
        if edge:
            guide[0, :, ::5] = 1.75
            guide[0, :, 1::5] = -0.6
        want = hashlib.sha256(run_apply(grid, guide, inp, True, "tex").tobytes()).hexdigest()
        assert got[f"apply{k}"] == want, (env, k)


def test_empty_batch_is_a_no_op():
    """bilateral_slice_apply.cu.cc:373-379: empty output => no launch."""
    out = hdrnet_ops.bilateral_slice_apply(torch.zeros(0, 4, 4, 4, 12).cuda(),
                                           torch.zeros(0, 8, 8).cuda(),
                                           torch.zeros(0, 8, 8, 3).cuda(), True)
    assert out.shape == (0, 8, 8, 3)


def test_layers_wrappers_on_6d_grid():
    """hdrnet/layers.py:99-148: 6-D coefficient grids, both packings; fused == slice + apply."""
    rng = np.random.RandomState(9)
    B, H, W, gh, gw, gd, n_out, n_in1 = 2, 24, 132, 4, 4, 8, 3, 4
    coeffs = rng.randn(B, gh, gw, gd, n_out, n_in1).astype(np.float32)
    guide = rng.rand(B, H, W).astype(np.float32)
    im = rng.rand(B, H, W, 3).astype(np.float32)
    fused = layers.bilateral_slice_apply(cuda(coeffs), cuda(guide), cuda(im), has_offset=True)
    sliced = layers.bilateral_slice(cuda(coeffs), cuda(guide))
    assert sliced.shape == (B, H, W, n_out, n_in1)
    unfused = layers.apply(sliced, cuda(im), has_affine_term=True)
    assert_parity(unfused.cpu().numpy(), fused.cpu().numpy())
    expected = checker().bilateral_slice_apply(coeffs.reshape(B, gh, gw, gd, 12), guide, im, True)
    assert_parity(fused.cpu().numpy(), expected)


def test_host_buffer_path_matches_device_path():
    """CPU tensors go through the pipelined host path (row bands, y offsets)."""
    grid, guide, inp = rand_case(31, 2, 700, 1024, 16, 16, 8, signed=True)
    dev = run_apply(grid, guide, inp, True)
    host = hdrnet_ops.bilateral_slice_apply(torch.from_numpy(grid).pin_memory(),
                                            torch.from_numpy(guide).pin_memory(),
                                            torch.from_numpy(inp).pin_memory(), True)
    assert not host.is_cuda
    assert np.array_equal(host.numpy(), dev)
    pageable = hdrnet_ops.bilateral_slice_apply(torch.from_numpy(grid), torch.from_numpy(guide),
                                                torch.from_numpy(inp), True)
    assert np.array_equal(pageable.numpy(), dev)


def test_non_default_stream_and_repeatability():
    grid, guide, inp = rand_case(41, 2, 64, 640, 8, 8, 8)
    g, u, i = cuda(grid), cuda(guide), cuda(inp)
    ref = hdrnet_ops.bilateral_slice_apply(g, u, i, True)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        outs = [hdrnet_ops.bilateral_slice_apply(g, u, i, True) for _ in range(5)]
    s.synchronize()
    for o in outs:
        assert torch.equal(o, ref)


def test_two_streams_on_large_images_do_not_share_a_workspace():
    """>= 2 Mi-pixel calls take the texture-assisted kernel, whose pre-pass writes the slab rows of
    THIS call into a lent workspace: two streams (and two threads -- ctypes releases the GIL) with
    different grids must not see each other's rows (round 1 kept one workspace per device)."""
    import threading
    cases = [rand_case(50 + k, 1, 1100, 2048, 16, 16, 8, signed=True) for k in range(2)]
    dev = [tuple(cuda(a) for a in c) for c in cases]
    want = [hdrnet_ops.bilateral_slice_apply(*d, True) for d in dev]
    torch.cuda.synchronize()
    streams = [torch.cuda.Stream() for _ in dev]
    got = [[] for _ in dev]

    def work(k):
        with torch.cuda.stream(streams[k]):
            for _ in range(12):
                got[k].append(hdrnet_ops.bilateral_slice_apply(*dev[k], True))
    threads = [threading.Thread(target=work, args=(k,)) for k in range(len(dev))]
    for t in threads: t.start()
    for t in threads: t.join()
    torch.cuda.synchronize()
    for k in range(len(dev)):
        for o in got[k]:
            assert torch.equal(o, want[k]), f"stream {k}: result changed under a concurrent call"


# ---- row bands: the multi-GPU fallback for fewer images than GPUs (SURVEY.md section 8e) ---------
@pytest.mark.parametrize("B,H,W,world", [(1, 67, 256, 4), (3, 50, 384, 8), (2, 5, 128, 8)])
def test_row_bands_tile_the_whole_image_call(B, H, W, world):
    """Every rank's part (parallel.slice_apply_sharded, ranks emulated one after the other on this
    GPU) placed into the output equals the whole-image call: against the oracle through AUTO, and bit
    for bit when band and whole image run the same row kernel."""
    from hdrnet_b200 import parallel
    grid, guide, inp = rand_case(77, B, H, W, 16, 16, 8, signed=True)
    g, u, i = cuda(grid), cuda(guide), cuda(inp)
    out = torch.full((B, H, W, 3), float("nan"), device="cuda")
    for rank in range(world):
        (kind, lo, hi), part = parallel.slice_apply_sharded(g, u, i, True, rank, world)
        assert kind == ("batch" if B >= world else "rows")
        if kind == "batch":
            out[lo:hi] = part
        else:
            out[:, lo:hi] = part
    assert_parity(out.cpu().numpy(), checker().bilateral_slice_apply(grid, guide, inp, True),
                  what=f"row bands {B}x{H}x{W} over {world} ranks")
    whole = hdrnet_ops.bilateral_slice_apply(g, u, i, True, variant=_lib.VARIANT_TMA)
    bands = torch.cat([hdrnet_ops.bilateral_slice_apply_rows(g, u[:, y0:y1], i[:, y0:y1], True, y0, H,
                                                            variant=_lib.VARIANT_TMA)
                       for y0, y1 in (parallel.shard_rows(H, r, world) for r in range(world)) if y1 > y0], dim=1)
    assert torch.equal(bands, whole)


def test_row_bands_of_a_4k_frame_take_the_workspace_kernels():
    """One 4K frame over two ranks: each band (1080 rows = 4.1 MP) is large enough for AUTO to lend a
    workspace and run the issuer-warp kernel with a non-zero row offset; the bands equal the rows of
    the whole-frame call bit for bit (every row-kernel form produces the same bits)."""
    from hdrnet_b200 import parallel
    grid, guide, inp = rand_case(78, 1, 2160, 3840, 16, 16, 8)
    g, u, i = cuda(grid), cuda(guide), cuda(inp)
    whole = hdrnet_ops.bilateral_slice_apply(g, u, i, True)
    for rank in range(2):
        (kind, y0, y1), part = parallel.slice_apply_sharded(g, u, i, True, rank, 2)
        assert kind == "rows" and (y0, y1) == (1080 * rank, 1080 * (rank + 1))
        assert torch.equal(part, whole[:, y0:y1]), f"band of rank {rank} differs from the whole-frame call"
    with pytest.raises(ValueError):
        hdrnet_ops.bilateral_slice_apply_rows(g, u[:, :100], i[:, :100], True, y_off=2100, height=2160)


# ---- BASELINE.json full size: 4K ------------------------------------------------------------
def test_4k_frame_against_full_oracle():
    """One 3840x2160 frame, grid 16x16x8 (config 3's per-image shape), full oracle compare."""
    grid, guide, inp = rand_case(1234, 1, 2160, 3840, 16, 16, 8)
    expected = checker().bilateral_slice_apply(grid, guide, inp, True)
    for v in ("tma", "generic", "tex", "tex_async"):
        got = run_apply(grid, guide, inp, True, v)
        assert_parity(got, expected, what=f"4K [{v}]")
    gidx = hdrnet_ops.slice_indices(cuda(guide), (16, 16, 8)).cpu().numpy()
    assert np.array_equal(gidx, oracle.port().slice_indices(guide, 16, 16, 8))


def test_benchmarked_call_against_the_full_oracle():
    """The call bench.py times -- 8 x 3840 x 2160, grid 16x16x8, AUTO with a lent workspace --
    compared element by element with the compiled reference loops (oracle/_ref), all 66 MP."""
    grid, guide, inp = rand_case(1234, 8, 2160, 3840, 16, 16, 8)
    expected = checker().bilateral_slice_apply(grid, guide, inp, True)
    got = run_apply(grid, guide, inp, True, "auto")
    assert_parity(got, expected, what="8 x 4K [auto]")
    del got, expected


def test_12mp_frame_and_largest_grid_against_the_full_oracle():
    """Config 4's frame size (3024 x 4032) and config 5's largest grid (32x32x16) through AUTO."""
    grid, guide, inp = rand_case(7, 1, 3024, 4032, 16, 16, 8, signed=True)
    assert_parity(run_apply(grid, guide, inp, True, "auto"),
                  checker().bilateral_slice_apply(grid, guide, inp, True), what="12 MP [auto]")
    grid, guide, inp = rand_case(8, 1, 2160, 3840, 32, 32, 16, signed=True)
    assert_parity(run_apply(grid, guide, inp, True, "auto"),
                  checker().bilateral_slice_apply(grid, guide, inp, True), what="4K 32x32x16 [auto]")


def test_4k_batch8_properties():
    """Config 3 (8 x 4K) through size-independent properties: the two kernel variants agree,
    the op is linear in the grid, an identity grid returns in * sum(w) with sum(w) in
    [0.9999, 1], and image b only depends on grid b."""
    B, H, W, gh, gw, gd = 8, 2160, 3840, 16, 16, 8
    gen = torch.Generator(device="cuda").manual_seed(1234)
    grid = torch.rand(B, gh, gw, gd, 12, device="cuda", generator=gen)
    guide = torch.rand(B, H, W, device="cuda", generator=gen)
    inp = torch.rand(B, H, W, 3, device="cuda", generator=gen)
    out = hdrnet_ops.bilateral_slice_apply(grid, guide, inp, True)
    gen_out = hdrnet_ops.bilateral_slice_apply(grid, guide, inp, True, variant=_lib.VARIANT_GENERIC)
    scale = out.abs().max().item()
    assert (out - gen_out).abs().max().item() / scale <= RTOL
    del gen_out
    # linearity in the grid
    grid2 = torch.rand(B, gh, gw, gd, 12, device="cuda", generator=gen)
    lin = hdrnet_ops.bilateral_slice_apply(2.0 * grid - 0.5 * grid2, guide, inp, True)
    out2 = hdrnet_ops.bilateral_slice_apply(grid2, guide, inp, True)
    assert (lin - (2.0 * out - 0.5 * out2)).abs().max().item() / scale <= 4 * RTOL
    del lin, out2, grid2
    # identity coefficients
    ident = torch.zeros(B, gh, gw, gd, 3, 4, device="cuda")
    for i in range(3):
        ident[..., i, i] = 1.0
    ido = hdrnet_ops.bilateral_slice_apply(ident.reshape(B, gh, gw, gd, 12), guide, inp, True)
    ratio = ido / inp.clamp_min(1e-3)
    mask = inp > 1e-3
    assert ratio[mask].max().item() <= 1.0 + 1e-5 and ratio[mask].min().item() >= 0.9999 - 1e-5
    # batch independence: permuting images permutes outputs
    perm = torch.tensor([3, 0, 7, 1, 6, 2, 5, 4], device="cuda")
    outp = hdrnet_ops.bilateral_slice_apply(grid[perm].contiguous(), guide[perm].contiguous(),
                                            inp[perm].contiguous(), True)
    assert torch.equal(outp, out[perm])
