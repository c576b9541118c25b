"""Generate the golden fixtures in tests/golden/ from the REFERENCE itself.

Needs the reference's sources (oracle/jax_shim.py imports its JAX file; oracle/_ref is built from its
.cc files by oracle/Makefile):   python tests/golden/make_golden.py [jax | vjp | ref]

Outputs are produced by the reference's own jax/bilateral_slice.py (:299-380), imported
unmodified under the numpy stand-in for jax (oracle/jax_shim.py), and -- for slice-apply --
the reference's ``apply`` semantics (hdrnet/layers.py:153-198).  Inputs follow the
reference's tests:

  ops_test_extents   hdrnet/hdrnet_ops_test.py:91-113, :267-292 -- np.random.seed(1234),
                     np.random.rand, B=3 H=30 W=25 gh=16 gw=12 gd=8, n_in=3, n_out=3
  jax_tf2_extents    hdrnet/hdrnet_ops_jax_tf2_test.py:28-34 grid 16x12x8x2 (guide reduced
                     from 640x480x4 to 2x96x128 to keep the fixture small)
  interpolate_kat    hdrnet/test/ops_test.py:61-86 (grid value = depth index)
  edge_cases         guide exactly 0 / 1 / out of [0,1], 1-pixel-wide image, gd = 1
  signed_random      signed grid and input (tests/util.py rand_case(11, ...)) on a non-square grid
  vjp_*              the reference's own VJPs of the slice (jax/bilateral_slice.py:26-108, :257-295) at
                     the extents of its gradient tests (hdrnet_ops_test.py:91-100, :185-195) and on a
                     grid coarser / finer than the image, and vjp_cell_centre: a guide on an exact
                     depth-cell centre, where the JAX helpers and the C++ op differ
  compiled_ref_sha256.json
                     the reference's own C++ loops (oracle/_ref): forward at three extents and all five
                     VJPs at hdrnet_ops_test.py:185-195's, on tests/util.py rand_case inputs.  The C
                     restatement must match them bit for bit, so only the SHA-256 of each output's
                     float32 bytes is stored
Each forward .npz stores inputs, outputs and the reference's cell indices.
"""
import hashlib
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.normpath(os.path.join(HERE, "..", "..")))
sys.path.insert(0, os.path.normpath(os.path.join(HERE, "..")))

from oracle import jax_shim  # noqa: E402


def save(name, **arrays):
    path = os.path.join(HERE, name + ".npz")
    np.savez_compressed(path, **arrays)
    print(f"{name}: {os.path.getsize(path) / 1024:.1f} KiB", {k: v.shape for k, v in arrays.items()})


def case(grid, guide, inp=None):
    gh, gw, gd = grid.shape[1:4]
    d = dict(grid=grid, guide=guide,
             slice=jax_shim.bilateral_slice(grid, guide),
             indices=jax_shim.slice_indices(guide, gh, gw, gd))
    if inp is not None:
        d["input"] = inp
        n_in = inp.shape[-1]
        if grid.shape[-1] % (n_in + 1) == 0:
            d["apply_offset"] = jax_shim.bilateral_slice_apply(grid, guide, inp, True)
        if grid.shape[-1] % n_in == 0:
            d["apply_nooffset"] = jax_shim.bilateral_slice_apply(grid, guide, inp, False)
    return d


def main():
    # hdrnet_ops_test.py:91-113 / :267-292
    np.random.seed(1234)
    B, H, W, gh, gw, gd, n_in, n_out = 3, 30, 25, 16, 12, 8, 3, 3
    grid = np.random.rand(B, gh, gw, gd, (n_in + 1) * n_out).astype(np.float32)
    guide = np.random.rand(B, H, W).astype(np.float32)
    inp = np.random.rand(B, H, W, n_in).astype(np.float32)
    save("ops_test_extents", **case(grid, guide, inp))

    # hdrnet_ops_jax_tf2_test.py:28-34 (reduced spatial size), unseeded there -> seeded here
    rng = np.random.RandomState(20240)
    grid = rng.rand(2, 16, 12, 8, 2).astype(np.float32)
    guide = rng.rand(2, 96, 128).astype(np.float32)
    save("jax_tf2_extents", **case(grid, guide))

    # hdrnet/test/ops_test.py:61-86: expected output == val (tolerance 5e-4 there)
    for val in range(3):
        grid = np.zeros((3, 3, 4, 3, 1), np.float32)
        grid[:, :, :, 1] = 1.0
        grid[:, :, :, 2] = 2.0
        guide = np.full((3, 10, 9), (val + 0.5) / 3.0, np.float32)
        save(f"interpolate_kat_{val}", **case(grid, guide))

    # Edge cases: guide on / beyond the range ends, W = 4 strip, gd = 1, non-square grid.
    rng = np.random.RandomState(7)
    grid = rng.randn(2, 5, 3, 4, 12).astype(np.float32)
    guide = rng.rand(2, 12, 16).astype(np.float32)
    guide[0, 0, :4] = [0.0, 1.0, -0.25, 1.5]
    guide[1, 3, :4] = [0.125, 0.5, 0.875, 1.0 - 2.0 ** -24]
    inp = rng.randn(2, 12, 16, 3).astype(np.float32)
    save("edge_guides", **case(grid, guide, inp))

    grid = rng.rand(1, 2, 2, 1, 12).astype(np.float32)  # gd = 1: both depth corners clamp to 0
    guide = rng.rand(1, 7, 4).astype(np.float32)
    inp = rng.rand(1, 7, 4, 3).astype(np.float32)
    save("edge_gd1", **case(grid, guide, inp))

    # Wide enough for the TMA row kernel (W % 4 == 0, W >= 128), ragged last segment.
    grid = rng.rand(2, 4, 6, 8, 12).astype(np.float32)
    guide = rng.rand(2, 5, 1100).astype(np.float32)
    inp = rng.rand(2, 5, 1100, 3).astype(np.float32)
    save("wide_rows", **case(grid, guide, inp))

    # Signed grid and input on a small non-square grid (tests/util.py draws them this way).
    from util import rand_case
    save("signed_random", **case(*rand_case(11, 2, 40, 36, 8, 6, 5, signed=True)))


def main_vjp():
    # (B, H, W, gh, gw, gd, gc): default test extents; hdrnet_ops_test.py:185-195; a coarse grid; an
    # image narrower than the grid (cells without a pixel centre).  Guides are generic random values:
    # where guide * gd - 0.5 is EXACTLY an integer the JAX helpers take floor == ceil as two corners
    # (the grid VJP counts the pixel twice, the guide VJP returns 0) while the C++ op -- which the
    # library and the oracle port follow -- uses cells k and k + 1; tests/test_oracle.py pins that corner.
    for k, (B, H, W, gh, gw, gd, gc) in enumerate([(3, 30, 25, 16, 12, 8, 12), (3, 8, 5, 6, 3, 7, 4),
                                                   (2, 21, 36, 5, 4, 6, 2), (1, 9, 7, 3, 12, 9, 5)]):
        rng = np.random.RandomState(900 + k)
        grid = rng.randn(B, gh, gw, gd, gc).astype(np.float32)
        guide = rng.rand(B, H, W).astype(np.float32)
        ct = rng.randn(B, H, W, gc).astype(np.float32)
        gv, uv = jax_shim.bilateral_slice_vjp(grid, guide, ct)
        save(f"vjp_{k}", grid=grid, guide=guide, codomain_tangent=ct, grid_vjp=gv, guide_vjp=uv)

    # One pixel's guide on the centre of depth cell 1 (guide * gd - 0.5 == 1 exactly in float32), zero grid:
    # the inputs of tests/test_oracle.py's exact-cell-centre test.
    gh, gw, gd, gc, h, w = 3, 2, 4, 1, 6, 5
    rng = np.random.RandomState(11)
    guide = rng.rand(1, h, w).astype(np.float32)
    guide[0, 2, 3] = 1.5 / gd
    ct = rng.randn(1, h, w, gc).astype(np.float32)
    grid = np.zeros((1, gh, gw, gd, gc), np.float32)
    gv, uv = jax_shim.bilateral_slice_vjp(grid, guide, ct)
    save("vjp_cell_centre", grid=grid, guide=guide, codomain_tangent=ct, grid_vjp=gv, guide_vjp=uv)


# tests/test_oracle.py test_port_is_bit_exact_with_compiled_reference's extents (B, H, W, gh, gw, gd)
COMPILED_REF_SHAPES = [(3, 30, 25, 16, 12, 8), (2, 64, 48, 3, 5, 4), (1, 8, 5, 6, 3, 7)]


def sha256(a):
    return hashlib.sha256(np.ascontiguousarray(a, np.float32).tobytes()).hexdigest()


def main_compiled_ref():
    import oracle
    from util import rand_case
    ref = oracle.ref()
    digests = {}
    for shape in COMPILED_REF_SHAPES:
        grid, guide, inp = rand_case(99, *shape, signed=True)
        digests["x".join(map(str, shape))] = {
            "slice": sha256(ref.bilateral_slice(grid, guide)),
            "apply_offset": sha256(ref.bilateral_slice_apply(grid, guide, inp, True)),
            "apply_nooffset": sha256(ref.bilateral_slice_apply(grid, guide, inp, False))}
    # the VJPs, as tests/test_oracle.py test_port_vjps_bit_exact_with_compiled_reference draws its inputs
    B, H, W, gh, gw, gd, n_in, n_out = 3, 8, 5, 6, 3, 7, 3, 4
    grid, guide, inp = rand_case(5, B, H, W, gh, gw, gd, n_in, n_out, True)
    rng = np.random.RandomState(6)
    ct = rng.rand(B, H, W, n_out).astype(np.float32)
    vjp = dict(zip(("apply_grid", "apply_guide", "apply_input"),
                   map(sha256, ref.bilateral_slice_apply_grad(grid, guide, inp, ct, True))))
    ct = rng.rand(B, H, W, grid.shape[-1]).astype(np.float32)
    vjp.update(zip(("slice_grid", "slice_guide"), map(sha256, ref.bilateral_slice_grad(grid, guide, ct))))
    digests["vjp"] = vjp
    path = os.path.join(HERE, "compiled_ref_sha256.json")
    with open(path, "w") as f:
        json.dump(digests, f, indent=1, sort_keys=True)
        f.write("\n")
    print(f"compiled_ref_sha256.json: {len(digests)} cases")


if __name__ == "__main__":
    what = sys.argv[1:] or ["jax", "vjp", "ref"]
    if "jax" in what:
        main()
    if "vjp" in what:
        main_vjp()
    if "ref" in what:
        main_compiled_ref()
