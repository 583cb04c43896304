"""GPU parity tests: every stage and the whole path, through the C ABI, against the CPU oracle.

Bars (BASELINE.json north_star): descriptors, integer disparities and the valid mask bit-exact;
corrmap within 1e-5 (float) / 1e-12 (double); subpixel disparity within 1e-3 px. The kernels
reproduce the reference's operation order, so the tests additionally report (and for float
require) exact equality.
"""

import numpy as np
import pytest

import libbicos_b200 as lb
from libbicos_b200 import Config, synth

pytestmark = pytest.mark.gpu


@pytest.fixture(params=["auto", "popc"])
def engine(request):
    """Both search engines: 'auto' = tensor cores (tcgen05) wherever they apply, 'popc' = the integer-pipe kernel."""
    lb.set_search_engine(request.param)
    yield request.param
    lb.set_search_engine("auto")


FLAG_NODUPES, FLAG_CONSISTENCY = 1, 2


def _cuda(a):
    import torch

    if a.dtype == np.uint16:
        return torch.from_numpy(a.view(np.int16)).cuda().view(torch.uint16)
    return torch.from_numpy(a).cuda()


def _words(desc, k, cols):
    """pitched int32 [rows, pitch] -> uint32 numpy [rows, cols, k]"""
    rows = desc.shape[0]
    return desc.cpu().numpy().view(np.uint32)[:, : cols * k].reshape(rows, cols, k)


def _same(a, b):
    return np.array_equal(a, b, equal_nan=True) if a.dtype.kind == "f" else np.array_equal(a, b)


# ------------------------------------------------------------------------- transform --
@pytest.mark.parametrize(
    "n,dtype,full,cols",
    [
        (2, np.uint8, False, 64), (3, np.uint8, False, 61), (4, np.uint16, False, 64),
        (9, np.uint8, False, 128), (10, np.uint8, False, 131), (17, np.uint16, False, 96),
        (18, np.uint8, False, 64), (33, np.uint8, False, 256), (33, np.uint16, False, 130),
        (34, np.uint8, False, 66), (64, np.uint8, False, 128), (65, np.uint16, False, 64),
        (2, np.uint8, True, 64), (5, np.uint8, True, 67), (6, np.uint16, True, 64),
        (8, np.uint8, True, 128), (9, np.uint16, True, 64), (12, np.uint8, True, 256),
        (13, np.uint8, True, 64), (16, np.uint16, True, 128), (16, np.uint8, True, 63),
    ],
)
def test_transform_bit_exact(handle, oracles, n, dtype, full, cols):
    rows = 40
    left, right, _ = synth.make_stacks(n, rows, cols, dtype, seed=n * 7 + cols)
    # extremes: saturated, zero and near-constant pixels stress the integer mean comparison
    left[:, 0, :] = np.iinfo(dtype).max
    left[:, 1, :] = 0
    left[:, 2, :] = 100
    left[n // 2, 2, ::3] = 101
    for stack in (left, right):
        want = oracles.port.descriptors(stack, full)
        desc, k = handle.transform(_cuda(stack), full)
        got = _words(desc, k, cols)
        assert k == want.shape[2]
        assert np.array_equal(got, want), f"{(got != want).any(axis=2).sum()} descriptors differ"


def test_transform_strided_view(handle, oracles):
    """Planes that are views into a wider allocation (pitch > cols) and an odd pitch (scalar path)."""
    import torch

    n, rows, cols = 33, 24, 100
    left, _, _ = synth.make_stacks(n, rows, cols + 7, np.uint8, seed=5)
    big = _cuda(left)
    view = big[:, :, 3 : 3 + cols]
    want = oracles.port.descriptors(np.ascontiguousarray(left[:, :, 3 : 3 + cols]), False)
    desc, k = handle.transform(view, False)
    assert np.array_equal(_words(desc, k, cols), want)
    assert torch.cuda.current_stream().query() or True


# ---------------------------------------------------------------------------- search --
def _random_desc(rng, rows, cols, k, bits):
    """Descriptors with few distinct values per word, so ties and duplicates are frequent."""
    return rng.integers(0, 1 << bits, size=(rows, cols, k), dtype=np.int64).astype(np.uint32)


@pytest.mark.parametrize("k", [1, 2, 4, 8, 12, 16])
@pytest.mark.parametrize("flags", [FLAG_NODUPES, FLAG_CONSISTENCY, FLAG_NODUPES | FLAG_CONSISTENCY])
@pytest.mark.parametrize("cols,bits", [(97, 3), (512, 8), (700, 32), (1300, 5)])
def test_search_postfilter_bit_exact(handle, oracles, engine, k, flags, cols, bits):
    import torch

    rng = np.random.default_rng(k * 100 + flags * 10 + cols)
    rows = 6
    d0 = _random_desc(rng, rows, cols, k, bits)
    d1 = _random_desc(rng, rows, cols, k, bits)
    # plant some true matches so that low costs and unique minima occur too
    src = rng.integers(0, cols, size=cols // 2)
    dst = rng.integers(0, cols, size=cols // 2)
    d0[:, dst] = d1[:, src] ^ (rng.integers(0, 2, size=(rows, cols // 2, k)) << 7).astype(np.uint32)
    max_lr = 3
    want = oracles.port.bicos(d0, d1, flags, max_lr)

    pitch = (cols * k + 3) // 4 * 4

    def pitched(d):
        buf = np.zeros((rows, pitch), dtype=np.uint32)
        buf[:, : cols * k] = d.reshape(rows, cols * k)
        return torch.from_numpy(buf.view(np.int32)).cuda()

    keys = handle.search(pitched(d0), pitched(d1), k, cols, flags)
    # postfilter only (threshold unset): the int16 disparity of reference bicos()
    dummy = torch.zeros((2, rows, cols), dtype=torch.uint8, device="cuda")
    cfg = Config(nxcorr_threshold=None, consistency=bool(flags & FLAG_CONSISTENCY), max_lr_diff=max_lr,
                 no_dupes=flags == 3)
    disp, corr, raw = handle.refine(dummy, dummy, cfg, keys)
    got = disp.cpu().numpy()
    assert corr is None and got.dtype == np.int16
    assert np.array_equal(got, want), f"{(got != want).sum()} of {got.size} disparities differ"
    assert np.array_equal(raw.cpu().numpy(), want)


# ------------------------------------------------------------------------- whole path --
CASES = [
    # n, dtype, rows, cols, config
    (33, np.uint8, 48, 320, dict(nxcorr_threshold=0.96, min_variance=2.0)),  # BASELINE config 1 (small)
    (33, np.uint8, 48, 320, dict(nxcorr_threshold=0.96, min_variance=2.0, subpixel_step=0.1, consistency=True,
                                 max_lr_diff=1)),  # BASELINE config 2 (small)
    (33, np.uint8, 40, 300, dict(nxcorr_threshold=None)),
    (33, np.uint8, 40, 300, dict(nxcorr_threshold=0.5)),
    (33, np.uint8, 40, 300, dict(nxcorr_threshold=0.9, subpixel_step=0.25, consistency=True, max_lr_diff=2,
                                 no_dupes=True)),
    (16, np.uint16, 40, 288, dict(nxcorr_threshold=0.9, mode_full=True, min_variance=1.0)),  # config 3 shape
    (16, np.uint16, 40, 288, dict(nxcorr_threshold=0.9, mode_full=True, subpixel_step=0.1, consistency=True)),
    (64, np.uint8, 32, 256, dict(nxcorr_threshold=0.9, min_variance=2.0)),  # config 4 shape: 256-bit
    (64, np.uint8, 32, 256, dict(nxcorr_threshold=0.9, subpixel_step=0.2, min_variance=2.0)),
    (9, np.uint8, 32, 200, dict(nxcorr_threshold=0.8, subpixel_step=0.3)),
    (17, np.uint16, 32, 200, dict(nxcorr_threshold=0.8, subpixel_step=0.15, min_variance=4.0)),
    (12, np.uint8, 32, 200, dict(nxcorr_threshold=0.7, mode_full=True, consistency=True, max_lr_diff=0)),
    (2, np.uint8, 16, 100, dict(nxcorr_threshold=0.5, subpixel_step=0.5)),
    (5, np.uint16, 16, 101, dict(nxcorr_threshold=0.5, min_variance=0.0)),
]


@pytest.mark.parametrize("n,dtype,rows,cols,kw", CASES)
def test_match_float_parity(handle, oracles, n, dtype, rows, cols, kw):
    left, right, _ = synth.make_stacks(n, 512, cols, dtype, seed=11 * n + cols, row0=128, rows=rows)
    want_d, want_c = oracles.port.match(left, right, **kw)
    disp, corr = handle.match(_cuda(left), _cuda(right), Config(**kw))
    got_d = disp.cpu().numpy()
    assert got_d.dtype == want_d.dtype
    if want_d.dtype == np.int16:
        assert np.array_equal(got_d, want_d)
        assert corr is None
        return
    got_c = corr.cpu().numpy()
    invalid_w = np.isnan(want_d) | (want_d == -32768)
    invalid_g = np.isnan(got_d) | (got_d == -32768)
    # pixels whose NXC sits within 1e-6 of the threshold may flip (north_star); none expected
    edge = np.abs(np.nan_to_num(want_c, nan=9.0) - kw["nxcorr_threshold"]) < 1e-6
    assert np.array_equal(invalid_g | edge, invalid_w | edge), "valid masks differ"
    assert np.array_equal(np.isnan(got_c), np.isnan(want_c))
    ok = ~np.isnan(want_c)
    assert np.max(np.abs(got_c[ok] - want_c[ok]), initial=0) <= 1e-5
    both = ~(invalid_w | invalid_g)
    assert np.max(np.abs(got_d[both] - want_d[both]), initial=0) <= 1e-3
    # stronger: the kernels follow the reference's operation order, so everything is identical
    assert _same(got_c, want_c), f"corrmap: {(~np.isclose(got_c, want_c, rtol=0, atol=0, equal_nan=True)).sum()} differ"
    assert _same(got_d, want_d)
    assert both.mean() > 0.2 or n <= 5, "test scene should have valid matches"


# The kernels behind the headline numbers: the one-pass consistency kernel (128-bit descriptors, Consistency without
# no_dupes) needs the two free top bits only bicos_b200_match vouches for; variant 2 of the two-pass search (one CTA
# per SM, left operand in TMEM) is only dispatched when the image has at least two (direction, row, 256-pixel) items
# per SM, and the column-term form only through bicos_b200_match. These scenes are large enough for both and small enough for the
# oracle; bicos_b200_last_search_kernel() proves which kernel ran, so a change of the dispatch rule cannot
# silently take them out of the suite.
BENCHED = [
    # n, dtype, rows, cols, config, kernel expected on a 148-SM B200
    (33, np.uint8, 160, 512, dict(nxcorr_threshold=0.96, min_variance=2.0, subpixel_step=0.1, consistency=True, max_lr_diff=1),
     "mma3<K=4,nodupes=0,ct=2,onepass=1>"),  # the bench workload's configuration: the one-pass consistency kernel
    (33, np.uint8, 131, 700, dict(nxcorr_threshold=0.9, subpixel_step=0.25, consistency=True, max_lr_diff=0), "mma3<K=4,nodupes=0,ct=2,onepass=1>"),  # ragged tile and block
    (12, np.uint8, 140, 640, dict(nxcorr_threshold=0.9, mode_full=True, consistency=True, max_lr_diff=2), "mma3<K=4,nodupes=0,ct=2,onepass=1>"),  # FULL, 123 of 128 bits
    (33, np.uint8, 152, 520, dict(nxcorr_threshold=0.96, min_variance=2.0), "mma2<K=4,nodupes=1,ct=1,dirs=1>"),  # C1, ragged last tile
    (33, np.uint8, 160, 512, dict(nxcorr_threshold=0.9, subpixel_step=0.25, consistency=True, max_lr_diff=2, no_dupes=True),
     "mma2<K=4,nodupes=1,ct=1,dirs=2>"),
    (64, np.uint8, 160, 512, dict(nxcorr_threshold=0.9, min_variance=2.0), "mma2<K=8,nodupes=1,ct=1,dirs=1>"),  # C4: 256 bits
    (64, np.uint8, 100, 700, dict(nxcorr_threshold=0.9, subpixel_step=0.2, consistency=True, max_lr_diff=1),
     "mma3<K=8,nodupes=0,ct=2,onepass=1>"),  # 256 bits through the one-pass kernel (popcount byte with its bias)
    (16, np.uint16, 120, 600, dict(nxcorr_threshold=0.9, mode_full=True, consistency=True, max_lr_diff=1),
     "mma3<K=8,nodupes=0,ct=2,onepass=1>"),  # FULL, u16, 227 of 256 bits
    (16, np.uint16, 160, 512, dict(nxcorr_threshold=0.9, mode_full=True, consistency=True, max_lr_diff=1, no_dupes=True),
     "mma2<K=8,nodupes=1,ct=1,dirs=2>"),  # C3: FULL, u16
]


@pytest.mark.parametrize("n,dtype,rows,cols,kw,kernel", BENCHED)
@pytest.mark.parametrize("double", [False, True])
def test_match_parity_on_the_benchmarked_kernels(handle, oracles, n, dtype, rows, cols, kw, kernel, double):
    import torch

    if torch.cuda.get_device_properties(0).multi_processor_count != 148:
        pytest.skip("kernel expectations are for the 148 SMs of a B200")
    left, right, _ = synth.make_stacks(n, 1024, cols, dtype, seed=7 * n + rows, row0=300, rows=rows)
    want_d, want_c = oracles.port.match(left, right, double=double, **kw)
    lb.set_search_engine("auto")
    disp, corr = handle.match(_cuda(left), _cuda(right), Config(double=double, **kw))
    assert lb.last_search_kernel() == kernel
    got_d, got_c = disp.cpu().numpy(), corr.cpu().numpy()
    invalid_w = np.isnan(want_d) | (want_d == -32768)
    invalid_g = np.isnan(got_d) | (got_d == -32768)
    assert np.array_equal(invalid_g, invalid_w), "valid masks differ"
    assert np.array_equal(np.isnan(got_c), np.isnan(want_c))
    ok = ~np.isnan(want_c)
    assert np.max(np.abs(got_c[ok] - want_c[ok]), initial=0) <= (1e-12 if double else 1e-5)
    assert np.max(np.abs(got_d[~invalid_w] - want_d[~invalid_w]), initial=0) <= 1e-3
    assert _same(got_d, want_d) and _same(got_c, want_c)  # in fact identical
    assert (~invalid_w).mean() > 0.3, "test scene should have valid matches"


@pytest.mark.parametrize("n,dtype,rows,cols,kw", [c for c in CASES if c[4].get("nxcorr_threshold") is not None][:8])
def test_match_double_parity(handle, oracles, n, dtype, rows, cols, kw):
    left, right, _ = synth.make_stacks(n, 512, cols, dtype, seed=3 * n + cols, row0=64, rows=rows)
    want_d, want_c = oracles.port.match(left, right, double=True, **kw)
    disp, corr = handle.match(_cuda(left), _cuda(right), Config(double=True, **kw))
    got_d, got_c = disp.cpu().numpy(), corr.cpu().numpy()
    assert got_c.dtype == np.float64 and got_d.dtype == np.float32
    invalid_w = np.isnan(want_d) | (want_d == -32768)
    invalid_g = np.isnan(got_d) | (got_d == -32768)
    assert np.array_equal(invalid_g, invalid_w)
    assert np.array_equal(np.isnan(got_c), np.isnan(want_c))
    ok = ~np.isnan(want_c)
    assert np.max(np.abs(got_c[ok] - want_c[ok]), initial=0) <= 1e-12
    both = ~invalid_w
    assert np.max(np.abs(got_d[both] - want_d[both]), initial=0) <= 1e-3


# ------------------------------------------------- wide-descriptor extension (FULL, 17..23 images) --
@pytest.mark.parametrize("n,dtype,cols", [(17, np.uint8, 200), (18, np.uint16, 131), (20, np.uint16, 288), (20, np.uint8, 97),
                                          (21, np.uint8, 160), (22, np.uint16, 66), (23, np.uint16, 200)])
def test_wide_extension_parity(handle, oracles, n, dtype, cols):
    """BASELINE.json configs[2] names 2x20 uint16 FULL stacks: 363 bits, which the reference rejects. With
    Config.wide_descriptors the path runs on 12- / 16-word descriptors; the oracle's wide path is pinned against
    the reference's stage templates (tests/test_oracle.py)."""
    import libbicos_b200 as lb

    rows = 24
    left, right, _ = synth.make_stacks(n, 512, cols, dtype, seed=5 * n + cols, row0=96, rows=rows)
    k_want = 12 if n <= 20 else 16
    for stack in (left, right):
        want = oracles.port.descriptors(stack, True, wide=True)
        desc, k = handle.transform(_cuda(stack), True, wide=True)
        assert k == k_want == want.shape[2]
        assert np.array_equal(_words(desc, k, cols), want)
    for kw in (dict(nxcorr_threshold=None), dict(nxcorr_threshold=0.9, min_variance=1.0),
               dict(nxcorr_threshold=None, consistency=True, max_lr_diff=1, no_dupes=True),
               dict(nxcorr_threshold=0.85, subpixel_step=0.2, consistency=True, max_lr_diff=1)):
        kw = dict(kw, mode_full=True, wide_descriptors=True)
        want_d, want_c = oracles.port.match(left, right, **kw)
        disp, corr = handle.match(_cuda(left), _cuda(right), Config(**kw))
        assert _same(disp.cpu().numpy(), want_d), kw
        assert (corr is None and want_c is None) or _same(corr.cpu().numpy(), want_c)
        if kw["nxcorr_threshold"] is not None:
            want_d, want_c = oracles.port.match(left, right, double=True, **kw)
            disp, corr = handle.match(_cuda(left), _cuda(right), Config(double=True, **kw))
            assert _same(disp.cpu().numpy(), want_d)
            ok = ~np.isnan(want_c)
            assert np.array_equal(np.isnan(corr.cpu().numpy()), ~ok)
            assert np.max(np.abs(corr.cpu().numpy()[ok] - want_c[ok]), initial=0) <= 1e-12
    valid = ~np.isnan(want_d)
    assert valid.mean() > 0.2 or cols < 150, "wide test scenes should have valid matches"
    # without the extension flag the reference's error stands
    with pytest.raises(lb.BicosError, match="too large"):
        handle.match(_cuda(left), _cuda(right), Config(mode_full=True))


@pytest.mark.parametrize("rows,cols", [(1, 1), (1, 2), (2, 3), (3, 31), (1, 129), (2, 513), (1, 1025)])
def test_tiny_and_ragged_images(handle, oracles, rows, cols):
    """Degenerate sizes: single pixels, single rows, widths just past a unit / chunk boundary."""
    n = 9
    left, right, _ = synth.make_stacks(n, 64, max(cols, 8), np.uint8, seed=rows * 100 + cols, rows=rows)
    left, right = np.ascontiguousarray(left[:, :, :cols]), np.ascontiguousarray(right[:, :, :cols])
    for kw in (dict(nxcorr_threshold=None), dict(nxcorr_threshold=0.5, consistency=True, max_lr_diff=1, no_dupes=True),
               dict(nxcorr_threshold=0.3, subpixel_step=0.5, min_variance=0.5)):
        want_d, want_c = oracles.port.match(left, right, **kw)
        disp, corr = handle.match(_cuda(left), _cuda(right), Config(**kw))
        assert _same(disp.cpu().numpy(), want_d), (rows, cols, kw)
        if want_c is not None:
            assert _same(corr.cpu().numpy(), want_c), (rows, cols, kw)


@pytest.mark.parametrize("k,cols,flags", [(8, 4100, 3), (4, 4100, 2), (1, 9000, 1), (2, 2050, 3)])
def test_search_wide_rows_split_units(handle, oracles, engine, k, cols, flags):
    """Wide rows: several chunks per unit and up to 8 CTAs per unit merged by atomicMin (popc); 33 column tiles
    per item (tensor). 9000 columns are beyond the tensor-core engine: auto falls back to popc."""
    import torch

    rng = np.random.default_rng(k * 7 + cols)
    rows = 3
    d0 = _random_desc(rng, rows, cols, k, 6)
    d1 = _random_desc(rng, rows, cols, k, 6)
    src = rng.integers(0, cols, size=cols // 2)
    dst = rng.integers(0, cols, size=cols // 2)
    d0[:, dst] = d1[:, src]
    want = oracles.port.bicos(d0, d1, flags, 2)
    pitch = (cols * k + 3) // 4 * 4

    def pitched(d):
        buf = np.zeros((rows, pitch), dtype=np.uint32)
        buf[:, : cols * k] = d.reshape(rows, cols * k)
        return torch.from_numpy(buf.view(np.int32)).cuda()

    keys = handle.search(pitched(d0), pitched(d1), k, cols, flags)
    dummy = torch.zeros((2, rows, cols), dtype=torch.uint8, device="cuda")
    cfg = Config(nxcorr_threshold=None, consistency=bool(flags & FLAG_CONSISTENCY), max_lr_diff=2, no_dupes=flags == 3)
    disp, _, _ = handle.refine(dummy, dummy, cfg, keys)
    assert np.array_equal(disp.cpu().numpy(), want)


@pytest.mark.parametrize("k,rows,cols,flags", [(4, 700, 384, 3), (4, 40, 2048, 2), (8, 500, 300, 1), (8, 12, 2448, 3),
                                               (12, 330, 256, 2), (16, 310, 200, 3), (4, 1300, 130, 0), (4, 90, 1000, 2),
                                               (8, 200, 520, 2)])
@pytest.mark.parametrize("top_bit_free", [False, True, 2])
def test_search_engines_identical(handle, oracles, k, rows, cols, flags, top_bit_free):
    """The tensor-core engine (int8 GEMM + argmin epilogue) reproduces the popcount engine's four key arrays bit
    for bit, at sizes where a persistent CTA walks several work items (rows x M tiles x directions > resident CTAs)
    and with descriptors drawn from a small pool, so that exact ties are the rule. With `top_bit_free` the top
    descriptor bit is clear and the tensor-core engine is told so (BICOS_B200_FLAG_TOP_BIT_FREE): the column-term
    kernels bicos_b200_match uses, in both kernel variants; with top_bit_free = 2 the top two bits are clear
    (BICOS_B200_FLAG_TOP2_BITS_FREE) and 128-bit consistency searches take the one-pass kernel. The postfiltered
    disparity of the tensor-core keys is also compared with the oracle's bicos()."""
    import torch

    rng = np.random.default_rng(k + rows + cols + flags)
    pool = rng.integers(0, 2**32, size=(48, k), dtype=np.uint64).astype(np.uint32)

    def draw():
        d = pool[rng.integers(0, len(pool), size=(rows, cols))]
        flip = rng.integers(0, 4, size=(rows, cols, 1)) > 1
        bit = rng.integers(0, 32 * k - 2, size=(rows, cols))
        mask = np.zeros((rows, cols, k), dtype=np.uint32)
        np.put_along_axis(mask, (bit // 32)[..., None], (np.uint32(1) << (bit % 32).astype(np.uint32))[..., None], axis=2)
        d = d ^ (mask * flip)
        if top_bit_free:
            d[..., k - 1] &= np.uint32(0x3FFFFFFF if top_bit_free == 2 else 0x7FFFFFFF)
        return d

    pitch = (cols * k + 3) // 4 * 4

    def pitched(d):
        buf = np.zeros((rows, pitch), dtype=np.uint32)
        buf[:, : cols * k] = d.reshape(rows, cols * k)
        return torch.from_numpy(buf.view(np.int32)).cuda()

    n0, n1 = draw(), draw()
    d0, d1 = pitched(n0), pitched(n1)
    got, keys = {}, None
    try:
        for name in ("popc", "tensor"):
            lb.set_search_engine(name)
            keys = handle.search(d0, d1, k, cols, flags, top_bit_free=top_bit_free)
            got[name] = [None if a is None else a.cpu().numpy() for a in keys]
            kernel = lb.last_search_kernel()
            assert kernel.startswith("popc<" if name == "popc" else "mma"), kernel
    finally:
        lb.set_search_engine("auto")
    onepass = top_bit_free == 2 and k in (4, 8) and flags == FLAG_CONSISTENCY
    assert f"ct={2 if onepass else int(bool(top_bit_free) and k in (4, 8))}" in kernel, kernel
    if onepass:
        assert kernel.startswith("mma3<"), kernel
    elif torch.cuda.get_device_properties(0).multi_processor_count == 148:
        dirs = 2 if flags & FLAG_CONSISTENCY else 1
        v2 = k in (4, 8) and dirs * rows * ((cols + 255) // 256) >= 296
        assert kernel.startswith("mma2<" if v2 else "mma1<"), kernel
    for a, b, what in zip(got["popc"], got["tensor"], ("fwd_first", "fwd_last", "rev_first", "rev_last")):
        assert (a is None) == (b is None)
        if a is not None:
            assert np.array_equal(a, b), f"{what}: {(a != b).sum()} of {a.size} keys differ"
    if flags:  # flags 0 (plain first minimum) is a building block no Config reaches
        want = oracles.port.bicos(n0, n1, flags, 2)
        dummy = torch.zeros((2, rows, cols), dtype=torch.uint8, device="cuda")
        cfg = Config(nxcorr_threshold=None, consistency=bool(flags & FLAG_CONSISTENCY), max_lr_diff=2, no_dupes=flags == 3)
        disp, _, _ = handle.refine(dummy, dummy, cfg, keys)
        assert np.array_equal(disp.cpu().numpy(), want)


def test_tensor_engine_refuses_what_it_cannot_do(handle):
    """Forced tensor engine: 32-bit descriptors and rows beyond 8192 pixels are errors, not silent fallbacks."""
    import torch

    try:
        lb.set_search_engine("tensor")
        d = torch.zeros((2, 64), dtype=torch.int32, device="cuda")
        with pytest.raises(lb.BicosError):
            handle.search(d, d, 1, 64, FLAG_NODUPES)
        wide = torch.zeros((1, 9000 * 4), dtype=torch.int32, device="cuda")
        with pytest.raises(lb.BicosError):
            handle.search(wide, wide, 4, 9000, FLAG_NODUPES)
    finally:
        lb.set_search_engine("auto")
    assert lb.search_engine() == "auto"


def test_randomised_configurations(handle, oracles):
    """Seeded sweep over stack sizes, depths, modes, variants, steps and image shapes: every
    dispatch branch (descriptor width, unit size A, split count, full / partial stacks, packed and
    scalar subpixel paths, odd step counts) against the oracle, bit for bit."""
    rng = np.random.default_rng(20261018)
    checked = 0
    for trial in range(48):
        full = bool(rng.integers(0, 2)) and trial % 3 == 0
        n = int(rng.integers(2, 17)) if full else int(rng.choice([2, 3, 4, 5, 8, 9, 10, 16, 17, 18, 25, 32, 33, 34, 48, 64, 65]))
        dtype = np.uint16 if rng.integers(0, 2) else np.uint8
        rows, cols = int(rng.integers(1, 12)), int(rng.choice([17, 64, 100, 255, 256, 300, 513, 640, 777, 1100]))
        kw = dict(mode_full=full)
        kind = trial % 4
        if kind == 0:
            kw.update(nxcorr_threshold=None)
        else:
            kw.update(nxcorr_threshold=float(rng.choice([0.3, 0.7, 0.9, 0.96])))
            if rng.integers(0, 2):
                kw.update(min_variance=float(rng.choice([0.0, 1.0, 4.0])))
            if kind >= 2:
                kw.update(subpixel_step=float(rng.choice([0.1, 0.125, 0.2, 0.3, 0.4, 0.5, 0.7, 1.0])))
        if rng.integers(0, 2):
            kw.update(consistency=True, max_lr_diff=int(rng.integers(0, 4)), no_dupes=bool(rng.integers(0, 2)))
        double = kind == 3 and bool(rng.integers(0, 2))
        left, right, _ = synth.make_stacks(n, 256, cols, dtype, seed=1000 + trial, row0=int(rng.integers(0, 200)), rows=rows)
        want_d, want_c = oracles.port.match(left, right, double=double, **kw)
        disp, corr = handle.match(_cuda(left), _cuda(right), Config(double=double, **kw))
        assert _same(disp.cpu().numpy(), want_d), (trial, n, dtype, rows, cols, kw, double)
        if want_c is not None:
            assert _same(corr.cpu().numpy(), want_c), (trial, n, dtype, rows, cols, kw, double)
        checked += 1
    assert checked == 48


def _reference_outputs():
    import importlib.util
    import os

    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "make_reference_outputs.py")
    spec = importlib.util.spec_from_file_location("make_reference_outputs", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_match_against_unmodified_reference(handle, oracles):
    """Same comparison, but against the compiled reference sources themselves, or without them against the
    reference's outputs stored in tests/golden/reference/ (tests/golden/make_reference_outputs.py)."""
    ro = _reference_outputs()
    left, right = ro.gpu_inputs()
    live = oracles.ref.available()
    if not live:
        ro.check_inputs("gpu_match", left, right)
    for i, kw in enumerate(ro.GPU_KWS):
        disp, corr = handle.match(_cuda(left), _cuda(right), Config(**kw))
        got_d, got_c = disp.cpu().numpy(), corr.cpu().numpy()
        if live:
            want_d, want_c = oracles.ref.match(left, right, **kw)
            assert _same(got_d, want_d)
            assert _same(got_c, want_c)
        else:
            ro.check(f"gpu_match/{i}/disp", got_d)
            ro.check(f"gpu_match/{i}/corr", got_c)


def test_double_precision_against_reference_cuda_build(handle, oracles):
    """Pins the double-precision NXC (which the reference's CPU build does not have) against the
    reference's own CUDA backend, compiled unmodified for sm_100a (oracle/_ref/libbicos_refcuda.so), or without
    it against that backend's outputs stored in tests/golden/reference/ (the whole disparity, the corrmap on a
    seeded sample of pixels): same valid mask, correlation within 1e-12 wherever the reference evaluated it.
    Integer mode: the reference's CUDA build contracts the subpixel polynomial, so subpixel results are not
    comparable bit for bit (covered against the CPU oracle instead)."""
    import oracle

    ro = _reference_outputs()
    live = oracle.refcuda.available()
    for n, dtype, kw in ro.DOUBLE_CASES:
        left, right = ro.double_inputs(n, dtype)
        disp, corr = handle.match(_cuda(left), _cuda(right), Config(**kw))
        got_d, got_c = disp.cpu().numpy(), corr.cpu().numpy()
        sample = slice(None)
        if live:
            ref_d, ref_c = oracle.refcuda.match(left, right, **kw)
        else:
            ro.check_inputs(f"double_{n}", left, right)
            ref_d, ref_c = ro.stored()[1][f"double_{n}_disp"], ro.stored()[1][f"double_{n}_corr_sample"]
            sample = ro.double_sample(*got_d.shape)
        assert ref_d.dtype == np.int16 and ref_c.dtype == np.float64 and got_c.dtype == np.float64
        valid_ref = ref_d != -32768
        valid_got = got_d != -32768
        assert np.array_equal(valid_ref, valid_got)
        assert np.array_equal(ref_d[valid_ref].astype(np.float32), got_d[valid_got])
        # the reference leaves corrmap cells it never evaluated uninitialised: compare where we evaluated
        ev = ~np.isnan(got_c)
        assert ev.sum() > 0.5 * ev.size
        ref_c, got_c, ev = ref_c.reshape(-1), got_c.reshape(-1)[sample], ev.reshape(-1)[sample]
        assert np.max(np.abs(ref_c[ev] - got_c[ev])) <= 1e-12


def test_negative_threshold_evaluates_but_rejects_nothing(handle, oracles):
    """BICOS::Config{.nxcorr_threshold = -1}: what the reference CLI uses for --corrmap without
    --threshold (cli.cpp:150-153). The correlation map equals that of any other threshold, and every
    pixel whose correlation was evaluated keeps its raw disparity."""
    left, right, _ = synth.make_stacks(33, 256, 320, np.uint8, seed=12, row0=90, rows=40)
    l, r = _cuda(left), _cuda(right)
    raw, _ = handle.match(l, r, Config(nxcorr_threshold=None, consistency=True, max_lr_diff=1))
    d0, c0 = handle.match(l, r, Config(nxcorr_threshold=0.9, consistency=True, max_lr_diff=1, min_variance=2.0))
    dm, cm = handle.match(l, r, Config(nxcorr_threshold=-1.0, consistency=True, max_lr_diff=1, min_variance=2.0))
    want_c = oracles.port.match(left, right, nxcorr_threshold=0.0, consistency=True, max_lr_diff=1, min_variance=2.0)[1]
    assert _same(c0.cpu().numpy(), want_c) and _same(cm.cpu().numpy(), want_c)
    raw, dm, cm = raw.cpu().numpy(), dm.cpu().numpy(), cm.cpu().numpy()
    evaluated = ~np.isnan(cm)
    assert evaluated.mean() > 0.5 and (cm[evaluated] < 0.9).any()  # some matches a threshold of 0.9 rejects
    assert np.array_equal(dm[evaluated], raw[evaluated].astype(np.float32))
    assert (dm[~evaluated] == -32768).all()
    assert (d0.cpu().numpy()[evaluated & (cm < 0.9)] == -32768).all()


def test_match_host_and_rows(handle, oracles):
    """Host-buffer entry point and the row-sharded entry point give the same answer."""
    import torch

    kw = dict(nxcorr_threshold=0.9, subpixel_step=0.1, consistency=True, max_lr_diff=1, min_variance=2.0)
    left, right, _ = synth.make_stacks(33, 96, 256, np.uint8, seed=4)
    want_d, want_c = oracles.port.match(left, right, **kw)
    d, c = handle.match_host(left, right, Config(**kw))
    assert _same(d, want_d) and _same(c, want_c)
    l, r = _cuda(left), _cuda(right)
    disp = torch.full((96, 256), 7.0, dtype=torch.float32, device="cuda")
    corr = torch.full((96, 256), 7.0, dtype=torch.float32, device="cuda")
    for rb, re in ((0, 31), (31, 64), (64, 96)):
        handle.match(l, r, Config(**kw), out=(disp, corr), rows_range=(rb, re))
    assert _same(disp.cpu().numpy(), want_d) and _same(corr.cpu().numpy(), want_c)


def test_match_host_pipelined(handle, oracles):
    """bicos_b200_match_host_begin/_end: two frames in flight on two handles, non-contiguous planes too."""
    import libbicos_b200 as lb

    kw = dict(nxcorr_threshold=0.9, subpixel_step=0.2, min_variance=2.0)
    frames = [synth.make_stacks(17, 400, 192, np.uint16, seed=8, frame=f)[:2] for f in range(3)]
    want = [oracles.port.match(l, r, **kw) for l, r in frames]
    other = lb.Handle(0)
    hs = [handle, other]
    got = []
    for f, (l, r) in enumerate(frames):
        hs[f % 2].match_host_end()
        if f == 2:  # planes that are not back to back in memory: the per-plane upload path
            l = np.ascontiguousarray(np.concatenate([l, l], axis=1))[:, :400]
            assert not l.flags.c_contiguous
        got.append(hs[f % 2].match_host_begin(l, r, Config(**kw)))
    with pytest.raises(lb.BicosError, match="already in flight"):
        hs[0].match_host_begin(frames[0][0], frames[0][1], Config(**kw))
    for x in hs:
        x.match_host_end()
    for (d, c), (wd, wc) in zip(got, want):
        assert _same(d, wd) and _same(c, wc)
    other.close()


def test_match_batch_equals_single_matches(handle, oracles):
    """bicos_b200_match_batch (frames through two internal streams, frame f + 1's search beside frame f's refine, key
    buffers alternating) gives every frame exactly what bicos_b200_match gives it, and what the oracle gives."""
    import torch

    kw = dict(nxcorr_threshold=0.96, min_variance=2.0, subpixel_step=0.1, consistency=True, max_lr_diff=1)
    cfg = Config(**kw)
    host = [synth.make_stacks(33, 1024, 512, np.uint8, seed=31, frame=f, row0=200, rows=160)[:2] for f in range(5)]
    frames = [(_cuda(l), _cuda(r)) for l, r in host]
    single = [handle.match(l, r, cfg) for l, r in frames]
    torch.cuda.synchronize()
    for rep in range(3):
        outs = handle.match_batch(frames, cfg)
        assert lb.last_search_kernel() == "mma3<K=4,nodupes=0,ct=2,onepass=1>"
        # stream-ordered: consuming the results on the current stream needs no synchronisation of our own
        for (d, c), (sd, sc) in zip(outs, single):
            assert torch.equal(torch.nan_to_num(d, nan=-9.0), torch.nan_to_num(sd, nan=-9.0))
            assert torch.equal(torch.nan_to_num(c, nan=-9.0), torch.nan_to_num(sc, nan=-9.0))
    for f in (0, 4):
        want_d, want_c = oracles.port.match(host[f][0], host[f][1], **kw)
        assert _same(outs[f][0].cpu().numpy(), want_d) and _same(outs[f][1].cpu().numpy(), want_c)
    # reused outputs, no threshold (int16, no corrmap), odd batch of one
    cfg_i = Config(nxcorr_threshold=None)
    one = handle.match_batch(frames[:1], cfg_i)
    assert one[0][1] is None and _same(one[0][0].cpu().numpy(), oracles.port.match(host[0][0], host[0][1], nxcorr_threshold=None)[0])
    outs2 = handle.match_batch(frames, cfg, outs=outs)
    assert outs2[0][0] is outs[0][0]
    # overlap switched off: the same frames one after the other on the caller's stream, same bits
    handle.set_overlap(False)
    try:
        outs3 = handle.match_batch(frames, cfg)
    finally:
        handle.set_overlap(True)
    for (d, c), (sd, sc) in zip(outs3, single):
        assert torch.equal(torch.nan_to_num(d, nan=-9.0), torch.nan_to_num(sd, nan=-9.0))
        assert torch.equal(torch.nan_to_num(c, nan=-9.0), torch.nan_to_num(sc, nan=-9.0))
    with pytest.raises(lb.BicosError, match="agree"):
        handle.match_batch([frames[0], (frames[1][0][:, :100].contiguous(), frames[1][1][:, :100].contiguous())], cfg)


@pytest.mark.parametrize("n,dtype,full,rows,cols,kw", [
    (33, np.uint8, False, 7, 300, dict(nxcorr_threshold=0.9, subpixel_step=0.25, consistency=True, max_lr_diff=1, no_dupes=True)),
    (33, np.uint8, False, 150, 513, dict(nxcorr_threshold=0.9, subpixel_step=0.5, consistency=True)),  # one-pass search, ragged tiles
    (64, np.uint8, False, 150, 300, dict(nxcorr_threshold=0.9)),  # search_mma2, 256 bits
    (16, np.uint16, True, 5, 131, dict(nxcorr_threshold=0.9, double=True, min_variance=1.0)),
    (9, np.uint8, False, 3, 1, dict(nxcorr_threshold=None)),  # 32-bit descriptors: popcount engine
    (20, np.uint16, True, 4, 129, dict(nxcorr_threshold=0.8, wide_descriptors=True, consistency=True)),  # 12 words, variant 1
])
def test_kernels_write_only_their_buffers(handle, n, dtype, full, rows, cols, kw):
    """Our own memcheck for stores (compute-sanitizer is closed on this GPU pool): descriptors, the four key arrays,
    disparity and corrmap sit inside one allocation each, surrounded by guard words; after the three stages and after
    the whole match every guard word is intact and the interior is completely written. Stage entry points through the
    C ABI with interior pointers."""
    import ctypes

    import torch

    from libbicos_b200 import capi

    L = lb.lib()
    cfg = Config(mode_full=full, **kw)
    ccfg = cfg.to_c()
    left, right, _ = synth.make_stacks(n, 64, max(cols, 16), dtype, seed=n + cols, rows=rows)
    l, r = _cuda(np.ascontiguousarray(left[:, :, :cols])), _cuda(np.ascontiguousarray(right[:, :, :cols]))
    p0, _, _, _, pitch, depth = handle._stack_info(l)
    p1 = handle._stack_info(r)[0]
    k = lb.descriptor_words(n, full, cfg.wide_descriptors)
    pw = (cols * k + 3) // 4 * 4
    GUARD, MARK = 1024, 0x5A5A5A5A  # int32 words

    def guarded(words):
        buf = torch.full((GUARD + words + GUARD,), MARK, dtype=torch.int32, device="cuda")
        return buf, buf.data_ptr() + 4 * GUARD

    def intact(buf, words, what, filled=True):
        assert bool((buf[:GUARD] == MARK).all()) and bool((buf[GUARD + words:] == MARK).all()), f"{what}: guard words overwritten"
        if filled:
            assert int((buf[GUARD : GUARD + words] == MARK).sum()) == 0, f"{what}: interior not completely written"

    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    mode = int(full) | (capi.MODE_WIDE if cfg.wide_descriptors else 0)
    px = rows * cols
    for engine in ("auto", "popc"):
        lb.set_search_engine(engine)
        try:
            d = [guarded(rows * pw) for _ in range(2)]
            for planes, (buf, ptr) in zip((p0, p1), d):
                capi._check(L.bicos_b200_transform(handle._h, planes, n, rows, cols, pitch, depth, mode, ptr, pw, st))
            keys = [guarded(px) for _ in range(4)]
            flags = cfg.flags
            ptrs = [keys[0][1], keys[1][1] if flags & 1 else None, keys[2][1] if flags & 2 else None, keys[3][1] if flags == 3 else None]
            capi._check(L.bicos_b200_search(handle._h, d[0][1], d[1][1], k, rows, cols, pw, flags | capi.FLAG_TOP2_BITS_FREE, *ptrs, st))  # as bicos_b200_match: the transform's output
            disp_words = px if cfg.nxcorr_threshold is not None else (px + 1) // 2
            corr_words = px * (2 if cfg.double else 1)
            raw, disp, corr = guarded((px + 1) // 2), guarded(disp_words), guarded(corr_words)
            disp_pitch = cols * (4 if cfg.nxcorr_threshold is not None else 2)
            capi._check(L.bicos_b200_refine(handle._h, p0, p1, n, rows, cols, pitch, depth, ctypes.byref(ccfg), *ptrs, raw[1],
                                            disp[1], disp_pitch, corr[1] if cfg.nxcorr_threshold is not None else None,
                                            cols * (8 if cfg.double else 4), st))
            torch.cuda.synchronize()
            odd = px % 2 == 1  # the last int16 of an odd image shares its word with the guard pattern
            for (buf, _), what in zip(d, ("desc0", "desc1")):
                intact(buf, rows * pw, what, filled=pw == cols * k)
            for (buf, _), ptr, what in zip(keys, ptrs, ("fwd_first", "fwd_last", "rev_first", "rev_last")):
                intact(buf, px, what, filled=ptr is not None)
            intact(raw[0], (px + 1) // 2, "raw disparity", filled=not odd)
            intact(disp[0], disp_words, "disparity", filled=cfg.nxcorr_threshold is not None or not odd)
            intact(corr[0], corr_words, "corrmap", filled=cfg.nxcorr_threshold is not None)
            # the whole path into fresh guarded outputs
            disp2, corr2 = guarded(disp_words), guarded(corr_words)
            capi._check(L.bicos_b200_match(handle._h, p0, p1, n, rows, cols, pitch, depth, ctypes.byref(ccfg), disp2[1], disp_pitch,
                                           corr2[1] if cfg.nxcorr_threshold is not None else None, cols * (8 if cfg.double else 4), st))
            torch.cuda.synchronize()
            intact(disp2[0], disp_words, "match disparity", filled=cfg.nxcorr_threshold is not None or not odd)
            intact(corr2[0], corr_words, "match corrmap", filled=cfg.nxcorr_threshold is not None)
            assert torch.equal(disp2[0], disp[0]) and torch.equal(corr2[0], corr[0])
        finally:
            lb.set_search_engine("auto")


def test_out_buffers_are_validated(handle):
    """Caller-supplied output buffers of the wrong type, shape, device or layout are refused before any kernel
    or copy can write past them (the C ABI takes plain pointers and trusts them)."""
    import torch

    left, right, _ = synth.make_stacks(9, 32, 64, np.uint8, seed=3)
    l, r = _cuda(left), _cuda(right)
    thr, nothr = Config(nxcorr_threshold=0.5), Config(nxcorr_threshold=None)
    f32 = lambda *shape: torch.empty(shape, dtype=torch.float32, device="cuda")  # noqa: E731
    i16 = torch.empty((32, 64), dtype=torch.int16, device="cuda")
    handle.match(l, r, thr, out=(f32(32, 64), f32(32, 64)))
    handle.match(l, r, nothr, out=(i16, None))
    for cfg, out in ((thr, (i16, f32(32, 64))),  # int16 disparity buffer with a thresholded (float32) configuration
                     (thr, (f32(32, 64), None)),  # threshold set but no corrmap buffer
                     (thr, (f32(32, 64), torch.empty((32, 64), dtype=torch.float64, device="cuda"))),  # float64 corrmap, SINGLE
                     (Config(nxcorr_threshold=0.5, double=True), (f32(32, 64), f32(32, 64))),  # float32 corrmap, DOUBLE
                     (thr, (f32(16, 64), f32(32, 64))),  # too small
                     (thr, (f32(64, 32).t(), f32(32, 64))),  # transposed view
                     (thr, (torch.empty((32, 64), dtype=torch.float32), f32(32, 64))),  # host tensor
                     (nothr, (i16, f32(32, 64)))):  # corrmap without a threshold
        with pytest.raises(lb.BicosError, match="out "):
            handle.match(l, r, cfg, out=out)
    good = (np.empty((32, 64), np.float32), np.empty((32, 64), np.float32))
    handle.match_host(left, right, thr, out=good)
    for out in ((np.empty((32, 64), np.int16), good[1]), (good[0], None), (np.empty((64, 32), np.float32).T, good[1]),
                (np.empty((32, 32), np.float32), good[1])):
        with pytest.raises(lb.BicosError, match="out "):
            handle.match_host(left, right, thr, out=out)


def test_matches_on_different_streams_share_the_workspace_safely(handle, oracles):
    """Two matches enqueued back to back on different streams through one handle: the second waits on the device
    for the first (it reuses the descriptor and key buffers), so both results are right."""
    import torch

    kw = dict(nxcorr_threshold=0.9, subpixel_step=0.2, consistency=True, max_lr_diff=1)
    a = synth.make_stacks(33, 160, 512, np.uint8, seed=21)[:2]
    b = synth.make_stacks(33, 160, 512, np.uint8, seed=22)[:2]
    want = [oracles.port.match(l, r, **kw) for l, r in (a, b)]
    dev = [(_cuda(l), _cuda(r)) for l, r in (a, b)]
    torch.cuda.synchronize()
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    for rep in range(3):
        got = []
        for (l, r), st in zip(dev, streams):
            with torch.cuda.stream(st):
                got.append(handle.match(l, r, Config(**kw)))
        torch.cuda.synchronize()
        for (d, c), (wd, wc) in zip(got, want):
            assert _same(d.cpu().numpy(), wd) and _same(c.cpu().numpy(), wc), rep


def test_errors(handle):
    import torch

    import libbicos_b200 as lb

    one = torch.zeros((1, 8, 8), dtype=torch.uint8, device="cuda")
    with pytest.raises(lb.BicosError, match="at least two"):
        handle.match(one, one, Config())
    many = torch.zeros((20, 8, 8), dtype=torch.uint8, device="cuda")
    with pytest.raises(lb.BicosError, match="363 bits"):
        handle.match(many, many, Config(mode_full=True))
    bad = torch.zeros((4, 8, 8), dtype=torch.float32, device="cuda")
    with pytest.raises(lb.BicosError, match="depths"):
        handle.match(bad, bad, Config())


# --------------------------------------------------------------------- golden vectors --
def _golden():
    import importlib.util
    import os

    here = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    spec = importlib.util.spec_from_file_location("make_golden", os.path.join(here, "make_golden.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod, here


@pytest.mark.parametrize("name", sorted(_golden()[0].CASES))
def test_gpu_matches_golden_reference_outputs(handle, name):
    """Every stage against fixtures produced by the unmodified reference (no oracle at run time)."""
    import os

    mg, here = _golden()
    case = mg.CASES[name]
    kw = case[7]
    left, right = mg.inputs(case)
    g = np.load(os.path.join(here, name + ".npz"))
    assert int(g["input_crc"]) == mg.crc(left, right)
    cols = left.shape[2]
    cfg = Config(**kw)
    l, r = _cuda(left), _cuda(right)
    d0, k = handle.transform(l, cfg.mode_full, cfg.wide_descriptors)
    d1, _ = handle.transform(r, cfg.mode_full, cfg.wide_descriptors)
    assert np.array_equal(_words(d0, k, cols), g["desc0"]) and np.array_equal(_words(d1, k, cols), g["desc1"])
    keys = handle.search(d0, d1, k, cols, cfg.flags)
    disp, corr, raw = handle.refine(l, r, cfg, keys)
    assert np.array_equal(raw.cpu().numpy(), g["raw"])
    assert _same(disp.cpu().numpy(), g["disp"])
    if corr is not None:
        assert _same(corr.cpu().numpy(), g["corr"])
    disp2, corr2 = handle.match(l, r, cfg)
    assert _same(disp2.cpu().numpy(), g["disp"])


def test_pybicos_drop_in(handle, oracles):
    """pybicos.match (host numpy lists -> BICOS_Match -> kernels) equals the oracle."""
    from libbicos_b200 import pybicos

    left, right, _ = synth.make_stacks(33, 512, 200, np.uint8, seed=77, row0=100, rows=40)
    cfg = pybicos.Config()
    cfg.nxcorr_threshold = 0.96
    cfg.min_variance = 2.0
    cfg.subpixel_step = 0.1
    cfg.set_consistency(1, False)
    disp, corr = pybicos.match(list(left), list(right), cfg)
    want_d, want_c = oracles.port.match(left, right, nxcorr_threshold=0.96, min_variance=2.0, subpixel_step=0.1,
                                        consistency=True, max_lr_diff=1)
    assert _same(disp, want_d) and _same(corr, want_c)
    cfg.precision = pybicos.Precision.DOUBLE
    disp, corr = pybicos.match(list(left), list(right), cfg)
    assert corr.dtype == np.float64 and disp.dtype == np.float32
    cfg.nxcorr_threshold = -1.0  # unset: int16 result, no corrmap
    disp, corr = pybicos.match(list(left), list(right), cfg)
    assert disp.dtype == np.int16 and corr is None
    with pytest.raises(RuntimeError, match="at least two"):
        pybicos.match([left[0]], [right[0]], cfg)


def test_full_size_properties(handle):
    """BASELINE sizes, where the oracle is too slow: size-independent properties of the path."""
    import torch

    n, rows, cols = 33, 1536, 2048
    l, r, dtrue = synth.make_stacks(n, rows, cols, np.uint8, xp=torch, device="cuda", bands=False)
    cfg = Config(nxcorr_threshold=0.96, min_variance=2.0, subpixel_step=0.1, consistency=True, max_lr_diff=1)
    disp, corr = handle.match(l, r, cfg)
    valid = ~torch.isnan(disp)
    assert valid.float().mean().item() > 0.8
    err = (disp - dtrue)[valid].abs()
    assert (err <= 0.5).float().mean().item() > 0.99  # recovers the planted disparity
    assert torch.equal(torch.isnan(corr), torch.isnan(corr) & ~valid | torch.isnan(corr))  # corr defined where valid
    assert (corr[valid] >= 0.96).all()
    # idempotence / determinism: same inputs, same bits (atomics only take minima)
    disp2, corr2 = handle.match(l, r, cfg)
    assert torch.equal(torch.nan_to_num(disp, nan=-9.0), torch.nan_to_num(disp2, nan=-9.0))
    assert torch.equal(torch.nan_to_num(corr, nan=-9.0), torch.nan_to_num(corr2, nan=-9.0))
    # a match of this size runs as three row bands through the two-stream pipeline: same bits as one unit on one stream
    handle.set_overlap(False)
    try:
        disp3, corr3 = handle.match(l, r, cfg)
    finally:
        handle.set_overlap(True)
    assert torch.equal(torch.nan_to_num(disp, nan=-9.0), torch.nan_to_num(disp3, nan=-9.0))
    assert torch.equal(torch.nan_to_num(corr, nan=-9.0), torch.nan_to_num(corr3, nan=-9.0))
    # row independence: matching a row band alone gives exactly the rows of the full match
    sub = handle.match(l[:, 700:764].contiguous(), r[:, 700:764].contiguous(), cfg)
    assert torch.equal(torch.nan_to_num(sub[0], nan=-9.0), torch.nan_to_num(disp[700:764], nan=-9.0))
    # exchanging the stacks mirrors the geometry: the integer search is symmetric
    cfg_i = Config(nxcorr_threshold=None, consistency=True, max_lr_diff=0)
    a = handle.match(l[:, :64].contiguous(), r[:, :64].contiguous(), cfg_i)[0]
    b = handle.match(r[:, :64].contiguous(), l[:, :64].contiguous(), cfg_i)[0]
    va = a != -32768
    cols_idx = torch.arange(cols, device="cuda").expand(64, cols)
    tgt = (cols_idx - a.long())[va]  # matched right column of every consistent left pixel
    rows_idx = torch.arange(64, device="cuda").unsqueeze(1).expand(64, cols)[va]
    assert (b[rows_idx, tgt] == -a[va]).all()  # with max_lr_diff=0 the match is mutual, disparity negated
