"""KL-NMF at the shape edges of the tensor-core path (gcc-nmf_b200/csrc/klnmf_tma.cu on the plane GEMM of tma_gemm.cuh) against a
float64 restatement of gccNMF/gccNMFFunctions.py:76-81.

The shapes below reach the edge code of the path: SIMT tail rows shared over one to sixteen m tiles, the extra m tile that replaces
them, k tails of half a 16-deep step, an 8-atom second m tile of the atom-major contractions, an empty k-split of the W-update
numerator, and the float32 SIMT path just outside the tensor-core conditions.

CPU part (no GPU): a numpy emulation of the tensor-core arithmetic (bf16 hi / lo operand planes, the lo.hi + hi.lo + hi.hi products
accumulated exactly, float32 rounding between stages, the planner's k-splits and row-sum slots) stays inside the error bars at every
shape, and each of five deliberate kernel mistakes falls outside them -- so the bars can tell a subtly wrong kernel from rounding.
GPU part: the fused loop, the fixed-dictionary loop, the staged API and the tile-width switches against the same float64 reference
and the same bars, with the workspace filled with NaN bytes before every run."""
import ctypes
import functools

import numpy as np
import pytest

from oracle import gccnmf_oracle as orc

B200_SMS = 148
KB = 32                 # k-block of the plane GEMM (tma_gemm_host.cuh kKB)
TAIL_ROWS_MAX = 8       # tma_gemm_host.cuh kTailRowsMax

# Error bars (float32 result against float64 reference), relative:
#   one iteration:                    element-wise max over every entry, and Frobenius
#   several iterations (alpha = 1):   Frobenius, and element-wise over entries >= 1e-4 x the largest
BAR1_ELEM, BAR1_FRO = 3e-5, 1e-5
BARN_ELEM, BARN_FRO, BARN_FLOOR = 1e-4, 3e-5, 1e-4

# (F, T2, K), whether the tensor-core path takes it, and the rows past the last full 128-row tile of the W.H contractions (G1 / G3)
# at the planned tile width: 'none', 'simt' (2..8 tail rows computed in float32 SIMT by the epilogue warps) or 'tile' (an extra,
# partly out-of-bounds m tile).
SHAPES = [
    ((128, 128, 32), True, 'none'),       # lower bound of every tensor-core condition; one tile per contraction
    ((130, 130, 40), True, 'simt'),       # 2 tail rows; Fp pad of 6; K = 32 + 8 (half a 16-step); 2-element F and T2 tails
    ((136, 258, 56), True, 'simt'),       # tail = kTailRowsMax; wh_tile = 256 turns it into an extra tile (test_switches)
    ((137, 200, 48), True, 'tile'),       # 9 tail rows: extra m tile with 119 out-of-bounds rows
    ((392, 330, 136), True, 'simt'),      # tail columns over 3 m tiles; K = 128 + 8: an 8-atom m tile, 2 active lanes of a W-update CTA
    ((255, 640, 200), True, 'tile'),      # F % 8 != 0, 127-row extra tile; K % 128 = 72
    ((513, 1040, 128), True, 'simt'),     # empty k-split of the W-update numerator (test_planner_branches)
    ((2049, 256, 32), True, 'simt'),      # 16 m tiles share the tail columns; minimum K
    ((127, 300, 64), False, None),        # F < 128
    ((300, 127, 64), False, None),        # T2 < 128
    ((300, 300, 36), False, None),        # K % 8 != 0
    ((300, 300, 24), False, None),        # K < 32
]
TC_SHAPES = [s for s, tc, _ in SHAPES if tc]
SWITCH_SHAPES = [(136, 258, 56), (392, 330, 136), (513, 1040, 128)]


def _id(shape):
    return 'x'.join(str(v) for v in shape)


# ------------------------------------------------------------------------------------------------ inputs and float64 references
@functools.lru_cache(maxsize=None)
def _inputs(shape):
    F, T2, K = shape
    rng = np.random.default_rng(F * 100003 + T2 * 101 + K)
    V = (rng.random((F, T2)) ** 3 + 1e-3).astype(np.float32)
    W0, H0 = orc.initKLNMF(F, T2, K)
    return V, W0, H0


@functools.lru_cache(maxsize=None)
def _reference(shape, iterations, alpha):
    """gccNMFFunctions.py:76-81 (oracle.klnmfIteration) on float64 copies of V, W0, H0."""
    V, W0, H0 = (a.astype(np.float64) for a in _inputs(shape))
    W, H = W0.copy(), H0.copy()
    for _ in range(iterations):
        orc.klnmfIteration(V, W, H, alpha)
    return W, H


def _reference_fixed(V, W, H0, iterations, alpha, epsilon=1e-16):
    """:76 repeated with a fixed dictionary, float64: H *= W^T (V / (W H)) / (colsum(W) + alpha + eps) -- the denominator of
    oracle.inferCoefficientsKLNMF, from a caller-given H0."""
    V, W, H = V.astype(np.float64), W.astype(np.float64), H0.astype(np.float64).copy()
    denom = W.sum(0)[:, None] + alpha + epsilon
    for _ in range(iterations):
        H *= (W.T @ (V / (W @ H))) / denom
    return H


def _errors(x, ref, floor=0.0):
    """(element-wise max relative error over the entries >= floor * max |ref|, Frobenius relative error); inf if x is not finite."""
    x = np.asarray(x, np.float64)
    if not np.isfinite(x).all():
        return float('inf'), float('inf')
    a = np.abs(ref)
    sel = a >= floor * a.max()
    elem = float((np.abs(x - ref)[sel] / a[sel]).max())
    return elem, float(np.linalg.norm(x - ref) / np.linalg.norm(ref))


def _within(W, H, Wr, Hr, iterations):
    """Worst (element-wise, Frobenius) of W and H and whether they meet the bar of this iteration count."""
    floor, be, bf = (0.0, BAR1_ELEM, BAR1_FRO) if iterations == 1 else (BARN_FLOOR, BARN_ELEM, BARN_FRO)
    eW, eH = _errors(W, Wr, floor), _errors(H, Hr, floor)
    elem, fro = max(eW[0], eH[0]), max(eW[1], eH[1])
    return elem, fro, elem <= be and fro <= bf


# ------------------------------------------------------------------------------------------------ tile plan (host logic of the library)
@functools.lru_cache(maxsize=None)
def _plan(shape, sm_count=B200_SMS):
    """gccnmf_klnmf_tile_plan: tile widths of G1 / G3 and G2, tile width and k-splits of G4, row-sum slots; None off the tensor-core path."""
    from gcc_nmf_b200 import _lib
    out = (ctypes.c_int * 8)()
    if _lib.load_library().gccnmf_klnmf_tile_plan(sm_count, *shape, out) != 0:
        return None
    return dict(bn_wh=out[0], bn_h=out[1], bn_w=out[2], splits=out[3], slots=out[4])


def _wh_rows(F, bn):
    """Which rows past the last full 128-row tile G1 / G3 compute, and how (launch_plane_gemm in tma_gemm_host.cuh)."""
    tail = F % 128
    if tail == 0:
        return 'none'
    return 'simt' if tail <= TAIL_ROWS_MAX and F > 128 and (F // 128) * 128 >= bn else 'tile'


def _split_ranges(T2, splits):
    """Frame ranges of the k-splits of G4 (kblocks_per_split = ceil(k-blocks / splits)); an empty split has an empty range."""
    total_kb = (T2 + KB - 1) // KB
    per = (total_kb + splits - 1) // splits
    return [(min(T2, z * per * KB), min(T2, (z + 1) * per * KB)) for z in range(splits)]


# ------------------------------------------------------------------------------------------------ emulation of the tensor-core arithmetic
def _bf16(x):
    """Round-to-nearest-even float32 -> bfloat16, as float32 (cvt.rn.bf16.f32)."""
    u = np.asarray(x, np.float32).view(np.uint32).astype(np.uint64)
    u = (u + 0x7FFF + ((u >> 16) & 1)) & 0xFFFF0000
    return u.astype(np.uint32).view(np.float32)


def _planes(x):
    hi = _bf16(x)
    return hi.astype(np.float64), _bf16(np.asarray(x, np.float32) - hi).astype(np.float64)


def _mm(a, b):
    """a . b as the plane GEMM forms it: lo.hi + hi.lo + hi.hi of the bf16 planes, accumulated exactly, rounded to float32 once."""
    ah, al = _planes(a)
    bh, bl = _planes(b)
    return ((ah + al) @ (bh + bl) - al @ bl).astype(np.float32)


MUTATIONS = ('tail_row', 'k_tail', 'split', 'rowsum_slot', 'unit_norm')


def _emulate(shape, iterations, alpha, mutation=None, epsilon=1e-16):
    """The tensor-core loop in numpy, in its (U, G) gauge (klnmf_tma.cu header), with one optional deliberate mistake:
    tail_row     the last row of V / (W H) is zeroed (a tail row left unwritten)
    k_tail       W H drops the last 8 atoms (the half 16-deep step of a K tail not issued)
    split        the first k-split slab of the W-update numerator is dropped
    rowsum_slot  the last row-sum slot of G is missing
    unit_norm    c = 1 instead of ||U[:, k]|| in the c (alpha + eps) term of the H update."""
    V, W0, H0 = _inputs(shape)
    F, T2, K = shape
    plan = _plan(shape) or dict(splits=1, slots=1, bn_h=T2)
    U, G = W0.copy(), H0.copy()
    c = np.ones(K, np.float32)
    kk = K - 8 if mutation == 'k_tail' else K

    def ratio():
        R = V / _mm(U[:, :kk], G[:kk])
        if mutation == 'tail_row':
            R[-1] = 0
        return R

    for _ in range(iterations):
        R = ratio()
        denom = U.sum(0, dtype=np.float32) + c * np.float32(alpha + epsilon)
        G = G * (_mm(U.T, R) * (np.float32(1) / denom)[:, None])
        R = ratio()
        numer = np.zeros((F, K), np.float32)
        for z, (t0, t1) in enumerate(_split_ranges(T2, plan['splits'])):
            if t1 > t0 and not (mutation == 'split' and z == 0):
                numer += _mm(R[:, t0:t1], G[:, t0:t1].T)
        slots = [G[:, s * plan['bn_h']:(s + 1) * plan['bn_h']].sum(1, dtype=np.float32) for s in range(plan['slots'])]
        if mutation == 'rowsum_slot':
            slots = slots[:-1]
        rowsum = np.sum(slots, 0, dtype=np.float32) if slots else np.zeros(K, np.float32)
        with np.errstate(divide='ignore', invalid='ignore'):
            U = U * (numer / rowsum)
        if mutation != 'unit_norm':
            c = np.sqrt((U * U).sum(0, dtype=np.float32))
    with np.errstate(divide='ignore', invalid='ignore'):
        norms = np.sqrt((U * U).sum(0, dtype=np.float32))
        return U / norms, G * norms[:, None]


# ------------------------------------------------------------------------------------------------ CPU tests
@pytest.fixture(scope='module')
def built():
    import __graft_entry__ as entry
    entry.build()


def test_planner_branches(built):
    """Each shape reaches the edge it is listed for, by the planner's arithmetic for a 148-SM B200."""
    for shape, tc, rows in SHAPES:
        F, T2, K = shape
        p = _plan(shape)
        assert (p is not None) == tc, shape
        if not tc:
            continue
        assert _wh_rows(F, p['bn_wh']) == rows, (shape, p)
    assert [_wh_rows(136, bn) for bn in (104, 112, 128, 256)] == ['simt'] * 3 + ['tile']
    # (392, 330, 136): tail columns of an n tile shared by 3 m tiles; (2049, 256, 32): by 16
    assert 392 // 128 == 3 and 2049 // 128 == 16
    # (513, 1040, 128): G4 contracts over 1040 frames = 33 k-blocks; with 8 splits of ceil(33 / 8) = 5 blocks split 7 starts at
    # block 35 and is empty -- at every tile width, since 148 SMs / (1 m tile x <= 5 n tiles) >= 8 and 33 // 4 >= 8 give 8 splits
    p = _plan((513, 1040, 128))
    assert p['splits'] == 8 and _split_ranges(1040, 8)[7] == (1040, 1040), p


@pytest.mark.parametrize('shape', [s for s, _, _ in SHAPES], ids=_id)
def test_emulation_within_bars(built, shape):
    """The emulated tensor-core arithmetic meets the bars: ~1.5-3e-6 after one iteration, <= ~5e-6 after four."""
    for iterations, alpha in ((1, 0.0), (4, 1.0)):
        W, H = _emulate(shape, iterations, alpha)
        elem, fro, ok = _within(W, H, *_reference(shape, iterations, alpha), iterations)
        assert ok, (shape, iterations, elem, fro)


@pytest.mark.parametrize('mutation', MUTATIONS)
def test_mutations_break_the_bars(built, mutation):
    """Every deliberate mistake is caught by the bars at every tensor-core shape (the norm one after four iterations with alpha = 1,
    the others after one)."""
    for shape in TC_SHAPES:
        iterations, alpha = (4, 1.0) if mutation == 'unit_norm' else (1, 0.0)
        W, H = _emulate(shape, iterations, alpha, mutation)
        elem, fro, ok = _within(W, H, *_reference(shape, iterations, alpha), iterations)
        assert not ok, (mutation, shape, elem, fro)


# ------------------------------------------------------------------------------------------------ GPU tests
@pytest.fixture(scope='module')
def h():
    from gcc_nmf_b200._lib import default_handle
    hd = default_handle()
    yield hd
    for name, value in (('wh_tile', 0), ('wh_split2', 0), ('w_cluster_reduce', 1), ('force_simt_nmf', 0)):
        hd.set_option(name, value)


def _sm_count(h):
    import torch
    return torch.cuda.get_device_properties(h.device).multi_processor_count


def _poison(h, shape):
    """NaN bytes (0xFF: NaN in float32 and bf16) in the whole KL-NMF workspace: a read of anything the call did not write shows."""
    F, T2, K = shape
    h.workspace('klnmf', h.lib.gccnmf_klnmf_workspace_bytes(F, T2, K)).fill_(0xFF)


def _fused(h, shape, iterations, alpha, update_W=True, H0=None):
    import torch
    V, W0, H0_ = _inputs(shape)
    W, H = h.to_device(W0.copy()), h.to_device((H0_ if H0 is None else H0).copy())
    _poison(h, shape)
    h.klnmf(h.to_device(V), W, H, iterations, sparsity_alpha=alpha, update_W=update_W)
    torch.cuda.synchronize()
    return W.cpu().numpy(), H.cpu().numpy()


def _staged(h, shape, iterations, alpha):
    import torch
    V, W0, H0 = _inputs(shape)
    F, T2, K = shape
    Vd, W, H = h.to_device(V), h.to_device(W0.copy()), h.to_device(H0.copy())
    numer = torch.full((F * K + K,), float('nan'), device=h.device)
    _poison(h, shape)
    h.klnmf_begin(Vd, W, H)
    for it in range(iterations):
        h.klnmf_step_numer(Vd, W, H, it, numer, sparsity_alpha=alpha)
        h.klnmf_step_apply(W, H, numer)
    h.klnmf_end(W, H, iterations)
    torch.cuda.synchronize()
    return W.cpu().numpy(), H.cpu().numpy()


def _check_dispatch(h, shape, tc):
    assert h.klnmf_uses_tensor_cores(*shape) == tc, shape
    if tc:
        assert _plan(shape, _sm_count(h)) == _plan(shape), 'the planned branches assume a 148-SM B200'


def _assert_bar(label, W, H, Wr, Hr, iterations):
    elem, fro, ok = _within(W, H, Wr, Hr, iterations)
    print('%s: element-wise %.2e, Frobenius %.2e' % (label, elem, fro))
    assert ok, (label, elem, fro)
    return elem, fro


@pytest.mark.gpu
@pytest.mark.parametrize('shape,tc', [(s, tc) for s, tc, _ in SHAPES], ids=[_id(s) for s, _, _ in SHAPES])
def test_one_iteration(h, shape, tc):
    """One iteration from the seeded W0, H0 against float64, W and H element-wise. B200: element-wise <= 4.4e-6, Frobenius <= 1.1e-6."""
    _check_dispatch(h, shape, tc)
    W, H = _fused(h, shape, 1, 0.0)
    _assert_bar('%s 1 iteration' % _id(shape), W, H, *_reference(shape, 1, 0.0), 1)


@pytest.mark.gpu
@pytest.mark.parametrize('shape,tc', [(s, tc) for s, tc, _ in SHAPES], ids=[_id(s) for s, _, _ in SHAPES])
def test_four_iterations_sparse(h, shape, tc):
    """Four iterations with alpha = 1: the column sums and sums of squares left by the W update (c = ||U[:, k]||) and the final
    normalisation. B200: element-wise <= 6.2e-6, Frobenius <= 1.6e-6.

    The sparsity term moves H by 100x the error of the run or more, so the comparison resolves it. (It moves H by only 2.8e-4 to
    5.7e-3 Frobenius: a per-atom constant in the H denominator is mostly undone by the next W update and the normalisation, and
    only its variation across atoms survives. test_mutations_break_the_bars shows the bars catch a wrong c in that term.)"""
    _check_dispatch(h, shape, tc)
    W1, H1 = _fused(h, shape, 4, 1.0)
    _, fro = _assert_bar('%s 4 iterations alpha 1' % _id(shape), W1, H1, *_reference(shape, 4, 1.0), 4)
    W0, H0 = _fused(h, shape, 4, 0.0)
    assert _errors(H1, H0.astype(np.float64))[1] > 100 * fro


@pytest.mark.gpu
@pytest.mark.parametrize('shape,tc', [(s, tc) for s, tc, _ in SHAPES], ids=[_id(s) for s, _, _ in SHAPES])
def test_fixed_dictionary(h, shape, tc):
    """klnmf(update_W = False), the loop behind inferCoefficientsKLNMF and online inference: three H updates with colsum(W)
    computed once; the W buffer is left bit for bit as it was. B200: element-wise <= 1.7e-5, Frobenius <= 1.0e-5, both at
    2049 x 256 x 32, where colsum(W) is one float32 sum over 2049 rows (<= 7.3e-6 / 2.3e-6 at the other shapes)."""
    _check_dispatch(h, shape, tc)
    V, W0, H0 = _inputs(shape)
    W, H = _fused(h, shape, 3, 1.0, update_W=False)
    assert np.array_equal(W, W0)
    elem, fro = _errors(H, _reference_fixed(V, W0, H0, 3, 1.0), BARN_FLOOR)
    print('%s fixed dictionary: element-wise %.2e, Frobenius %.2e' % (_id(shape), elem, fro))
    assert elem <= BARN_ELEM and fro <= BARN_FRO, (elem, fro)


@pytest.mark.gpu
def test_infer_coefficients_on_tensor_cores(h):
    import gcc_nmf_b200.gccNMFFunctions as G
    shape = (392, 330, 136)
    assert h.klnmf_uses_tensor_cores(*shape)
    V, W0, _ = _inputs(shape)
    W = (W0 / np.linalg.norm(W0, axis=0)).astype(np.float32)      # a normalised dictionary, as pretraining leaves it
    np.random.seed(0)
    H0 = np.random.random((shape[2], shape[1])).astype(np.float32) + 1e-16      # the function's seeded H init
    H = G.inferCoefficientsKLNMF(V, W, 3, 0.5)
    elem, fro = _errors(H, _reference_fixed(V, W, H0, 3, 0.5), BARN_FLOOR)
    assert elem <= BARN_ELEM and fro <= BARN_FRO, (elem, fro)


@pytest.mark.gpu
@pytest.mark.parametrize('cluster_reduce', [1, 0])
@pytest.mark.parametrize('shape', TC_SHAPES, ids=_id)
def test_staged_api(h, shape, cluster_reduce):
    """klnmf_begin / step_numer / step_apply / end, the single-GPU step of the sharded run, on tensor cores: the numerator either
    comes straight out of the cluster-reduced contraction (direct) or is summed from the k-split slabs by the pack kernel.
    B200: element-wise <= 6.2e-6, Frobenius <= 1.4e-6 after 3 iterations with alpha = 1."""
    import torch
    F, T2, K = shape
    h.set_option('w_cluster_reduce', cluster_reduce)
    try:
        direct = bool(h.lib.gccnmf_klnmf_pull_supported(h.h, F, T2, K) & 2)
        # the cluster-reduced numerator needs at least 2 k-splits (and every (1, 1, splits) cluster resident, true at these sizes)
        assert direct == (cluster_reduce == 1 and _plan(shape)['splits'] >= 2), (shape, _plan(shape))
        Ws, Hs = _staged(h, shape, 3, 1.0)
        Wf, Hf = _fused(h, shape, 3, 1.0)
    finally:
        h.set_option('w_cluster_reduce', 1)
    torch.cuda.synchronize()
    _assert_bar('%s staged (%s)' % (_id(shape), 'direct' if direct else 'pack'), Ws, Hs, *_reference(shape, 3, 1.0), 3)
    # The pack kernel adds the row-sum slots one after the other; the fused W update spreads them over 8 row groups (slot s in
    # group s % 8) and adds the groups. Up to 8 slots that is the same order; with more, the orders differ and so do the last bits
    # (9 slots at 513 x 1040 x 128: element-wise 1.1e-6 after 3 iterations).
    for a, b in ((Ws, Wf), (Hs, Hf)):
        elem, fro = _errors(a, b.astype(np.float64))
        assert fro <= 1e-6 and (elem <= 1e-6 or _plan(shape)['slots'] > 8), (elem, fro)


@pytest.mark.gpu
@pytest.mark.parametrize('shape', TC_SHAPES, ids=_id)
def test_deterministic(h, shape):
    """Two runs over a NaN-filled workspace give the same bits and no NaN (no read of pad columns, unwritten slabs or slots)."""
    a = _fused(h, shape, 4, 1.0)
    b = _fused(h, shape, 4, 1.0)
    for x, y in zip(a, b):
        assert np.isfinite(x).all() and np.array_equal(x, y)


@pytest.mark.gpu
@pytest.mark.parametrize('shape', SWITCH_SHAPES, ids=_id)
def test_switches(h, shape):
    """wh_tile (tile width of the W.H contractions) and wh_split2 (their k-split-pair form) pick a code path for a production
    result: each one meets the one-iteration bar. B200: element-wise <= 3.2e-6, Frobenius <= 8.3e-7 (wh_split2 over 4 iterations
    with alpha = 1: 5.1e-6 / 1.1e-6)."""
    assert h.klnmf_uses_tensor_cores(*shape)
    ref = _reference(shape, 1, 0.0)
    try:
        for tile in (104, 112, 128, 256):
            h.set_option('wh_tile', tile)
            _assert_bar('%s wh_tile %d (%s)' % (_id(shape), tile, _wh_rows(shape[0], tile)), *_fused(h, shape, 1, 0.0), *ref, 1)
        h.set_option('wh_tile', 0)
        if shape[2] >= 128:
            h.set_option('wh_split2', 1)
            _assert_bar('%s wh_split2' % _id(shape), *_fused(h, shape, 1, 0.0), *ref, 1)
            _assert_bar('%s wh_split2 4 iterations' % _id(shape), *_fused(h, shape, 4, 1.0), *_reference(shape, 4, 1.0), 4)
    finally:
        h.set_option('wh_tile', 0)
        h.set_option('wh_split2', 0)
