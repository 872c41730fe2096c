"""CPU: pin the oracle restatement (oracle/gccnmf_oracle.py) to fixtures produced by the
unmodified reference (oracle/make_golden.py).  Library arithmetic is the same numpy/scipy, so
float results are expected bit-identical; tolerances are stated where they are not zero."""
import hashlib

import numpy as np
import pytest

from oracle import gccnmf_oracle as orc


def eq(a, b):
    assert a.shape == b.shape and a.dtype == b.dtype, (a.shape, b.shape, a.dtype, b.dtype)
    np.testing.assert_array_equal(a, b)


def eq_digest(a, digest):
    """Bit-exact comparison with an array stored as its SHA-256 (oracle/make_golden.py:array_digest) to keep the fixture small."""
    a = np.ascontiguousarray(a)
    assert hashlib.sha256(('%s %s ' % (a.dtype.str, a.shape)).encode() + a.tobytes()).hexdigest() == str(digest), (a.dtype, a.shape)


def test_separation_flow_bit_exact(golden):
    g = golden('separation_mini')
    sr, N, hop, D, S, K, I = [int(v) for v in g['params']]
    r = orc.runSeparation(g['samples'], sr, N, hop, D, float(g['micSep']), S, K, I)
    eq(r['X'], g['X'])
    eq(r['V'], g['V'])
    eq(r['W'], g['W'])
    eq(r['H'], g['H'])
    eq(r['coherence'], g['coherence'])
    eq(r['angularSpectrogram'], g['angularSpectrogram'])
    assert list(r['targetTDOAIndexes']) == list(g['targetTDOAIndexes'])
    eq(r['targetTDOAGCCNMFs'], g['targetTDOAGCCNMFs'])
    eq(r['targetCoefficientMasks'], g['targetCoefficientMasks'])
    eq(r['targetSpectrogramEstimates'], g['targetSpectrogramEstimates'])
    eq(r['targetSignalEstimates'], g['targetSignalEstimates'])


def test_klnmf_init_and_single_iteration(golden):
    g = golden('separation_mini')
    K = int(g['params'][5])
    W0, H0 = orc.initKLNMF(g['V'].shape[0], g['V'].shape[1], K)
    eq(W0, g['W0'])
    eq(H0, g['H0'])
    W1, H1 = orc.performKLNMF(g['V'], K, 1, 0, W0=g['W0'], H0=g['H0'])
    eq(W1, g['W1'])
    eq(H1, g['H1'])
    W3, H3 = orc.performKLNMF(g['V'], K, 3, 0.5)
    eq(W3, g['W3_alpha'])
    eq(H3, g['H3_alpha'])


def test_angular_spectrogram_fast_form_matches(golden):
    g = golden('separation_mini')
    sr, N, hop, D = [int(v) for v in g['params'][:4]]
    f = np.linspace(0, sr / 2.0, N // 2 + 1)
    A = orc.getAngularSpectrogramFast(g['coherence'], f, float(g['micSep']), D)
    np.testing.assert_allclose(A, g['angularSpectrogram'], rtol=0, atol=1e-10)   # float64 reduction order only


def test_enhancement_flow(golden):
    g = golden('enhancement_mini')
    sr, N, hop, D, S, K, I = [int(v) for v in g['params']]
    r = orc.runEnhancement(g['samples'], sr, N, hop, D, float(g['micSep']), K, I)
    eq(r['X'], g['X'])
    eq(r['W'], g['W'])
    eq(r['H'], g['H'])
    assert list(r['targetTDOAIndexes']) == list(g['targetTDOAIndexes'])
    E = orc.getExpJOmegaTau(r['frequenciesInHz'], orc.getTDOAsInSeconds(float(g['micSep']), D))
    eq(orc.getGCCNMFAllTDOAs(r['coherence'], E, r['W']), g['gccNMF'])
    eq(r['argMaxGCCNMF'], g['argMaxGCCNMF'])
    eq(r['targetCoefficientMasks'], g['targetCoefficientMasks'])
    eq_digest(r['targetSpectrogramEstimates'], g['targetSpectrogramEstimates_sha256'])
    eq(r['targetSignalEstimates'], g['targetSignalEstimates'])


def test_online_loop(golden):
    g = golden('online_mini')
    sr, N, hop, D, K = [int(v) for v in g['params']]
    r = orc.performOnlineSpeechEnhancement(g['samples'], sr, g['W'], np.hanning(N), N, hop, D, float(g['micSep']),
                                           0.05 * D, gainPerFrame=True)
    eq(r['targetTDOAs'], g['targetTDOAs'])
    eq(r['atomMasks'], g['atomMasks'])
    eq(r['angularSpectrogram'], g['angularSpectrogram'])
    eq(r['wienerFilters'], g['wienerFilters'])
    eq(r['output'], g['output'])


def test_low_latency_loop_and_windows(golden):
    g = golden('lowlatency_mini')
    sr, N, hop, D, K, synth = [int(v) for v in g['params']]
    eq(orc.getAsymmetricAnalysisWindow(N, synth // 2, 0), g['analysisWindow'])
    eq(orc.getAsymmetricSynthesisWindow(N, synth // 2, 0), g['synthesisWindow'])
    for tag, win in (('sym', g['symmetricWindow']), ('asym', g['analysisWindow'])):
        r = orc.performOnlineSpeechEnhancement(g['samples'], sr, g['W'], win, N, hop, D, float(g['micSep']),
                                               0.05 * D, gainPerFrame=False)
        eq(r['targetTDOAs'], g[tag + '_targetTDOAs'])
        eq(r['atomMasks'], g[tag + '_atomMasks'])
        eq(r['wienerFilters'], g[tag + '_wienerFilters'])
        eq(r['output'], g[tag + '_output'])


def test_pretraining_float64_input(golden):
    g = golden('pretraining_mini')
    W, H = orc.performKLNMF(g['trainV'], 12, 20, 0, 1e-16, 0)
    eq(W, g['W'])
    eq(H, g['H'])
    eq(orc.getOrderedDictionary(W), g['orderedW'])


def test_stft_istft_edge_cases():
    with pytest.raises(ValueError):
        orc.stft(np.zeros(100, np.float32), 256, 64)
    x = np.random.default_rng(0).standard_normal(256).astype(np.float32)
    X = orc.stft(x, 256, 64)                       # exactly one frame
    assert X.shape == (129, 1) and X.dtype == np.complex64
    y = orc.istft(X, 64, 256)
    assert y.shape == (0,) and y.dtype == np.float32   # center trim removes the whole single frame


def test_realtime_processor_and_overlap_add_ring(golden):
    """a13 / f-2: the restatements against the UNMODIFIED reference classes run over the numpy stand-in for Theano
    (oracle/theano_numpy_shim.py, oracle/make_golden.py:golden_realtime): outputs, atom masks, per-atom TDOA argmax and
    localisation decisions bit for bit, for both mask modes and 1 / 4 frames per chunk, then the overlap-add ring around it."""
    g = golden('realtime_mini')
    sr, N, K, D = [int(v) for v in g['params']]
    assert list(g['modes']) == [orc.TARGET_MODE_BOXCAR, orc.TARGET_MODE_WINDOW_FUNCTION]
    for tag, nT, mode in (('w1', 1, orc.TARGET_MODE_WINDOW_FUNCTION), ('b4', 4, orc.TARGET_MODE_BOXCAR), ('w4', 4, orc.TARGET_MODE_WINDOW_FUNCTION)):
        p = orc.GCCNMFProcessorOracle(sr, N, nT, g['W'], D, float(g['micSep']), localizationEnabled=True, localizationWindowSize=6)
        p.targetMode = mode
        p.setTargetTDOARange(*g['targetRange'])
        for i in range(g[tag + '_frames'].shape[0]):
            y = p.processFrames(g[tag + '_frames'][i])
            eq(y, g[tag + '_y'][i])
            eq(p.lastHMask, g[tag + '_hmask'][i])
            eq(p.lastArgmax.astype(np.int32), g[tag + '_argmax'][i])
            assert float(p.targetTDOAIndex) == g[tag + '_target'][i]
    hop, B, nT = [int(v) for v in g['ola_params']]
    p = orc.GCCNMFProcessorOracle(sr, N, nT, g['W'], D, float(g['micSep']), localizationEnabled=True, localizationWindowSize=6)
    p.setTargetTDOARange(9.60, 5.0, 2.0, 0.0)
    ring = orc.OverlapAddProcessorOracle(2, N, hop, B, nT)
    x = g['ola_x']
    for b in range(x.shape[1] // B):
        out = ring.processFrames(x[:, b * B:(b + 1) * B].copy(), p.processFrames)
        eq(out, g['ola_out'][:, b * B:(b + 1) * B])
        eq(p.lastHMask, g['ola_hmask'][b])
        assert float(p.targetTDOAIndex) == g['ola_target'][b]
