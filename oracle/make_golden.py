"""Generate tests/golden/*.npz by EXECUTING THE UNMODIFIED REFERENCE in the build container.

TEST INFRASTRUCTURE ONLY (see gccnmf_oracle.py).  Run as

    python oracle/make_golden.py            # needs /root/reference (read-only mount)

Library stages come from `gccNMF.gccNMFFunctions` / `gccNMF.librosaSTFT` imported from
/root/reference; notebook-only flows (offline enhancement mask, online frame loop, asymmetric
windows) are obtained by exec()-ing the code cells of the reference's own .ipynb files, so the
arithmetic that produces every fixture is the reference's, not the oracle's.  Inputs are small
seeded synthetic clips (gcc-nmf_b200/synth.py) so that fixtures stay small and can travel to the
GPU box, where /root/reference does not exist.

Versions used are recorded inside each .npz (`versions`).
"""
import hashlib
import json
import os
import sys

import numpy as np
import scipy

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get('GCCNMF_REFERENCE', '/root/reference')
sys.path.insert(0, REF)
sys.path.insert(0, os.path.join(ROOT, 'gcc-nmf_b200'))

from synth import synthetic_stereo  # noqa: E402
import gccNMF.gccNMFFunctions as ref  # noqa: E402

OUT = os.path.join(ROOT, 'tests', 'golden')
VERSIONS = 'numpy %s scipy %s python %s reference 0b13e9e' % (np.__version__, scipy.__version__, sys.version.split()[0])


def notebook_cells(name):
    nb = json.load(open(os.path.join(REF, 'notebooks', name + '.ipynb')))
    return [''.join(c['source']) for c in nb['cells']]


def save(name, **arrays):
    arrays['versions'] = np.array(VERSIONS)
    path = os.path.join(OUT, name + '.npz')
    np.savez_compressed(path, **arrays)
    print('%-28s %8.1f KB' % (name, os.path.getsize(path) / 1024.0))


def array_digest(a):
    """SHA-256 of an array's dtype, shape and bytes (tests/test_oracle_golden.py computes the same): stands in for an array
    too large to store that a test compares bit for bit."""
    a = np.ascontiguousarray(a)
    return hashlib.sha256(('%s %s ' % (a.dtype.str, a.shape)).encode() + a.tobytes()).hexdigest()


def golden_separation():
    """gccNMF/runGCCNMF.py:36-52 order (that module itself cannot be imported: implicit-relative
    imports + matplotlib), with its hard-coded K=128/I=100 replaced by small values."""
    sr, N, hop, D, d, S, K, I = 16000, 256, 128, 32, 0.1, 2, 16, 25
    x = synthetic_stereo(0.5, seed=7)
    X = ref.computeComplexMixtureSpectrogram(x, N, hop, np.hanning)
    f = np.linspace(0, sr / 2.0, X.shape[1])
    V = np.concatenate(np.abs(X), axis=-1)
    W, H = ref.performKLNMF(V, dictionarySize=K, numIterations=I, sparsityAlpha=0)
    stereoH = np.array(np.hsplit(H, 2))
    coh = X[0] * X[1].conj() / np.abs(X[0]) / np.abs(X[1])
    A = ref.getAngularSpectrogram(coh, f, d, D)
    m = np.mean(A, axis=-1)
    idx = ref.estimateTargetTDOAIndexesFromAngularSpectrum(m, d, D, S)
    G = ref.getTargetTDOAGCCNMFs(coh, d, D, f, idx, W, stereoH)
    M = ref.getTargetCoefficientMasks(G, S)
    Sp = ref.getTargetSpectrogramEstimates(M, X, W, stereoH)
    y = ref.getTargetSignalEstimates(Sp, N, hop, np.hanning)
    # one teacher-forced KL-NMF iteration from the seeded init, and the sparsity variant
    np.random.seed(0)
    W0 = np.random.random((V.shape[0], K)).astype(np.float32) + 1e-16
    H0 = np.random.random((K, V.shape[1])).astype(np.float32) + 1e-16
    W1, H1 = ref.performKLNMF(V, K, 1, 0)
    W3s, H3s = ref.performKLNMF(V, K, 3, 0.5)
    save('separation_mini', params=np.array([sr, N, hop, D, S, K, I]), micSep=np.array(d), samples=x,
         X=X, V=V, W=W, H=H, coherence=coh, angularSpectrogram=A, meanAngularSpectrum=m,
         targetTDOAIndexes=np.array(idx), targetTDOAGCCNMFs=G, targetCoefficientMasks=M,
         targetSpectrogramEstimates=Sp, targetSignalEstimates=y,
         W0=W0, H0=H0, W1=W1, H1=H1, W3_alpha=W3s, H3_alpha=H3s)


def golden_enhancement():
    """notebooks/offlineSpeechEnhancement.ipynb: cells 12,17,22,27,29,36,41 exec()-ed verbatim."""
    cells = notebook_cells('offlineSpeechEnhancement')
    ns = {}
    exec('from gccNMF.gccNMFFunctions import *\nimport numpy as np', ns)
    ns.update(windowSize=256, fftSize=256, hopSize=64, windowFunction=np.hanning, numTDOAs=16,
              targetTDOAWindowSizePercent=0.05, dictionarySize=32, numIterations=15, sparsityAlpha=0,
              microphoneSeparationInMetres=0.1, numSources=1, sampleRate=16000)
    ns['stereoSamples'] = synthetic_stereo(0.5, seed=11)
    exec('hypothesisTDOAs = getTDOAsInSeconds(microphoneSeparationInMetres, numTDOAs)\n'
         'targetTDOAWindowSize = (hypothesisTDOAs[-1] - hypothesisTDOAs[0]) * targetTDOAWindowSizePercent', ns)  # cell 4 tail
    for i in (12, 17, 22, 27, 29, 36):
        exec(cells[i], ns)
    exec('targetSignalEstimates = getTargetSignalEstimates( targetSpectrogramEstimates, windowSize, hopSize, windowFunction )', ns)  # cell 41 minus the wav write
    save('enhancement_mini', params=np.array([16000, 256, 64, 16, 1, 32, 15]), micSep=np.array(0.1),
         samples=ns['stereoSamples'], X=ns['complexMixtureSpectrogram'], W=ns['W'], H=ns['H'],
         coherence=ns['spectralCoherenceV'], angularSpectrogram=ns['angularSpectrogram'],
         targetTDOAIndexes=np.array(ns['targetTDOAIndexes']), gccNMF=ns['gccNMF'],
         argMaxGCCNMF=ns['argMaxGCCNMF'], targetCoefficientMasks=ns['targetCoefficientMasks'],
         targetSpectrogramEstimates_sha256=np.array(array_digest(ns['targetSpectrogramEstimates'])),
         targetSignalEstimates=ns['targetSignalEstimates'])


def golden_online():
    """notebooks/onlineSpeechEnhancement.ipynb cells 21+23 and lowLatencySpeechEnhancement.ipynb
    cells 21,23,28,30 exec()-ed verbatim (numInferenceIterations = 0: the only branch that runs)."""
    x = synthetic_stereo(0.4, seed=23)
    N, hop, D, K = 256, 32, 32, 24
    Xs = ref.computeComplexMixtureSpectrogram(x, N, 64, np.hanning)
    W, _ = ref.performKLNMF(np.concatenate(np.abs(Xs), axis=-1), K, 30, 0)
    base = dict(stereoSamples=x, sampleRate=16000, numSamples=x.shape[1], W=W, dictionarySize=K,
                numTDOAs=D, targetTDOAEpsilon=0.05 * D, numInferenceIterations=0, sparsityAlpha=0,
                epsilon=1e-16, seedValue=0, microphoneSeparationInMetres=0.1,
                numFrequencies=W.shape[0], frequenciesInHz=ref.getFrequenciesInHz(16000, W.shape[0]))

    cells = notebook_cells('onlineSpeechEnhancement')
    ns = dict(base)
    exec('from gccNMF.gccNMFFunctions import *\nfrom numpy import *\nfrom numpy.fft import rfft, irfft', ns)
    ns.update(windowSize=N, hopSize=hop, window=np.hanning(N), stftGainFactor=hop / float(N) * 2)
    exec(cells[21], ns)
    exec(cells[23], ns)
    save('online_mini', params=np.array([16000, N, hop, D, K]), micSep=np.array(0.1), samples=x, W=W,
         output=ns['targetEstimateSamplesOLA'], targetTDOAs=ns['targetTDOAs'],
         angularSpectrogram=ns['angularSpectrogram'], atomMasks=ns['atomMasks'],
         wienerFilters=ns['wienerFilters'])

    cells = notebook_cells('lowLatencySpeechEnhancement')
    ns = dict(base)
    exec('from gccNMF.gccNMFFunctions import *\nfrom numpy import *\nfrom numpy.fft import rfft, irfft', ns)
    synth = 32
    ns.update(fftSize=N, analysisWindowSize=N, synthesisWindowSize=synth, asymmetricHopSize=(synth * 3) // 4,
              m=synth // 2, k=N, d=0, symmetricWindowSize=N, symmetricHopSize=(synth * 3) // 4)
    for i in (21, 23, 28, 30):
        exec(cells[i], ns)
    sym = ns['performOnlineSpeechEnhancement'](ns['symmetricWindow'], ns['symmetricWindow'], ns['symmetricHopSize'])
    asym = ns['performOnlineSpeechEnhancement'](ns['analysisWindow'], ns['synthesisWindow'], ns['asymmetricHopSize'])
    save('lowlatency_mini', params=np.array([16000, N, (synth * 3) // 4, D, K, synth]), micSep=np.array(0.1), samples=x, W=W,
         analysisWindow=ns['analysisWindow'], synthesisWindow=ns['synthesisWindow'], symmetricWindow=ns['symmetricWindow'],
         sym_output=sym[2], sym_targetTDOAs=sym[4], sym_atomMasks=sym[6], sym_wienerFilters=sym[7],
         asym_output=asym[2], asym_targetTDOAs=asym[4], asym_atomMasks=asym[6], asym_wienerFilters=asym[7])


def golden_pretraining():
    """gccNMF/realtime/gccNMFPretraining.py:80 call shape: performKLNMF on a float64, Fortran-ordered
    magnitude matrix (a column subset of data/chimeTrainSet.npy rows 0::8 to stay small), then
    getOrderedDictionary (:60-66)."""
    from gccNMF.realtime.gccNMFPretraining import getOrderedDictionary
    chime = np.load(os.path.join(REF, 'data', 'chimeTrainSet.npy'))
    trainV = np.asfortranarray(chime[::8, :96])
    W, H = ref.performKLNMF(trainV, 12, numIterations=20, sparsityAlpha=0, epsilon=1e-16, seedValue=0)
    save('pretraining_mini', trainV=trainV, W=W, H=H, orderedW=getOrderedDictionary(W))


def golden_c1_digest():
    """Config 1 (BASELINE.json configs[0]) on the shipped SiSEC mixture: a digest only (indices,
    mask sums, norms, strided samples) because the wav cannot travel."""
    x, sr = ref.loadMixtureSignal(os.path.join(REF, 'data', 'dev1_female3_liverec_130ms_1m_mix.wav'))
    N, hop, D, d, S = 1024, 512, 64, 1.0, 3
    X = ref.computeComplexMixtureSpectrogram(x, N, hop, np.hanning)
    f = np.linspace(0, sr / 2.0, X.shape[1])
    V = np.concatenate(np.abs(X), axis=-1)
    W, H = ref.performKLNMF(V, 128, 100, 0)
    stereoH = np.array(np.hsplit(H, 2))
    coh = X[0] * X[1].conj() / np.abs(X[0]) / np.abs(X[1])
    A = ref.getAngularSpectrogram(coh, f, d, D)
    idx = ref.estimateTargetTDOAIndexesFromAngularSpectrum(np.mean(A, axis=-1), d, D, S)
    G = ref.getTargetTDOAGCCNMFs(coh, d, D, f, idx, W, stereoH)
    M = ref.getTargetCoefficientMasks(G, S)
    Sp = ref.getTargetSpectrogramEstimates(M, X, W, stereoH)
    y = ref.getTargetSignalEstimates(Sp, N, hop, np.hanning)
    save('c1_digest', params=np.array([sr, N, hop, D, S, 128, 100]), micSep=np.array(d),
         X_shape=np.array(X.shape), X_strided=X[:, ::37, ::29], V_sum=np.array(V.sum(dtype=np.float64)),
         W_strided=W[::16, ::8], H_strided=H[::8, ::31], W_norm=np.array(np.linalg.norm(W.astype(np.float64))),
         H_norm=np.array(np.linalg.norm(H.astype(np.float64))), meanAngularSpectrum=np.mean(A, axis=-1),
         targetTDOAIndexes=np.array(idx), maskSums=M.sum(axis=(1, 2)), y_shape=np.array(y.shape),
         y_strided=y[:, :, ::997], y_norm=np.array(np.linalg.norm(y.astype(np.float64))))
    # teacher-forcing set for the stages after the NMF: the reference's W, H and its binary masks (bit-packed), a strided
    # view of the per-target GCC-NMFs and of the spectrogram estimates (the recording itself travels as tests/golden/*.wav)
    save('c1_full', W=W, H=H, masks_packed=np.packbits(M.astype(bool)), masks_shape=np.array(M.shape),
         G_strided=G[:, ::5, ::7], Sp_strided=Sp[:, :, ::37, ::29], y_head=y[:, :, 20000:24096])


def golden_wavfile():
    """gccNMF/wavfile.py: wavwrite (clip protection, float2pcm) and wavread (pcm2float) on a signal that exceeds 1 and
    one that does not, plus the unsigned-PCM offset; the written files travel as raw bytes."""
    import tempfile
    from gccNMF import wavfile as refwav
    rng = np.random.default_rng(3)
    quiet = (0.3 * rng.standard_normal((2, 400))).clip(-0.999, 0.999).astype(np.float32)
    loud = (2.0 * rng.standard_normal((2, 400))).astype(np.float32)
    d = tempfile.mkdtemp()
    out = {}
    for name, x in (('quiet', quiet), ('loud', loud)):
        path = os.path.join(d, name + '.wav')
        refwav.wavwrite(x, path, 16000)
        out[name + '_bytes'] = np.frombuffer(open(path, 'rb').read(), dtype=np.uint8)
        out[name + '_read'] = refwav.wavread(path)[0]
    u8 = np.arange(256, dtype=np.uint8)
    save('wavfile_mini', quiet=quiet, loud=loud, u8=u8, u8_float=refwav.pcm2float(u8), **out)


def golden_realtime():
    """gccNMF/realtime/gccNMFProcessor.py:167-276 (GCCNMFProcessor) and gccNMF/realtime/utils.py:72-116 (OverlapAddProcessor),
    UNMODIFIED, executed over oracle/theano_numpy_shim.py (Theano itself is absent: the stand-in evaluates the reference's own
    graph with numpy -- see its header for what that does and does not pin)."""
    sys.path.insert(0, ROOT)
    from oracle import theano_numpy_shim
    theano_numpy_shim.install()
    from gccNMF.realtime.gccNMFProcessor import GCCNMFProcessor, TARGET_MODE_BOXCAR, TARGET_MODE_WINDOW_FUNCTION
    from gccNMF.realtime.utils import OverlapAddProcessor, SharedMemoryCircularBuffer
    sr, N, K, D = 16000, 256, 64, 32
    rng = np.random.default_rng(77)
    W = (rng.random((N // 2 + 1, K)) ** 3).astype(np.float32)
    out = dict(params=np.array([sr, N, K, D]), micSep=np.array(0.1), W=W, targetRange=np.array([10.0, 3.0, 2.0, 0.01]),
               modes=np.array([TARGET_MODE_BOXCAR, TARGET_MODE_WINDOW_FUNCTION]))

    def make(nT, mode):
        p = GCCNMFProcessor(sr, N, nT, {'Pretrained': {K: W}}, 'Pretrained', K, 0, 0.1, True, 6,
                            gccPHATHistory=SharedMemoryCircularBuffer((D, 128)), tdoaHistory=SharedMemoryCircularBuffer((1, 128)))
        p.numTDOAs = D
        p.targetMode = mode
        p.reset()
        p.setTargetTDOARange(10.0, 3.0, 2.0, 0.01)
        return p

    for tag, nT, mode in (('w1', 1, TARGET_MODE_WINDOW_FUNCTION), ('b4', 4, TARGET_MODE_BOXCAR), ('w4', 4, TARGET_MODE_WINDOW_FUNCTION)):
        p = make(nT, mode)
        steps = 12
        frames_all, y_all, tgt, hm, am, gp = [], [], [], [], [], []
        for step in range(steps):
            # a delayed copy in the right channel gives a well-defined TDOA peak
            s = rng.standard_normal((N + 8, nT)).astype(np.float32)
            frames = np.stack([s[4:4 + N], 0.8 * s[2:2 + N] + 0.05 * rng.standard_normal((N, nT)).astype(np.float32)])
            target_before = float(p.targetTDOAIndex.get_value())
            y = p.processFrames(frames)
            target_after = float(p.targetTDOAIndex.get_value())
            realGCC = p.getComplexGCC()[0].real                    # (F, nT, D) of the spectrogram just processed
            gccNMF = p.getGCCNMF(realGCC)[0]                       # (D, nT, K)
            # the mask of this call used the target index of BEFORE its localisation update
            p.targetTDOAIndex.set_value(np.float32(target_before))
            hmask = p.getTFMask(realGCC)[1]
            p.targetTDOAIndex.set_value(np.float32(target_after))
            frames_all.append(frames); y_all.append(y); tgt.append(target_after)
            hm.append(np.asarray(hmask, np.float64)); am.append(np.argmax(gccNMF, axis=0).T.astype(np.int32))
            gp.append(np.nanmean(realGCC, axis=0).T.astype(np.float32))
        out.update({tag + '_frames': np.stack(frames_all), tag + '_y': np.stack(y_all), tag + '_target': np.array(tgt),
                    tag + '_hmask': np.stack(hm), tag + '_argmax': np.stack(am), tag + '_gccphat': np.stack(gp)})
    # the overlap-add ring driving the processor (gccNMFProcessor.py:97), 24 blocks
    hop, B = 128, 256
    nT = B // hop
    p = make(nT, TARGET_MODE_WINDOW_FUNCTION)
    p.setTargetTDOARange(9.60, 5.0, 2.0, 0.0)                       # the headless runner's messages (runRealtimeGCCNMF.py:141-161)
    n = 24 * B
    s = rng.standard_normal(n + 8).astype(np.float32)
    x = (0.2 * np.stack([s[4:4 + n], 0.8 * s[2:2 + n] + 0.05 * rng.standard_normal(n).astype(np.float32)])).astype(np.float32)
    inputFrames, outputFrames = np.zeros((2, B), np.float32), np.zeros((2, B), np.float32)
    olad = OverlapAddProcessor(2, N, hop, B, nT, inputFrames, outputFrames)
    blocks, targets, masks = [], [], []
    for b in range(n // B):
        inputFrames[:] = x[:, b * B:(b + 1) * B]
        target_before = float(p.targetTDOAIndex.get_value())
        olad.processFrames(p.processFrames)
        target_after = float(p.targetTDOAIndex.get_value())
        p.targetTDOAIndex.set_value(np.float32(target_before))
        masks.append(np.asarray(p.getTFMask(p.getComplexGCC()[0].real)[1], np.float64))     # the atom mask this block was filtered with
        p.targetTDOAIndex.set_value(np.float32(target_after))
        blocks.append(outputFrames.copy())
        targets.append(target_after)
    out.update(ola_params=np.array([hop, B, nT]), ola_x=x, ola_out=np.concatenate(blocks, axis=1), ola_target=np.array(targets),
               ola_hmask=np.stack(masks))
    save('realtime_mini', **out)


if __name__ == '__main__':
    os.makedirs(OUT, exist_ok=True)
    golden_realtime()
    golden_wavfile()
    golden_separation()
    golden_enhancement()
    golden_online()
    golden_pretraining()
    golden_c1_digest()
