"""CPU ORACLE (test infrastructure, NOT product code) -- numpy restatement of
honk2's ``AudioProcessor.compute_mfccs``.

Follows /root/reference/utils/audio_processor.py:8-30.  The arithmetic itself lives in
third-party code that is absent from the reference tree and un-pinned there:
``librosa`` (requirements.txt:6, no version; the positional
``librosa.feature.melspectrogram(data, sr=...)`` call at audio_processor.py:19-26 needs
librosa < 0.10) and ``scipy.fftpack.dct`` (audio_processor.py:28).  The published librosa<0.10
algorithm is restated here:

    feature.melspectrogram -> core.spectrum._spectrogram -> core.stft (center=True,
    pad_mode='reflect', window='hann' periodic, float64 FFT stored as complex64),
    |S|**2 (float32), filters.mel (Slaney scale, norm='slaney', float32), np.dot.

PARITY PIN: the reference holds no golden vectors for this path (SURVEY.md section 8c) and
librosa cannot be installed here, so at the librosa boundary this oracle is "parity
unpinned"; it is cross-checked against torchaudio's independent MelSpectrogram
(tests/test_oracle_mfcc.py) and frozen in tests/golden/mfcc_*.npz.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
import this module.
"""
import numpy as np

SR = 16000
N_FFT = 480
HOP = 160
N_MELS = 40
F_MIN = 20.0
F_MAX = 4000.0


def hz_to_mel(freq):
    """Slaney mel scale (librosa.core.convert.hz_to_mel, htk=False)."""
    freq = np.asanyarray(freq, dtype=np.float64)
    f_sp = 200.0 / 3
    mels = freq / f_sp
    min_log_hz = 1000.0
    min_log_mel = min_log_hz / f_sp
    logstep = np.log(6.4) / 27.0
    big = freq >= min_log_hz
    safe = np.where(big, freq, min_log_hz)
    return np.where(big, min_log_mel + np.log(safe / min_log_hz) / logstep, mels)


def mel_to_hz(mels):
    """Inverse of hz_to_mel (librosa.core.convert.mel_to_hz, htk=False)."""
    mels = np.asanyarray(mels, dtype=np.float64)
    f_sp = 200.0 / 3
    freqs = f_sp * mels
    min_log_hz = 1000.0
    min_log_mel = min_log_hz / f_sp
    logstep = np.log(6.4) / 27.0
    big = mels >= min_log_mel
    return np.where(big, min_log_hz * np.exp(logstep * (mels - min_log_mel)), freqs)


def mel_filterbank(sr=SR, n_fft=N_FFT, n_mels=N_MELS, fmin=F_MIN, fmax=F_MAX):
    """librosa.filters.mel(sr, n_fft, n_mels, fmin, fmax, htk=False, norm='slaney'),
    float32 [n_mels, 1 + n_fft//2] (call site audio_processor.py:19-26)."""
    if fmax is None:
        fmax = sr / 2.0
    n_bins = 1 + n_fft // 2
    weights = np.zeros((n_mels, n_bins), dtype=np.float32)
    fftfreqs = np.linspace(0, float(sr) / 2, n_bins, endpoint=True)
    mel_f = mel_to_hz(np.linspace(hz_to_mel(fmin), hz_to_mel(fmax), n_mels + 2))
    fdiff = np.diff(mel_f)
    ramps = np.subtract.outer(mel_f, fftfreqs)
    for i in range(n_mels):
        lower = -ramps[i] / fdiff[i]
        upper = ramps[i + 2] / fdiff[i + 1]
        weights[i] = np.maximum(0, np.minimum(lower, upper))
    enorm = 2.0 / (mel_f[2:n_mels + 2] - mel_f[:n_mels])
    weights *= enorm[:, np.newaxis]
    return weights


def hann_periodic(n=N_FFT):
    """scipy.signal.get_window('hann', n, fftbins=True) in float64."""
    return 0.5 - 0.5 * np.cos(2.0 * np.pi * np.arange(n) / n)


def n_frames(n_samples, hop=HOP):
    return 1 + n_samples // hop


def mel_power(y, sr=SR, n_fft=N_FFT, hop=HOP, n_mels=N_MELS, fmin=F_MIN, fmax=F_MAX):
    """[n_mels, T] float32 mel power spectrogram == librosa.feature.melspectrogram(y, ...)."""
    y = np.asarray(y)
    if y.ndim != 1:
        raise ValueError("compute_mfccs expects a 1-D waveform")
    if not np.issubdtype(y.dtype, np.floating):
        raise ValueError("Audio data must be floating-point")  # librosa.util.valid_audio
    if not np.isfinite(y).all():
        raise ValueError("Audio buffer is not finite everywhere")
    pad = n_fft // 2
    y_pad = np.pad(y, pad, mode="reflect")
    T = n_frames(len(y), hop)
    idx = np.arange(n_fft)[:, None] + hop * np.arange(T)[None, :]
    frames = y_pad[idx]                                  # [n_fft, T], dtype of y
    win = hann_periodic(n_fft)[:, None]                  # float64
    stft = np.fft.rfft(win * frames, axis=0).astype(np.complex64)
    power = np.abs(stft) ** 2.0                          # float32
    W = mel_filterbank(sr, n_fft, n_mels, fmin, fmax)
    return np.dot(W, power).astype(np.float32)


def compute_mfccs(y, **kw):
    """== AudioProcessor.compute_mfccs (audio_processor.py:18-30): float32 [(T, 40, 1)].

    log where > 0 (:27); scipy.fftpack.dct over the length-1 last axis of each (40,1)
    column slice (:28) is an un-normalised DCT-II of one sample == 2*x; stacked to
    (T, 40, 1) float32 (:29)."""
    data = mel_power(y, **kw)
    pos = data > 0
    data[pos] = np.log(data[pos])
    data = 2.0 * data
    return np.ascontiguousarray(data.T[:, :, None]).astype(np.float32)


def compute_mfccs_batch(waves, **kw):
    """The collate loop of data_loader/audio_data_loader.py:26-29: per-sample compute_mfccs,
    reshape(1, -1, n_mels), concatenate on dim 0 -> float32 [B, T, n_mels] (n_mels = 40 by default)."""
    n_mels = kw.get("n_mels", N_MELS)
    return np.concatenate([compute_mfccs(w, **kw).reshape(1, -1, n_mels) for w in waves], 0)
