"""Host side of the streaming-window path (SURVEY 8f-1): what ``StreamingDataset`` (dataset/dataset_utils.py:20-95)
does around the audio, restated for a stream that is already one array -- window count, window targets -- plus
``evaluate_stream``: features of all sliding windows from the shared-frame front-end, then the model, batch by batch;
and ``LiveStreams``, the same windows for many streams whose audio arrives a chunk at a time.
"""
import collections
import ctypes as C

import numpy as np
import torch

from . import _native
from .audio_processor import AudioProcessor


def n_stream_windows(total_num_samples, window_size, shift_size):
    """StreamingDataset.num_samples (dataset_utils.py:31)."""
    return AudioProcessor.n_stream_windows(total_num_samples, window_size, shift_size)


def stream_window_targets(segment_lengths, segment_labels, n_labels, window_size, shift_size, n_windows=None):
    """Target label of every window of a stream made of labelled segments (audio files played back to back).

    The reference keeps a running ``label_counter`` over the samples of the current window and picks the label with
    the largest count, the LOWEST label index winning ties (strict ``>`` while enumerating, dataset_utils.py:74-81).
    Its incremental bookkeeping (:58-62, :84-92) always equals the label histogram of
    stream[k*shift : k*shift + window]; this computes all windows at once from per-label prefix sums.
    Returns int64 [n_windows]."""
    segment_lengths = np.asarray(segment_lengths, dtype=np.int64)
    segment_labels = np.asarray(segment_labels, dtype=np.int64)
    if segment_lengths.shape != segment_labels.shape or segment_lengths.ndim != 1:
        raise ValueError("segment_lengths and segment_labels must be 1-D and of equal length")
    if (segment_lengths < 0).any() or ((segment_labels < 0) | (segment_labels >= n_labels)).any():
        raise ValueError("negative segment length or label outside [0, n_labels)")
    total = int(segment_lengths.sum())
    avail = n_stream_windows(total, window_size, shift_size)
    if n_windows is None:
        n_windows = avail
    if n_windows > avail:
        raise ValueError(f"{n_windows} windows requested, the stream has {avail}")
    if n_windows <= 0:
        return np.zeros((0,), dtype=np.int64)
    # prefix[c, i] = number of samples with label c among stream[:i], evaluated only where windows start / end
    bounds = np.concatenate(([0], np.cumsum(segment_lengths)))
    starts = np.arange(n_windows, dtype=np.int64) * shift_size
    ends = starts + window_size
    counts = np.zeros((n_windows, n_labels), dtype=np.int64)
    for c in range(n_labels):
        seg_c = np.where(segment_labels == c, segment_lengths, 0)
        cum_c = np.concatenate(([0], np.cumsum(seg_c)))          # label-c samples in the first j segments

        def prefix(pos):
            j = np.searchsorted(bounds, pos, side="right") - 1    # segment containing position pos
            j = np.minimum(j, len(segment_lengths) - 1)
            inside = pos - bounds[j]
            return cum_c[j] + np.where(segment_labels[j] == c, inside, 0)

        counts[:, c] = prefix(ends) - prefix(starts)
    return np.argmax(counts, axis=1).astype(np.int64)


def evaluate_stream(model, audio_processor, stream, window_size=16000, shift_size=160, targets=None,
                    batch_size=8192):
    """Logits (and accuracy, if targets are given) of every window of a CUDA stream tensor [L].

    Replaces iterating a StreamingDataset through AudioDataLoader + run/test.py:evaluate (18-41): per batch ONE
    front-end call that computes each shared frame once (AudioProcessor.compute_mfccs_stream) and one model call;
    correct/total accumulate on the device, one host sync at the end."""
    if not (isinstance(stream, torch.Tensor) and stream.is_cuda and stream.dim() == 1):
        raise ValueError("evaluate_stream expects a 1-D CUDA tensor")
    n = n_stream_windows(stream.numel(), window_size, shift_size)
    from .metric import Acc
    logits = []
    acc = Acc()
    tgt = None
    if targets is not None:
        tgt = torch.as_tensor(np.asarray(targets), dtype=torch.int64, device=stream.device)
        if tgt.numel() != n:
            raise ValueError(f"{tgt.numel()} targets for {n} windows")
    with torch.no_grad():
        for first in range(0, n, batch_size):
            count = min(batch_size, n - first)
            feats = audio_processor.compute_mfccs_stream(stream, window_size, shift_size, first=first, count=count)
            y = model(feats)
            logits.append(y)
            if tgt is not None:
                acc.accumulate(y, tgt[first:first + count])     # kws_acc_accumulate: counts stay on the device
    out = torch.cat(logits) if logits else torch.empty((0, 0), device=stream.device)
    if tgt is None:
        return out
    return out, {"correct": acc.counts()[0], "total": n}


RaggedPlan = collections.namedtuple("RaggedPlan", "stream_ids window_ids row_bound window_bound")


def ragged_push_plan(seen, lengths, window_size, shift_size):
    """Host plan of a ragged push (``LiveStreams.push_ragged``, ``kws_live_push_ragged``): stream s has seen ``seen[s]``
    samples and brings ``lengths[s]`` more.  It completes windows k with
    ``max(0, floor((seen - W) / H) + 1) <= k <= floor((seen + n - W) / H)``; returns their ``stream_ids`` and
    ``window_ids`` (int64, ordered by stream, then window), and the bounds the library sizes its launches with:
    ``row_bound = sum(ceil(n / 160))`` new frame-table rows and ``window_bound = sum(ceil(n / H))`` windows."""
    seen = np.asarray(seen, dtype=np.int64)
    n = np.asarray(lengths, dtype=np.int64)
    first = np.maximum(0, (seen - window_size) // shift_size + 1)
    count = np.maximum(0, (seen + n - window_size) // shift_size + 1 - first)
    stream_ids = np.repeat(np.arange(seen.size, dtype=np.int64), count)
    starts = np.cumsum(count) - count                   # each stream's first row in the compacted list
    window_ids = np.arange(stream_ids.size, dtype=np.int64) - np.repeat(starts - first, count)
    return RaggedPlan(stream_ids, window_ids, int((-(-n // 160)).sum()), int((-(-n // shift_size)).sum()))


class _LiveState(object):
    """What the live states share: device selection, the host's copy of the sample counters, the checks of a uniform
    push's chunk and of a ragged push's samples and lengths, the validity mask of a uniform push's slots, reset and
    pickling.  Subclasses name their C functions (``_create``, ``_reset_fn``, ``_destroy_fn``) and add their own device
    buffers."""
    _kind = "live state"

    def __init__(self, audio_processor, n_streams, window_size, shift_size, max_push, device):
        self.audio_processor = audio_processor   # owns the front-end tables the state reads
        self.n_streams = int(n_streams)
        self.window_size = int(window_size)
        self.shift_size = int(shift_size)
        self.max_push = int(max_push)
        dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        if dev.type != "cuda":
            raise _native.NativeError(f"{type(self).__name__} needs a CUDA device: there is no CPU path")
        self.device = torch.device("cuda", dev.index if dev.index is not None else torch.cuda.current_device())
        self.n_frames = audio_processor.n_frames(self.window_size)
        self._handle = None
        self._seen = np.zeros(self.n_streams, dtype=np.int64)

    def _state(self):
        if self._handle is None:
            self._handle = self._create(_native.load())
            self._seen[:] = 0
            # reset's stream ids: pinned staging buffer, device copy, and the event that marks the staging buffer free
            self._ids_host = torch.empty(self.n_streams, dtype=torch.int64, pin_memory=True)
            self._ids_dev = torch.empty(self.n_streams, dtype=torch.int64, device=self.device)
            self._ids_copied = torch.cuda.Event()
        return self._handle

    @property
    def samples_seen(self):
        """Samples pushed into each stream since its last reset: CPU int64 [S]."""
        return torch.from_numpy(self._seen.copy())

    def _check_chunk(self, chunk):
        """A uniform push's chunk as the C call takes it: (contiguous chunk, pcm16?)."""
        name = type(self).__name__
        if not (isinstance(chunk, torch.Tensor) and chunk.is_cuda):
            raise _native.NativeError(f"{name}.push needs a CUDA tensor: there is no CPU path")
        if chunk.dim() != 2 or chunk.shape[0] != self.n_streams:
            raise ValueError(f"expected a chunk shaped [{self.n_streams}, n], got {tuple(chunk.shape)}")
        if chunk.device != self.device:
            raise ValueError(f"the chunk is on {chunk.device}, the live state on {self.device}")
        misaligned = np.flatnonzero(self._seen % 160)
        if misaligned.size:
            s = int(misaligned[0])
            raise ValueError(f"stream {s} has seen {int(self._seen[s])} samples, not a multiple of the 160-sample hop "
                             "(a ragged push left it so); push needs aligned counts: use push_ragged")
        pcm16 = chunk.dtype == torch.int16
        if not pcm16 and chunk.dtype != torch.float32:
            chunk = chunk.float()
        return chunk.contiguous(), pcm16

    def _check_ragged(self, samples, lengths):
        """A ragged push's arguments as the C call takes them: (contiguous samples, lengths int64 [S], pcm16?)."""
        name = type(self).__name__
        if not (isinstance(samples, torch.Tensor) and samples.is_cuda):
            raise _native.NativeError(f"{name}.push_ragged needs a CUDA tensor: there is no CPU path")
        if samples.dim() != 1:
            raise ValueError(f"expected 1-D samples, got shape {tuple(samples.shape)}")
        if samples.device != self.device:
            raise ValueError(f"the samples are on {samples.device}, the live state on {self.device}")
        if samples.dtype not in (torch.float32, torch.int16):
            raise ValueError(f"samples must be float32 or int16 PCM, got {samples.dtype}")
        if isinstance(lengths, torch.Tensor) and lengths.is_cuda:
            raise ValueError("push_ragged takes host lengths: the host checks them and keeps samples_seen")
        n = np.asarray(lengths).reshape(-1)
        if n.size != self.n_streams or not np.issubdtype(n.dtype, np.integer):
            raise ValueError(f"expected {self.n_streams} integer lengths, got {n.size} of {n.dtype}")
        n = n.astype(np.int64)
        if ((n < 0) | (n > self.max_push)).any():
            s = int(np.flatnonzero((n < 0) | (n > self.max_push))[0])
            raise ValueError(f"stream {s} brings {int(n[s])} samples; a push takes 0 to max_push = {self.max_push}")
        if int(n.sum()) != samples.numel():
            raise ValueError(f"the lengths add up to {int(n.sum())} samples, the tensor holds {samples.numel()}")
        return samples.contiguous(), n, samples.dtype == torch.int16

    def _advance(self, n):
        """After a uniform push of n samples: the host-side validity mask [S, K] of its slots; counters advance."""
        # window index of slot j: floor((c - W) / H) + 1 + j, c = samples before this push
        first = (self._seen - self.window_size) // self.shift_size + 1
        valid = torch.from_numpy(first[:, None] + np.arange(n // self.shift_size)[None, :] >= 0)
        self._seen += n
        return valid

    def reset(self, stream_ids):
        """Restart the given streams at sample 0; the others are not affected.  stream_ids: host integers (a list, a
        numpy array or a CPU tensor) in [0, S); repeats are allowed."""
        if isinstance(stream_ids, torch.Tensor) and stream_ids.is_cuda:
            raise ValueError("reset takes host stream ids: the host checks them and keeps samples_seen")
        ids = np.unique(np.asarray(stream_ids, dtype=np.int64).reshape(-1))
        if ((ids < 0) | (ids >= self.n_streams)).any():
            raise ValueError(f"stream ids must lie in [0, {self.n_streams})")
        if ids.size == 0:
            return
        lib = _native.load()
        handle = self._state()
        m = ids.size
        st = torch.cuda.current_stream(self.device)
        self._ids_copied.synchronize()   # the previous reset's copy out of the staging buffer (long done, in practice)
        self._ids_host[:m].copy_(torch.from_numpy(ids))
        with torch.cuda.device(self.device):
            self._ids_dev[:m].copy_(self._ids_host[:m], non_blocking=True)
            self._ids_copied.record(st)
            _native.check(getattr(lib, self._reset_fn)(handle, C.c_void_p(self._ids_dev.data_ptr()), m,
                                                       C.c_void_p(st.cuda_stream)), self._reset_fn)
        self._seen[ids] = 0

    def __del__(self):
        try:
            lib = _native.loaded()   # (never dlopen from a destructor)
            if lib is not None and self._handle is not None:
                getattr(lib, self._destroy_fn)(self._handle)
                self._handle = None
        except Exception:
            pass

    _device_buffers = ()

    def __getstate__(self):  # device state never crosses a process boundary
        d = dict(self.__dict__)
        d["_handle"] = None
        for k in self._device_buffers:
            d[k] = None
        d["_seen"] = np.zeros_like(self._seen)
        for k in ("_ids_host", "_ids_dev", "_ids_copied"):
            d.pop(k, None)
        return d


class LiveStreams(_LiveState):
    """Live keyword-spotting front-end for ``n_streams`` microphones, fed a chunk at a time (``kws_live_*``).

    Each stream keeps a device-resident sample ring, frame ring and sample counter.  ``push(chunk)`` hands every stream
    the same number n of new samples (a CUDA ``[S, n]`` float32 or int16 PCM tensor; n a multiple of ``shift_size`` in
    ``[shift_size, max_push]``) and returns the features of the K = n / shift_size window indices the push completes per
    stream, ``[S, K, T, n_mels]``, with a host-side bool mask ``valid [S, K]``.  Window k of a stream is its samples
    ``[k * shift_size, k * shift_size + window_size)`` since its last reset -- the windows of ``StreamingDataset`` and
    ``compute_mfccs_stream``.  Slot j is window ``floor((c - window_size) / shift_size) + 1 + j`` for the sample count
    c before the push, so the last slot is the newest complete window; a slot is valid iff its window index is >= 0,
    and the features of invalid slots (the warm-up of a fresh stream) are exactly zero.  Valid features are
    bit-identical to ``compute_mfccs_batch`` on the materialised windows.  Only the new frames are computed: n / 160
    frame-table rows per stream and the four reflect-padded edge frames of each window.

    ``samples_seen`` is the host's copy of the counters, so building the mask never synchronises with the device.
    ``reset`` takes host ids, checks them and updates that copy; it stages them through buffers allocated with the
    state, so neither ``push`` nor ``reset`` allocates device memory or waits for the device.  A copy made by pickling
    holds no device state and starts every stream afresh.

    ``push_ragged(samples, lengths)`` lets every stream bring its own number of samples, and returns only the windows
    the push completes, compacted, with the stream and window index of each (see ``ragged_push_plan``)."""
    _reset_fn, _destroy_fn = "kws_live_reset", "kws_live_destroy"
    _device_buffers = ("_ragged_ws",)

    def __init__(self, audio_processor, n_streams, window_size=16000, shift_size=160, max_push=1600, device=None):
        super().__init__(audio_processor, n_streams, window_size, shift_size, max_push, device)
        self._ragged_ws = None   # device workspace of push_ragged, allocated by the first ragged push
        self._state()

    def _create(self, lib):
        fe = self.audio_processor._frontend(self.device)
        out = C.c_void_p()
        with torch.cuda.device(self.device):
            _native.check(lib.kws_live_create(fe, self.n_streams, self.window_size, self.shift_size, self.max_push,
                                              C.byref(out)), "kws_live_create")
        return out

    def state_bytes(self):
        """Device bytes the state holds (kws_live_state_bytes)."""
        lib = _native.load()
        return int(lib.kws_live_state_bytes(self.audio_processor._frontend(self.device), self.n_streams,
                                            self.window_size, self.shift_size, self.max_push))

    def push(self, chunk, model=None, out=None):
        """chunk: CUDA [S, n] float32 or int16 PCM.  Returns (features [S, K, T, n_mels], valid [S, K] CPU bool); with
        a model, (logits [S, K, n_labels], valid) where the logits are model(features.view(S * K, T, n_mels)) on the
        current stream.  ``out``: optional preallocated features buffer.

        Every stream's sample count must be a multiple of 160 (the hop).  Only ``push_ragged`` can break that; after a
        ragged push that leaves a count unaligned, ``push`` raises ValueError and changes nothing, until ragged pushes
        (or a reset) realign the counts."""
        chunk, pcm16 = self._check_chunk(chunk)
        n = chunk.shape[1]
        K = n // self.shift_size
        shape = (self.n_streams, K, self.n_frames, self.audio_processor.n_mels)
        if out is None:
            out = torch.empty(shape, dtype=torch.float32, device=self.device)
        elif out.shape != shape or out.dtype != torch.float32 or not out.is_contiguous() or out.device != self.device:
            raise ValueError(f"out must be a contiguous float32 {list(shape)} tensor on {self.device}")
        lib = _native.load()
        handle = self._state()
        fn = lib.kws_live_push_pcm16 if pcm16 else lib.kws_live_push
        with torch.cuda.device(self.device):
            _native.check(fn(handle, C.c_void_p(chunk.data_ptr()), n, C.c_void_p(out.data_ptr()),
                             C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)),
                          "kws_live_push_pcm16" if pcm16 else "kws_live_push")
        valid = self._advance(n)
        if model is None:
            return out, valid
        logits = model(out.view(self.n_streams * K, self.n_frames, self.audio_processor.n_mels))
        return logits.view(self.n_streams, K, -1), valid

    def push_ragged(self, samples, lengths, model=None, out=None):
        """Stream s brings ``lengths[s]`` new samples, any number in ``[0, max_push]``.

        samples: 1-D CUDA float32 or int16 PCM tensor, all streams' new samples back to back in stream order
        (``sum(lengths)`` of them).  lengths: host sequence of S ints.  Returns ``(features [M, T, n_mels],
        stream_ids [M], window_ids [M])`` for the M windows the push completes, ordered by stream, then window; the ids
        are CPU int64 from the host's copy of the counters (``ragged_push_plan``), so nothing waits for the device.
        With a model, ``(logits [M, n_labels], stream_ids, window_ids)``, the logits being ``model(features)`` on the
        current stream; when M = 0 the samples are still pushed, the model is not called and the tensors are empty.
        ``out``: optional preallocated contiguous float32 features buffer of at least ``sum(ceil(n / shift_size))``
        rows (which bounds M); the features are its first M rows."""
        samples, n, pcm16 = self._check_ragged(samples, lengths)
        plan = ragged_push_plan(self._seen, n, self.window_size, self.shift_size)
        shape = (plan.window_bound, self.n_frames, self.audio_processor.n_mels)
        if out is None:
            out = torch.empty(shape, dtype=torch.float32, device=self.device)
        elif out.dim() != 3 or out.shape[0] < shape[0] or out.shape[1:] != shape[1:] or out.dtype != torch.float32 \
                or not out.is_contiguous() or out.device != self.device:
            raise ValueError(f"out must be a contiguous float32 [>= {shape[0]}, {shape[1]}, {shape[2]}] tensor on "
                             f"{self.device}")
        lib = _native.load()
        handle = self._state()
        if self._ragged_ws is None:
            self._ragged_ws = torch.empty(max(1, int(lib.kws_live_ragged_workspace_bytes(handle))), dtype=torch.uint8,
                                          device=self.device)
        lengths32 = np.ascontiguousarray(n, dtype=np.int32)
        fn = lib.kws_live_push_ragged_pcm16 if pcm16 else lib.kws_live_push_ragged
        with torch.cuda.device(self.device):
            _native.check(fn(handle, C.c_void_p(samples.data_ptr()), C.c_void_p(lengths32.ctypes.data),
                             C.c_void_p(out.data_ptr()), None, None, out.shape[0], None,
                             C.c_void_p(self._ragged_ws.data_ptr()), self._ragged_ws.numel(),
                             C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)),
                          "kws_live_push_ragged_pcm16" if pcm16 else "kws_live_push_ragged")
        self._seen += n
        M = plan.stream_ids.size
        ids = torch.from_numpy(plan.stream_ids), torch.from_numpy(plan.window_ids)
        feats = out[:M]
        if model is None:
            return (feats,) + ids
        if M == 0:
            return (torch.empty((0, model.n_labels), dtype=torch.float32, device=self.device),) + ids
        return (model(feats),) + ids



class LiveCNN(_LiveState):
    """Live keyword spotting with a CNN for ``n_streams`` microphones (``kws_live_cnn_*``): a live front-end and the
    bf16 tensor-core CNN in one state, where each push returns the logits of the windows it completes.

    The slots, the validity mask, ``samples_seen`` and ``reset`` are those of ``LiveStreams``.  The CNN's convolutions
    do not pad in time, so a window's convolution rows are its stream's rows except the four of each convolution that
    read the window's reflect-padded edge frames: a push computes n / 160 new rows of each convolution per stream and
    those four per window, instead of the whole network per window.  The logits are bit-identical to
    ``LiveStreams.push(chunk, model)`` on the same audio.

    ``push_ragged(samples, lengths)`` lets every stream bring its own number of samples and returns the logits of only
    the windows the push completes, compacted, as ``LiveStreams.push_ragged(samples, lengths, model)`` does and
    bit-identical to it; it too computes each convolution row of a stream once.  The two pushes may be mixed on one
    state while every stream's sample count is a multiple of 160.

    ``model`` must be a ``honk2_b200.CNN`` with ``precision == "bf16"`` whose shape has the tensor-core path, and
    ``1 + window_size / 160`` must be its ``time``.  The state copies the model's weights when it is created: later
    changes to the model do not reach it.  ``max_push`` defaults to 10 shifts."""
    _reset_fn, _destroy_fn = "kws_live_cnn_reset", "kws_live_cnn_destroy"
    _device_buffers = ("_ragged_ws",)

    def __init__(self, model, n_streams, window_size=16000, shift_size=160, max_push=None, audio_processor=None,
                 device=None):
        from .model import CNN
        if not isinstance(model, CNN):
            raise ValueError(f"LiveCNN runs a honk2_b200.CNN, got {type(model).__name__}")
        if model.precision != "bf16":
            raise ValueError(f"LiveCNN runs the bf16 tensor-core CNN; the model's precision is {model.precision!r}")
        if max_push is None:
            max_push = 10 * int(shift_size)
        super().__init__(audio_processor if audio_processor is not None else AudioProcessor(), n_streams, window_size,
                         shift_size, max_push, device)
        self.n_labels = model.n_labels
        self._ragged_ws = None   # device workspace of push_ragged, allocated by the first ragged push
        self._model = model   # held until the state exists; the state keeps its own copy of the weights
        self._state()
        self._model = None

    def _model_handle(self, lib):
        model = self._model
        if model is None:
            raise _native.NativeError("a LiveCNN restored from a pickle has no model to copy the weights from")
        _, st = model._state(self.device)   # packs the current weights
        return st["handle"]

    def _create(self, lib):
        fe = self.audio_processor._frontend(self.device)
        out = C.c_void_p()
        with torch.cuda.device(self.device):
            handle = self._model_handle(lib)
            _native.check(lib.kws_live_cnn_create(handle, fe, self.n_streams, self.window_size, self.shift_size,
                                                  self.max_push, C.byref(out)), "kws_live_cnn_create")
            self._state_bytes = int(lib.kws_live_cnn_state_bytes(handle, fe, self.n_streams, self.window_size,
                                                                 self.shift_size, self.max_push))
        return out

    def state_bytes(self):
        """Device bytes the state holds (kws_live_cnn_state_bytes)."""
        if self._handle is None:
            raise _native.NativeError("the state holds no device memory")
        return self._state_bytes

    def push(self, chunk, out=None):
        """chunk: CUDA [S, n] float32 or int16 PCM, n a multiple of ``shift_size`` in ``[shift_size, max_push]``.
        Returns (logits [S, K, n_labels], valid [S, K] CPU bool), K = n / shift_size; invalid slots are all zeros.
        ``out``: optional preallocated logits buffer."""
        chunk, pcm16 = self._check_chunk(chunk)
        n = chunk.shape[1]
        shape = (self.n_streams, n // self.shift_size, self.n_labels)
        if out is None:
            out = torch.empty(shape, dtype=torch.float32, device=self.device)
        elif out.shape != shape or out.dtype != torch.float32 or not out.is_contiguous() or out.device != self.device:
            raise ValueError(f"out must be a contiguous float32 {list(shape)} tensor on {self.device}")
        lib = _native.load()
        handle = self._state()
        fn = lib.kws_live_cnn_push_pcm16 if pcm16 else lib.kws_live_cnn_push
        with torch.cuda.device(self.device):
            _native.check(fn(handle, C.c_void_p(chunk.data_ptr()), n, C.c_void_p(out.data_ptr()),
                             C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)),
                          "kws_live_cnn_push_pcm16" if pcm16 else "kws_live_cnn_push")
        return out, self._advance(n)

    def push_ragged(self, samples, lengths, out=None):
        """Stream s brings ``lengths[s]`` new samples, any number in ``[0, max_push]``; samples and lengths as for
        ``LiveStreams.push_ragged``.  Returns ``(logits [M, n_labels], stream_ids [M], window_ids [M])`` for the M windows
        the push completes, ordered by stream, then window; the ids are CPU int64 from the host's copy of the counters
        (``ragged_push_plan``), so nothing waits for the device.  When M = 0 the push still runs: it computes the
        convolution rows the streams' next windows read.  ``out``: optional preallocated contiguous float32 logits
        buffer of at least ``sum(ceil(n / shift_size))`` rows (which bounds M); the logits are its first M rows."""
        samples, n, pcm16 = self._check_ragged(samples, lengths)
        plan = ragged_push_plan(self._seen, n, self.window_size, self.shift_size)
        if out is None:
            out = torch.empty((plan.window_bound, self.n_labels), dtype=torch.float32, device=self.device)
        elif out.dim() != 2 or out.shape[0] < plan.window_bound or out.shape[1] != self.n_labels \
                or out.dtype != torch.float32 or not out.is_contiguous() or out.device != self.device:
            raise ValueError(f"out must be a contiguous float32 [>= {plan.window_bound}, {self.n_labels}] tensor on "
                             f"{self.device}")
        lib = _native.load()
        handle = self._state()
        if self._ragged_ws is None:
            self._ragged_ws = torch.empty(max(1, int(lib.kws_live_cnn_ragged_workspace_bytes(handle))),
                                          dtype=torch.uint8, device=self.device)
        lengths32 = np.ascontiguousarray(n, dtype=np.int32)
        name = "kws_live_cnn_push_ragged_pcm16" if pcm16 else "kws_live_cnn_push_ragged"
        with torch.cuda.device(self.device):
            _native.check(getattr(lib, name)(handle, C.c_void_p(samples.data_ptr()), C.c_void_p(lengths32.ctypes.data),
                                             C.c_void_p(out.data_ptr()), None, None, out.shape[0], None,
                                             C.c_void_p(self._ragged_ws.data_ptr()), self._ragged_ws.numel(),
                                             C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)), name)
        self._seen += n
        M = plan.stream_ids.size
        return out[:M], torch.from_numpy(plan.stream_ids), torch.from_numpy(plan.window_ids)
