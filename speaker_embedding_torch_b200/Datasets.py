"""Training collation on the device: drop-in for the reference's ``Datasets.Collater`` (Datasets.py:72-86).

The reference collater draws one ``frame_length`` per batch, crops every utterance at a random offset or reflect-pads
it to that length (``Correction``, Datasets.py:9-19), stacks the results with numpy and upcasts the fp16 patterns to a
``FloatTensor[N*M, Mel_Dim, T]`` on the host.  Here the collater only does the cheap part on the host -- the random
draws, in the reference's order and from the same ``np.random`` stream, and one concatenation of the patterns as they
are stored (fp16) -- and returns a ``RaggedMel``.  The crop / reflect-pad / upcast happens inside the encoder's first
kernel (``spk_encoder_forward_ragged``): no padded or cropped copy of the batch exists on either side of PCIe.

    collater = Collater(min_frame_length, max_frame_length)        # same constructor as the reference
    loader = DataLoader(dataset, collate_fn=collater, pin_memory=True, ...)
    for features in loader:
        features = features.to(device, non_blocking=True)           # Train.py:143, unchanged
        embeddings = model(features)                                # GE2E.forward accepts a RaggedMel

``RaggedMel.dense()`` materialises the reference's tensor on the host (used by the tests: bit-identical to the numpy
collater under the same seed).
"""
import numpy as np
import torch


class RaggedMel:
    """A batch of variable-length patterns: ``data`` [Mel_Dim, total_frames] (fp16 or fp32), ``table`` int32 [B, 3] =
    (start column, length, crop offset) per slice, and the batch's common frame count.

    ``segments`` (optional, int32 [U + 1]): slices ``segments[u] .. segments[u+1] - 1`` form utterance ``u``, and
    ``GE2E.forward`` returns one d-vector per utterance (the mean over its slices; ``Modules.utterance_slices`` builds
    such a batch).  Without it the slices group in runs of ``samples``.  An input gradient (``data.requires_grad``)
    needs the column spans of different utterances to be disjoint; the host copy of the table is kept to check that
    without a device synchronisation."""

    def __init__(self, data, table, frames, segments=None, _checked=False, _host=None):
        self.data, self.table, self.frames, self.segments = data, table, int(frames), segments
        self._host = _host              # (table, segments) on the host, when known
        if not _checked and not table.is_cuda:      # host-side construction: validate once, before the copy
            t = table.to(torch.int64)
            if table.dim() != 2 or table.size(1) != 3 or data.dim() != 2 or self.frames < 1:
                raise RuntimeError("RaggedMel: data must be [Mel_Dim, total_frames], table [B, 3]")
            if t.numel() and (int((t[:, 0] + t[:, 1]).max()) > data.size(1) or int(t[:, 1].min()) < 1
                              or int(t[:, 0].min()) < 0 or int(t[:, 2].min()) < 0
                              or bool(((t[:, 1] > self.frames) & (t[:, 2] + self.frames > t[:, 1])).any())):
                raise RuntimeError("RaggedMel: table entries point outside the pattern array")
            if segments is not None:
                if segments.is_cuda:
                    raise RuntimeError("RaggedMel: table and segments must both be host tensors (or both on the device)")
                g = segments.to(torch.int64)
                if (g.dim() != 1 or g.numel() < 2 or int(g[0]) != 0 or int(g[-1]) != table.size(0)
                        or bool((g[1:] <= g[:-1]).any())):
                    raise RuntimeError("RaggedMel: segments must be increasing from 0 to the number of slices %d "
                                       "(every utterance at least one slice)" % table.size(0))
            self._host = (table, segments)

    @property
    def utterances(self):
        """Number of d-vectors with segments; None without (the slices group by ``samples``)."""
        return None if self.segments is None else self.segments.numel() - 1

    def spans_disjoint(self, samples=1):
        """True when the column spans of different utterances do not overlap (utterance = segment, or a run of
        ``samples`` slices without segments).  Uses the host copy of the table; synchronises only when there is none."""
        key = ("disjoint", samples)
        cache = getattr(self, "_cache", None)
        if cache is None:
            cache = self._cache = {}
        if key not in cache:
            table, segments = self._host if self._host is not None else (self.table.cpu(), None)
            if segments is None and self.segments is not None:
                segments = self.segments.cpu()
            t = table.to(torch.int64)
            B = t.size(0)
            if segments is None:
                segments = torch.arange(0, B + 1, samples, dtype=torch.int64)
            g = segments.to(torch.int64)
            group = torch.repeat_interleave(torch.arange(g.numel() - 1), g[1:] - g[:-1])
            lo = torch.full((g.numel() - 1,), 2 ** 62, dtype=torch.int64).scatter_reduce(0, group, t[:, 0], "amin")
            hi = torch.zeros(g.numel() - 1, dtype=torch.int64).scatter_reduce(0, group, t[:, 0] + t[:, 1], "amax")
            order = torch.argsort(lo)
            cache[key] = bool((lo[order][1:] >= hi[order][:-1]).all())
        return cache[key]

    # --- the little of the tensor API that Train.py touches
    @property
    def shape(self):
        return torch.Size((self.table.size(0), self.data.size(0), self.frames))

    def size(self, dim=None):
        return self.shape if dim is None else self.shape[dim]

    def dim(self):
        return 3

    @property
    def device(self):
        return self.data.device

    @property
    def is_cuda(self):
        return self.data.is_cuda

    def pin_memory(self):
        return RaggedMel(self.data.pin_memory(), self.table.pin_memory(), self.frames,
                         None if self.segments is None else self.segments.pin_memory(), _checked=True,
                         _host=self._host)

    def to(self, device, non_blocking=False):
        return RaggedMel(self.data.to(device, non_blocking=non_blocking),
                         self.table.to(device, non_blocking=non_blocking), self.frames,
                         None if self.segments is None else self.segments.to(device, non_blocking=non_blocking),
                         _checked=True, _host=self._host)

    def cuda(self, non_blocking=False):
        return self.to("cuda", non_blocking=non_blocking)

    def dense(self):
        """The reference collater's output, FloatTensor [B, Mel_Dim, T] (host restatement of Datasets.py:9-19)."""
        data = self.data.cpu().numpy()
        out = []
        for start, length, offset in self.table.cpu().numpy().tolist():
            feature = data[:, start:start + length]
            if length > self.frames:
                out.append(feature[:, offset:offset + self.frames])
            else:
                pad = (self.frames - length) / 2
                out.append(np.pad(feature, [[0, 0], [int(np.floor(pad)), int(np.ceil(pad))]], mode="reflect"))
        return torch.FloatTensor(np.stack(out, axis=0).astype(np.float32))


class Collater:
    """``Collater(min_frame_length, max_frame_length)(batch)`` with ``batch`` = list (speakers) of lists of
    ``(feature [Mel_Dim, L], speaker)`` as ``Datasets.Dataset.__getitem__`` returns them (Datasets.py:50-66)."""

    def __init__(self, min_frame_length, max_frame_length):
        self.min_frame_length = min_frame_length
        self.max_frame_length = max_frame_length

    def __call__(self, batch):
        # same draws, same order as the reference: one frame_length, then one offset per utterance that is longer
        frame_length = np.random.randint(self.min_frame_length, self.max_frame_length + 1)
        features = [feature for pattern in batch for feature, _ in pattern]
        table = np.zeros((len(features), 3), dtype=np.int32)
        start = 0
        for i, feature in enumerate(features):
            length = feature.shape[1]
            offset = np.random.randint(0, length - frame_length) if length > frame_length else 0
            table[i] = (start, length, offset)
            start += length
        dtype = np.float16 if all(f.dtype == np.float16 for f in features) else np.float32
        data = np.concatenate([np.asarray(f, dtype=dtype) for f in features], axis=1)
        return RaggedMel(torch.from_numpy(np.ascontiguousarray(data)), torch.from_numpy(table), frame_length)
