"""Host-side runtime around the kernels: CUDA-graph replay, utterance sharding, reference patching.

The path has no collective: every utterance is independent (SURVEY.md §8e), so multi-GPU
inference is one process per GPU, each running its shard; ``torch.distributed`` is used only for
the final gather of the waveforms and the timing barrier.
"""
from __future__ import annotations

import sys
from typing import Callable, Dict, List, Sequence, Tuple

import torch


def to_pcm16(audio: torch.Tensor, scale_norm: str = "max", prompt_audio_max=1.0, order: str = "plm",
             per_utterance: bool = False) -> torch.Tensor:
    """int16 PCM of a generated waveform, on the device (the step after the path, SURVEY.md §8f3).

    ``order="plm"``: ``audio / |audio|.max() * 32767.0 * s`` with s = 0.999, or ``prompt_audio_max`` when
    ``scale_norm == "prompt"`` (inference_plm.py:183-188); ``order="speechsr"``: ``... * 0.999 * 32767.0``
    (inference_speechsr.py:39-41).  Bit-exact with the reference's fp32 arithmetic + ``astype('int16')``.
    With ``per_utterance=True`` and ``scale_norm="prompt"``, ``prompt_audio_max`` may be a floating CUDA tensor of one
    value per row (each utterance's own prompt peak): row b then equals ``to_pcm16(row b, "prompt",
    float(prompt_audio_max[b]))``."""
    from . import ops
    if isinstance(prompt_audio_max, torch.Tensor):
        if order != "plm" or scale_norm != "prompt" or not per_utterance:
            raise ValueError("a per-row prompt_audio_max needs order='plm', scale_norm='prompt', per_utterance=True")
        if not prompt_audio_max.is_floating_point() or prompt_audio_max.dim() != 1:
            raise ValueError("prompt_audio_max must be a 1-D floating tensor, one value per row")
        rows = audio.numel() // audio.shape[-1] if audio.dim() and audio.shape[-1] else 0
        if prompt_audio_max.numel() != rows:
            raise ValueError(f"prompt_audio_max has {prompt_audio_max.numel()} values for {rows} rows")
        # fp32 rounding, as ctypes.c_float rounds the scalar
        s2 = prompt_audio_max.detach().to(torch.float32).contiguous()
        return ops.peak_norm_pcm16_rows(audio.detach().contiguous(), s2)[0]
    if order == "plm":
        s1, s2 = 32767.0, (float(prompt_audio_max) if scale_norm == "prompt" else 0.999)
    elif order == "speechsr":
        s1, s2 = 0.999, 32767.0
    else:
        raise ValueError("order must be 'plm' or 'speechsr'")
    pcm, _ = ops.peak_norm_pcm16(audio.detach().contiguous(), s1, s2, per_row=per_utterance)
    return pcm


class CudaGraphRunner:
    """Capture ``fn(*tensors)`` once per input-shape signature and replay it.

    One forward of the vocoder is ~290 small kernels; replaying them as a CUDA graph removes the
    launch gaps that dominate batch-1 latency.  Inputs are copied into static buffers; the returned
    tensors are the graph's static outputs (valid until the next call with the same shapes).

    A captured graph bakes in raw pointers to the folded / packed weights and to the operand workspaces, so the
    cache key carries the epochs that every event which can move those bumps (``load_state_dict`` on any hsv
    module, ``invalidate_caches()``, ``remove_weight_norm()``, ``ops.clear_workspace()``, workspace eviction) plus a
    ``config_token`` for host-side switches read at capture time (``parallel_blocks``, the fusion threshold):
    entries from an older epoch are dropped and recaptured, never replayed.  The cache is an LRU of at most
    ``max_graphs`` shapes; a shape is only captured on its ``capture_after``-th call (default: the first), earlier
    calls run eagerly -- set it to 2 under variable-length traffic so one-off lengths never pay a capture.

    Keyword arguments are passed to ``fn`` unchanged and are part of the signature (one graph per value): they take
    hashable host values, such as an output length or a flag."""

    def __init__(self, fn: Callable, warmup: int = 2, max_graphs: int = 16, capture_after: int = 1):
        from collections import OrderedDict
        self.fn = fn
        self.warmup = warmup
        self.max_graphs = max_graphs
        self.capture_after = capture_after
        self._graphs: "OrderedDict[Tuple, Tuple]" = OrderedDict()
        self._seen: Dict[Tuple, int] = {}
        self._pb_mods = None
        self.captures = 0

    def _version(self):
        from . import modules as M, ops
        if self._pb_mods is None:   # the (few) modules that carry the multi-stream switch, found once
            self._pb_mods = [m for m in (self.fn.modules() if hasattr(self.fn, "modules") else [])
                             if hasattr(m, "parallel_blocks")]
        par = tuple(bool(m.parallel_blocks) for m in self._pb_mods)
        return (M._CACHE_EPOCH[0], ops.WORKSPACE_EPOCH[0], M.FUSE_MAX_CHANNELS[0], M.FUSE_MAX_ELEMS[0],
                M.SEPARATE_MAX_ELEMS[0], ops.MHA_VARIANT[0], par)

    def _key(self, args, kwargs=None):
        key = tuple((tuple(a.shape), a.dtype, a.device.index) for a in args)
        if not kwargs:
            return key
        if any(isinstance(v, torch.Tensor) for v in kwargs.values()):
            raise TypeError("CudaGraphRunner: pass tensors positionally (keyword arguments are host values)")
        return key + (tuple(sorted(kwargs.items())),)

    def __call__(self, *args: torch.Tensor, **kwargs):
        from . import ops
        for a in args:
            if not a.is_cuda:
                raise RuntimeError("CudaGraphRunner: CUDA tensors only")
        key = self._key(args, kwargs)
        entry = self._graphs.get(key)
        if entry is not None and entry[3] != self._version():
            del self._graphs[key]          # stale pointers (weights refolded / workspaces moved): never replay
            entry = None
        if entry is None:
            self._seen[key] = self._seen.get(key, 0) + 1
            if len(self._seen) > 4096:
                self._seen.clear()
            if self._seen[key] < self.capture_after:
                with torch.no_grad():
                    return self.fn(*args, **kwargs)
            static_in = [torch.empty_like(a) for a in args]
            for s, a in zip(static_in, args):
                s.copy_(a)
            ops._pin_depth[0] += 1         # the pointers seen during warm-up must be the ones captured
            try:
                side = torch.cuda.Stream()
                side.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(side), torch.no_grad():
                    for _ in range(self.warmup):  # folds weights, allocates workspaces, loads modules
                        self.fn(*static_in, **kwargs)
                torch.cuda.current_stream().wait_stream(side)
                torch.cuda.synchronize()
                version = self._version()      # after warm-up: folding / packing may have happened in it
                graph = torch.cuda.CUDAGraph()
                with torch.no_grad(), torch.cuda.graph(graph):
                    static_out = self.fn(*static_in, **kwargs)
            finally:
                ops._pin_depth[0] -= 1
            if version != self._version():
                raise RuntimeError("CudaGraphRunner: weights or workspaces changed during capture")
            entry = (graph, static_in, static_out, version)
            self._graphs[key] = entry
            self.captures += 1
            while len(self._graphs) > self.max_graphs:
                self._graphs.popitem(last=False)
        self._graphs.move_to_end(key)
        graph, static_in, static_out, _ = entry
        for s, a in zip(static_in, args):
            if s.data_ptr() != a.data_ptr():
                s.copy_(a, non_blocking=True)
        graph.replay()
        return static_out

    def ready(self, *args, **kwargs) -> bool:
        """Whether a call with arguments of these shapes would replay a current graph (no eager run, no capture)."""
        entry = self._graphs.get(self._key(args, kwargs))
        return entry is not None and entry[3] == self._version()

    def static_inputs(self, *args, **kwargs):
        """The static input buffers for this shape signature (capture first if needed)."""
        self(*args, **kwargs)
        return self._graphs[self._key(args, kwargs)][1]

    def clear(self):
        self._graphs.clear()
        self._seen.clear()


def shard_utterances(lengths: Sequence[int], world_size: int, rank: int) -> List[int]:
    """Indices of the utterances rank ``rank`` processes: sort by length (longest first), deal
    round-robin in a serpentine order so every rank gets the same count (+-1) and near-equal total
    length.  Deterministic; the union over ranks is a partition of range(len(lengths))."""
    if not (0 <= rank < world_size):
        raise ValueError("rank out of range")
    order = sorted(range(len(lengths)), key=lambda i: (-int(lengths[i]), i))
    mine = []
    for pos, idx in enumerate(order):
        rnd, slot = divmod(pos, world_size)
        owner = slot if rnd % 2 == 0 else world_size - 1 - slot
        if owner == rank:
            mine.append(idx)
    return mine


def bucket_by_length(indices: Sequence[int], lengths: Sequence[int], max_batch: int) -> List[List[int]]:
    """Micro-batches of equal-length utterances (the Generator takes no masks, and replicate padding
    inside Activation1d makes padded batching differ near the boundary: SURVEY.md §8e)."""
    by_len: Dict[int, List[int]] = {}
    for i in indices:
        by_len.setdefault(int(lengths[i]), []).append(i)
    out = []
    for L in sorted(by_len, reverse=True):
        ids = by_len[L]
        for s in range(0, len(ids), max_batch):
            out.append(ids[s:s + max_batch])
    return out


def ragged_batches(indices: Sequence[int], lengths: Sequence[int], max_batch: int,
                   frame_multiple: int = 50) -> List[Tuple[List[int], int]]:
    """Micro-batches of utterances of different lengths for the ``lengths=`` path of the vocoder / SpeechSR modules:
    [(ids, T_padded)], sorted longest first and cut into consecutive runs of at most ``max_batch``; each batch is padded
    to its longest utterance rounded up to a multiple of ``frame_multiple``, which bounds the number of distinct
    padded shapes (one captured CUDA graph each) while keeping the padded fraction small.  Deterministic (ties keep
    index order); the batches partition ``indices``."""
    if max_batch < 1 or frame_multiple < 1:
        raise ValueError("max_batch and frame_multiple must be >= 1")
    order = sorted(indices, key=lambda i: (-int(lengths[i]), i))
    out = []
    for s in range(0, len(order), max_batch):
        ids = order[s:s + max_batch]
        longest = int(lengths[ids[0]])
        out.append((ids, -(-longest // frame_multiple) * frame_multiple))
    return out


def ragged_prompt_batches(indices: Sequence[int], lengths: Sequence[int], prompt_lengths: Sequence[int], max_batch: int,
                          frame_multiple: int = 50, prompt_multiple: int = 50) -> List[Tuple[List[int], int, int]]:
    """Micro-batches for the per-item voice-conversion calls (``HierSpeechSynthesizer.*(..., per_item=True)``):
    ``ragged_batches`` of the source lengths, each with its prompts padded to their longest rounded up to a multiple
    of ``prompt_multiple``: [(ids, T_padded, Tm_padded)].  Both roundings bound the number of distinct padded shapes
    (one captured CUDA graph each)."""
    if prompt_multiple < 1:
        raise ValueError("prompt_multiple must be >= 1")
    out = []
    for ids, T in ragged_batches(indices, lengths, max_batch, frame_multiple):
        longest = max(int(prompt_lengths[i]) for i in ids)
        out.append((ids, T, -(-longest // prompt_multiple) * prompt_multiple))
    return out


def gather_packed(flat: torch.Tensor, dst: int = 0):
    """The collective under ``gather_waveforms``: every rank contributes one 1-D buffer of the SAME size and dtype
    (pad to the largest shard), rank ``dst`` gets a [world, n] tensor, the others None.  No metadata exchange, no
    host synchronisation; the bytes travel as uint8 (NCCL has no int16)."""
    import torch.distributed as dist

    world, rank = dist.get_world_size(), dist.get_rank()
    wire = flat.contiguous().view(torch.uint8)
    if rank == dst:
        recv = torch.empty(world, flat.numel(), dtype=flat.dtype, device=flat.device)
        dist.gather(wire, list(recv.view(torch.uint8).view(world, -1).unbind(0)), dst=dst)
        return recv
    dist.gather(wire, None, dst=dst)
    return None


def gather_waveforms(local: Dict[int, torch.Tensor], dst: int = 0, sizes: Dict[int, int] = None):
    """Final gather of {utterance index: waveform} onto rank ``dst`` -- the only collective of the job.

    The payload moves as ONE flat tensor per rank through ``torch.distributed.gather`` (NCCL over NVLink for CUDA
    tensors -- no host staging, no pickling of audio; gloo for the CPU tests): every rank concatenates its
    waveforms (any common dtype: the int16 PCM of ``to_pcm16`` for the real job, fp32 for checks) into a buffer
    padded to the largest per-rank total, rank ``dst`` receives ``world`` such buffers into one preallocated
    tensor and returns views into it (original shapes).  Only the (index, shape) lists -- a few bytes per
    utterance -- are exchanged as Python objects; ``sizes`` = {utterance index: samples}, if given, is checked
    against them."""
    import torch.distributed as dist

    if not dist.is_available() or not dist.is_initialized() or dist.get_world_size() == 1:
        return dict(local)
    world, rank = dist.get_world_size(), dist.get_rank()
    mine = [(int(k), tuple(v.shape)) for k, v in sorted(local.items())]
    any_t = next(iter(local.values())) if local else None
    hello = [None] * world                    # (index, shape) lists + dtype/device: a few bytes per utterance
    dist.all_gather_object(hello, (mine, None if any_t is None else (str(any_t.dtype), any_t.device.type)))
    layout = [h[0] for h in hello]
    meta = [h[1] for h in hello if h[1] is not None]
    if sizes is not None:
        for part in layout:
            for k, shp in part:
                if int(sizes[k]) != int(torch.Size(shp).numel()):
                    raise ValueError(f"utterance {k}: {torch.Size(shp).numel()} samples, expected {sizes[k]}")
    layout = [[(k, shp, int(torch.Size(shp).numel())) for k, shp in part] for part in layout]
    totals = [sum(n for _, _, n in part) for part in layout]
    cap = max(totals) if totals else 0
    if not meta or cap == 0:
        return {} if rank == dst else None
    dtype = getattr(torch, meta[0][0].split(".")[-1])
    dev = any_t.device if any_t is not None else (torch.device("cuda", torch.cuda.current_device())
                                                  if meta[0][1] == "cuda" else torch.device("cpu"))
    flat = torch.zeros(cap, dtype=dtype, device=dev)
    off = 0
    for k, _shp in mine:
        n = local[k].numel()
        flat[off:off + n].copy_(local[k].reshape(-1))
        off += n
    # the payload travels as raw bytes: NCCL has no int16
    wire = flat.view(torch.uint8)
    if rank == dst:
        recv = torch.empty(world, cap, dtype=dtype, device=dev)
        dist.gather(wire, list(recv.view(torch.uint8).view(world, -1).unbind(0)), dst=dst)
        merged = {}
        for r, part in enumerate(layout):
            off = 0
            for k, shp, n in part:
                merged[k] = recv[r, off:off + n].view(shp)
                off += n
        return merged
    dist.gather(wire, None, dst=dst)
    return None


def patch_reference(modules=None, front: bool = True) -> List[str]:
    """Swap the reference's hot-path classes for the B200 ones in already-imported reference modules
    (``hierspeechpp_speechsynthesizer``, ``speechsr24k.speechsr``, ``speechsr48k.speechsr``,
    ``alias_free_torch``), so the reference's own ``SynthesizerTrn``/inference scripts build and call
    them.  Returns the list of patched attributes.  See INTEGRATION.md."""
    from . import front as FR
    from . import modules as M

    mods = modules if modules is not None else sys.modules
    patched = []

    def _set(modname, attr, obj):
        m = mods.get(modname)
        if m is not None:
            setattr(m, attr, obj)
            patched.append(f"{modname}.{attr}")

    for attr, obj in (("Generator", M.Generator), ("SourceNetwork", M.SourceNetwork), ("AMPBlock1", M.AMPBlock1),
                      ("DBlock", M.DBlock), ("Activation1d", M.Activation1d)):
        _set("hierspeechpp_speechsynthesizer", attr, obj)
    _set("speechsr24k.speechsr", "Generator", M.SpeechSR24Generator)
    _set("speechsr24k.speechsr", "AMPBlock0", M.AMPBlock0)
    _set("speechsr24k.speechsr", "Activation1d", M.Activation1d)
    _set("speechsr48k.speechsr", "Generator", M.SpeechSR48Generator)
    _set("speechsr48k.speechsr", "AMPBlock0", M.AMPBlock0)
    _set("speechsr48k.speechsr", "Activation1d", M.Activation1d)
    for attr, obj in (("Activation1d", M.Activation1d), ("UpSample1d", M.UpSample1d),
                      ("DownSample1d", M.DownSample1d), ("LowPassFilter1d", M.LowPassFilter1d)):
        _set("alias_free_torch", attr, obj)
    _set("activations", "SnakeBeta", M.SnakeBeta)
    if front:
        # the step before the vocoder (SURVEY.md §8f2): enc_p_l, flow_l / flow, emb_g of SynthesizerTrn
        for attr, obj in (("PosteriorSFEncoder", FR.PosteriorSFEncoder),
                          ("ResidualCouplingBlock_Transformer", FR.ResidualCouplingBlock_Transformer),
                          ("StyleEncoder", FR.StyleEncoder)):
            _set("hierspeechpp_speechsynthesizer", attr, obj)
        # ... and the tail of the text-to-vec model that feeds it (SURVEY.md §8f4, partial); only when the caller has
        # imported ttv_v1.t2w2v_transformer (its SynthesizerTrn builds self.w2v_decoder / self.pp from these names)
        from . import ttv as TV
        _set("ttv_v1.t2w2v_transformer", "W2VDecoder", TV.W2VDecoder)
        _set("ttv_v1.t2w2v_transformer", "PitchPredictor", TV.PitchPredictor)
    return patched
